#!/usr/bin/env python3
"""Command-line front end with the reference's flags (reference raytracer/src/main.rs:78-107):

    python yart_cli.py --scene david [--output out.png] [--width W] [--height H] [--samples N]
                       [--max-depth D] [--vfov F] [--aperture A]            (reference flags)
                       [--seed S] [--order near|reference] [--device D] [--gpus N]   (additions)
                       [--preview-every N] [--checkpoint FILE] [--resume]    (additions)
                       [--unbiased-light-pick] [--russian-roulette] [--depth-zero-black] [--next-event]   (better sampling, off by default)
                       [--aovs [--aov-samples N]]                            (denoiser inputs)
                       [--denoise]                                           (built-in denoiser)

`--workers` is accepted for compatibility and ignored (the render runs on the GPU).  Option resolution
follows resolve_render_options / resolve_dimensions (main.rs:166-209); the image is finalised exactly like
main.rs:710-718 and written as PNG (main.rs:769-774).  There is no CPU mode.

Progressive output and checkpoints rest on one property of yart_render (tests/test_gpu_render.py): the film is
the per-pixel SUM of samples added in sample order, so rendering [0, a) and then [a, b) into the same film is
bit-identical to rendering [0, b) at once.  `--preview-every N` writes the PNG of what exists after every N
samples per pixel; `--checkpoint FILE` stores (film, samples done, the options that define the image) as .npz at
the same moments; `--resume` continues from FILE if it matches the request.

`--gpus N` renders on GPUs device .. device+N-1 of this box: every GPU takes its share of each sample range and the
films are combined by the library's NCCL reduce (yet-another-raytracer_b200/sharding.py, yart_film_reduce).  The three
sampling flags change the ESTIMATOR (SURVEY.md 8(f) row 4) and are off unless asked for; they are part of a
checkpoint's identity.

`--aovs` also writes the inputs of a denoiser such as Open Image Denoise (`oidnDenoise --hdr <stem>.color.pfm --alb
<stem>.albedo.pfm --nrm <stem>.normal.pfm`) next to the PNG: <stem>.color.pfm is the film as linear RGB
(yart_film_finalize_linear), and <stem>.albedo.pfm, <stem>.normal.pfm and <stem>.depth.pfm (one channel: the mean
distance of the samples that hit, 0 where none did) are the first-hit means of samples [0, --aov-samples) (default
min(16, --samples)), the very camera samples the beauty pass started with (yart_render_aovs).  They are rendered once,
after the beauty pass, on the first GPU, and are not part of a checkpoint.

`--denoise` also writes <stem>.denoised.png and <stem>.denoised.pfm (linear RGB): the film denoised on the GPU by the
library's own a-trous filter (yart_denoise), guided by the first-hit planes of samples [0, --aov-samples), rendered as
for --aovs whether or not --aovs is given.  The main PNG is the same with or without it.
"""
import argparse
import importlib
import os
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def positive_int(text):  # parse_positive_usize (main.rs:148-158)
    try:
        v = int(text)
    except ValueError as e:
        raise argparse.ArgumentTypeError("invalid integer `%s`: %s" % (text, e))
    if v <= 0:
        raise argparse.ArgumentTypeError("value must be greater than 0")
    return v


def build_parser(scene_names):
    ap = argparse.ArgumentParser(description="Render predefined raytracer scenes")
    ap.add_argument("--scene", required=True, choices=scene_names)
    ap.add_argument("--output", default=None)
    ap.add_argument("--width", type=positive_int, default=None)
    ap.add_argument("--height", type=positive_int, default=None)
    ap.add_argument("--samples", type=positive_int, default=None)
    ap.add_argument("--max-depth", type=positive_int, default=None, dest="max_depth")
    ap.add_argument("--workers", type=positive_int, default=None)
    ap.add_argument("--vfov", type=float, default=None)
    ap.add_argument("--aperture", type=float, default=None)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--order", choices=["near", "reference"], default="near")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--gpus", type=positive_int, default=1, help="render on this many GPUs (device, device+1, ...)")
    ap.add_argument("--unbiased-light-pick", action="store_true", dest="unbiased_light_pick",
                    help="sample ALL lights (the reference never samples the last one, hittable.rs:113-122)")
    ap.add_argument("--russian-roulette", action="store_true", dest="russian_roulette")
    ap.add_argument("--depth-zero-black", action="store_true", dest="depth_zero_black",
                    help="paths cut at --max-depth contribute 0 (the reference returns 1.0, main.rs:544-546)")
    ap.add_argument("--next-event", action="store_true", dest="next_event",
                    help="next-event estimation with MIS: one shadow ray toward a light per diffuse hit "
                         "(implies --unbiased-light-pick)")
    ap.add_argument("--preview-every", type=positive_int, default=None, dest="preview_every",
                    help="write the image after every N samples per pixel")
    ap.add_argument("--checkpoint", default=None, help=".npz file holding the film and the samples done so far")
    ap.add_argument("--resume", action="store_true", help="continue from --checkpoint if it matches this render")
    ap.add_argument("--aovs", action="store_true",
                    help="also write <stem>.color/.albedo/.normal/.depth.pfm next to the PNG (denoiser inputs)")
    ap.add_argument("--aov-samples", type=positive_int, default=None, dest="aov_samples",
                    help="samples per pixel of the albedo / normal / depth images (default min(16, --samples))")
    ap.add_argument("--denoise", action="store_true",
                    help="also write <stem>.denoised.png / .denoised.pfm, denoised by yart_denoise")
    return ap


def _identity(args, o):
    """Everything that decides what sample k of pixel p is; a checkpoint is only valid for the same values."""
    ident = [args.scene, int(o["width"]), int(o["height"]), int(o["max_depth"]), float(o["vfov"]), float(o["aperture"]),
             int(args.seed)]
    flags = _flags(args)
    return ident + ([flags] if flags else [])  # (unchanged for the reference's estimator: old checkpoints stay valid)


def _flags(args):
    y = importlib.import_module("yet-another-raytracer_b200")
    return ((y.FLAG_UNBIASED_LIGHT_PICK if args.unbiased_light_pick else 0) | (y.FLAG_RUSSIAN_ROULETTE if args.russian_roulette else 0) |
            (y.FLAG_DEPTH_ZERO_BLACK if args.depth_zero_black else 0) | (y.FLAG_NEXT_EVENT if args.next_event else 0))


def save_checkpoint(path, film, done, ident):
    import json
    import numpy as np
    tmp = path + ".tmp.npz"
    np.savez(tmp, film=film, samples_done=np.int64(done), identity=np.array(json.dumps(ident)))
    os.replace(tmp, path)  # a kill during the write leaves the previous checkpoint intact


def load_checkpoint(path, ident):
    import json
    import numpy as np
    with np.load(path) as z:
        if json.loads(str(z["identity"])) != ident:
            raise SystemExit("checkpoint %s was made with other options: %s" % (path, str(z["identity"])))
        return np.ascontiguousarray(z["film"]), int(z["samples_done"])


def write_png(ctx, film, spp_done, path):
    parent = os.path.dirname(path)
    if parent:
        os.makedirs(parent, exist_ok=True)
    from PIL import Image
    Image.fromarray(ctx.film_finalize(film, spp_done), "RGBA").save(path)


def write_pfm(path, img):
    """A portable float map: (H, W, 3) -> "PF", (H, W) -> "Pf"; little-endian f32, rows bottom to top."""
    import numpy as np
    img = np.asarray(img, dtype="<f4")
    with open(path, "wb") as f:
        f.write(b"%s\n%d %d\n-1.0\n" % (b"PF" if img.ndim == 3 else b"Pf", img.shape[1], img.shape[0]))
        f.write(np.ascontiguousarray(img[::-1]).tobytes())


def read_pfm(path):
    """write_pfm's inverse (either byte order)."""
    import numpy as np
    with open(path, "rb") as f:
        kind = f.readline().strip()
        w, h = (int(v) for v in f.readline().split())
        scale = float(f.readline())
        data = np.frombuffer(f.read(), dtype="<f4" if scale < 0 else ">f4")
    shape = (h, w, 3) if kind == b"PF" else (h, w)
    return data.reshape(shape)[::-1].astype(np.float32)


def aov_paths(output_path):
    stem = os.path.splitext(output_path)[0]
    return {k: "%s.%s.pfm" % (stem, k) for k in ("color", "albedo", "normal", "depth")}


def denoised_paths(output_path):
    stem = os.path.splitext(output_path)[0]
    return {"png": stem + ".denoised.png", "pfm": stem + ".denoised.pfm"}


def write_aovs(y, ctx, cam, o, args, order, flags, film, spp):
    """The first-hit planes of samples [0, --aov-samples), then what --aovs and --denoise write from them."""
    n = args.aov_samples or min(16, spp)
    planes, _ = ctx.render_aovs(cam, o["width"], o["height"], 0, n, o["max_depth"], args.seed, order, flags=flags)
    if args.aovs:
        means = y.aov_means(planes)
        paths = aov_paths(o["output_path"])
        write_pfm(paths["color"], ctx.film_finalize_linear(film, spp))
        for k in ("albedo", "normal", "depth"):
            write_pfm(paths[k], means[k])
    if args.denoise:
        from PIL import Image
        rgb, rgba = ctx.denoise(film, spp, planes, rgba=True)
        paths = denoised_paths(o["output_path"])
        write_pfm(paths["pfm"], rgb)
        Image.fromarray(rgba, "RGBA").save(paths["png"])


def main(argv=None):
    y = importlib.import_module("yet-another-raytracer_b200")
    args = build_parser(y.SCENE_NAMES).parse_args(argv)
    preset = y.ScenePreset(args.scene, seed=args.seed)
    if preset.note:
        print("note: " + preset.note, file=sys.stderr)
    o = preset.resolve_render_options(args.output, args.width, args.height, args.samples, args.max_depth,
                                      args.workers, args.vfov, args.aperture)
    start = time.time()  # the reference's timer starts in render(), after the scene is built (main.rs:591)
    cam = preset.camera(o["width"], o["height"], o["vfov"], o["aperture"])
    order = y.ORDER_NEAR if args.order == "near" else y.ORDER_REFERENCE
    flags = _flags(args)
    total = o["samples_per_pixel"]
    ident = _identity(args, o)
    film, done = None, 0
    if args.resume:
        if not args.checkpoint:
            raise SystemExit("--resume needs --checkpoint FILE")
        if os.path.exists(args.checkpoint):
            film, done = load_checkpoint(args.checkpoint, ident)
            if done > total:  # the film already holds more samples than asked for: dividing it by `total` would over-expose
                raise SystemExit("checkpoint %s already holds %d samples per pixel, more than --samples %d; "
                                 "ask for at least that many" % (args.checkpoint, done, total))
            print("resuming %s at %d of %d samples per pixel" % (args.checkpoint, done, total))
    step = args.preview_every or total
    paths = rays = 0
    gpu_ms = 0.0
    multi = None
    if args.gpus > 1:
        if args.device + args.gpus > y.device_count():
            raise SystemExit("--gpus %d from --device %d: only %d GPU(s) visible" % (args.gpus, args.device, y.device_count()))
        sharding = importlib.import_module("yet-another-raytracer_b200.sharding")
        multi = sharding.MultiGpuRenderer(y, range(args.device, args.device + args.gpus))
        multi.set_scene(preset)
        ctx = multi.contexts[0]
        if film is not None:
            multi.load_film(film)
    else:
        ctx = y.Context(args.device)
        ctx.set_scene(preset)
    while done < total:
        nxt = min(total, done + step)
        if multi is not None:
            sts = multi.render(cam, o["width"], o["height"], done, nxt, o["max_depth"], args.seed, order, flags)
            paths, rays = paths + sum(s.paths for s in sts), rays + sum(s.rays for s in sts)
            gpu_ms, done = gpu_ms + max(s.gpu_ms for s in sts), nxt
            if done < total or args.checkpoint or done == total:
                film = multi.film()
        else:
            film, st = ctx.render(cam, o["width"], o["height"], done, nxt, o["max_depth"], args.seed, order, film=film, flags=flags)
            paths, rays, gpu_ms, done = paths + st.paths, rays + st.rays, gpu_ms + st.gpu_ms, nxt
        if done < total or args.checkpoint:
            if args.checkpoint:
                save_checkpoint(args.checkpoint, film, done, ident)
            if done < total:
                write_png(ctx, film, done, o["output_path"])  # normalised by the samples that exist so far
    if film is None:  # (resumed a finished render)
        raise SystemExit("nothing to do")
    write_png(ctx, film, total, o["output_path"])
    if args.aovs or args.denoise:
        write_aovs(y, ctx, cam, o, args, order, flags, film, total)
    if multi is not None:
        multi.close()
    print("%s rendered in %d seconds" % (o["output_path"], int(time.time() - start)))  # main.rs:763-767
    print("  %d paths, %d rays, %.1f Mrays/s on the device" % (paths, rays, rays / max(gpu_ms, 1e-9) / 1e3))
    return 0


if __name__ == "__main__":
    sys.exit(main())

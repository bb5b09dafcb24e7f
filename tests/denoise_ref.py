"""numpy restatement of yart_denoise (include/yart.h): the edge-avoiding a-trous filter guided by the AOV planes.

Vectorised over pixels, with the levels and the 25 taps looped in the header's order and every expression evaluated in
the header's order in f64, so the f32 image equals the library's bit for bit.  numpy does no FMA contraction and calls
no libm here, and the library is built with -fmad=false."""
import numpy as np

DEFAULT_LEVELS, MAX_LEVELS = 5, 10
DEFAULT_SIGMAS = (8.0, 0.3, 0.05)  # sigma_color, sigma_normal, sigma_depth (DESIGN section 8)
H = (1.0 / 16.0, 1.0 / 4.0, 3.0 / 8.0, 1.0 / 4.0, 1.0 / 16.0)


def resolve(levels=0, sigma_color=0.0, sigma_normal=0.0, sigma_depth=0.0):
    """(levels, sigma_color, sigma_normal, sigma_depth) after the header's defaults; ValueError where the library
    returns YART_ERR_INVALID."""
    sig = (sigma_color, sigma_normal, sigma_depth)
    if not 0 <= levels <= MAX_LEVELS or not all(np.isfinite(s) for s in sig):
        raise ValueError("levels must be 0..%d and the sigmas finite" % MAX_LEVELS)
    return (levels or DEFAULT_LEVELS,) + tuple(float(s) if s > 0 else d for s, d in zip(sig, DEFAULT_SIGMAS))


def film_linear(film, spp):
    """film_linear_rgb of device_shade.cuh over a whole film, in f64 and without the tile mask."""
    mul, den = 720.0 - 360.0, 106.856895 * float(spp)
    c = [film[..., k] * mul / den for k in range(3)]
    r = 2.6896552 * c[0] - 1.2758621 * c[1] - 0.4137931 * c[2]
    g = -1.0221082 * c[0] + 1.9782866 * c[1] + 0.0438216 * c[2]
    b = 0.0612245 * c[0] - 0.2244898 * c[1] + 1.1632653 * c[2]
    return np.stack([r, g, b], axis=2)


def _shift(a, dy, dx, fill):
    """b[y, x] = a[y + dy, x + dx], `fill` outside the image."""
    h, w = a.shape[:2]
    b = np.full_like(a, fill)
    ys, yd = (slice(dy, h), slice(0, h - dy)) if dy >= 0 else (slice(0, h + dy), slice(-dy, h))
    xs, xd = (slice(dx, w), slice(0, w - dx)) if dx >= 0 else (slice(0, w + dx), slice(-dx, w))
    if ys.stop > ys.start and xs.stop > xs.start:
        b[yd, xd] = a[ys, xs]
    return b


def denoise(film, spp, planes, levels=0, sigma_color=0.0, sigma_normal=0.0, sigma_depth=0.0):
    """The filtered image in f64, (H, W, 3), 0 at invalid pixels; .astype(np.float32) is yart_denoise's rgb."""
    L, sc, sn, sz = resolve(levels, sigma_color, sigma_normal, sigma_depth)
    albedo, normal, depth = (np.asarray(planes[k], dtype=np.float64) for k in ("albedo", "normal", "depth"))
    film = np.asarray(film, dtype=np.float64)
    with np.errstate(all="ignore"):
        valid = depth[..., 2] > 0.0
        hit = valid & (depth[..., 1] > 0.0)
        samples = np.where(valid, depth[..., 2], 1.0)[..., None]
        m = albedo / samples + 1.0 / 128.0
        c = np.where(valid[..., None], film_linear(film, spp) / m, 0.0)
        n = np.where(valid[..., None], normal / samples, 0.0)
        z = np.where(hit, depth[..., 0] / np.where(hit, depth[..., 1], 1.0), 0.0)
        iz = np.where(hit, 1.0 / ((sz * sz * z) * z), 0.0)
        kn = 1.0 / (sn * sn)
        for i in range(L):
            s = 1 << i
            kc = float(4.0 ** i) / (sc * sc)
            W = np.zeros(valid.shape)
            S = np.zeros(c.shape)
            for dy in range(-2, 3):
                for dx in range(-2, 3):
                    h = H[dy + 2] * H[dx + 2]
                    if dy == 0 and dx == 0:
                        use, w = valid, np.full(valid.shape, h)
                        cq = c
                    else:
                        vq = _shift(valid, dy * s, dx * s, False)
                        hq = _shift(hit, dy * s, dx * s, False)
                        cq = _shift(c, dy * s, dx * s, 0.0)
                        nq = _shift(n, dy * s, dx * s, 0.0)
                        zq = _shift(z, dy * s, dx * s, 0.0)
                        use = valid & vq & (hq == hit)
                        d = cq - c
                        e = nq - n
                        x = (((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]) * kc
                             + ((e[..., 0] * e[..., 0] + e[..., 1] * e[..., 1]) + e[..., 2] * e[..., 2]) * kn)
                        dz = zq - z
                        x = np.where(hit, x + (dz * dz) * iz, x)
                        t = 1.0 / (1.0 + x * 0.125)
                        t = t * t
                        t = t * t
                        t = t * t
                        w = h * t
                    W = np.where(use, W + w, W)
                    S = np.where(use[..., None], S + w[..., None] * cq, S)
            c = np.where(valid[..., None], S / np.where(valid, W, 1.0)[..., None], 0.0)
        return np.where(valid[..., None], c * m, 0.0)


def display_rgba(out, depth):
    """yart_denoise's rgba8 from the f64 image, with numpy's pow for the sRGB curve (gamma_channel and
    clamp_display_channel of device_shade.cuh).  Also returns 256 * gamma, since where that lies next to an integer a
    last-bit difference between CUDA's pow and numpy's can move a byte."""
    valid = np.asarray(depth)[..., 2] > 0.0
    with np.errstate(all="ignore"):
        lin = np.fmax(out, 0.0)
        g = np.where(lin <= 0.0031308, 12.92 * lin, 1.055 * np.power(lin, 1.0 / 2.4) - 0.055)
        v = 256.0 * np.clip(g, 0.0, 0.999)
    rgba = np.zeros(out.shape[:2] + (4,), np.uint8)
    rgba[..., :3] = np.where(valid[..., None], np.where(np.isnan(v), 0.0, v), 0.0).astype(np.uint8)
    rgba[..., 3] = np.where(valid, 255, 0)
    return rgba, 256.0 * g


def rel_mse(img, ref, valid):
    """Mean over the valid pixels and the channels of (img - ref)^2 / (ref^2 + 0.01), on linear RGB."""
    img, ref = np.asarray(img, np.float64)[valid], np.asarray(ref, np.float64)[valid]
    return float(np.mean((img - ref) ** 2 / (ref * ref + 0.01)))

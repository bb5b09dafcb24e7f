#!/usr/bin/env python3
"""A/B builds of libyart_b200.so with other -D knobs (e.g. YART_SHADE_MIN_BLOCKS=3) into ab/<tag>.so.

    python tools/ab_build.py tag1:-DYART_SHADE_MIN_BLOCKS=3 tag2:-DYART_TRAVERSE_MIN_BLOCKS=5,-DFOO=1 ...

Only yart_device.cu is recompiled per variant; the other objects come from the regular build (build/).  Run a variant
with YART_LIB_PATH=ab/<tag>.so.  ab/ is scratch (git-ignored through *.so) but travels to the GPU box."""
import importlib
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
b = importlib.import_module("yet-another-raytracer_b200.build")


def one(spec):
    tag, _, flags = spec.partition(":")
    flags = [f for f in flags.split(",") if f]
    b.build()
    obj = ROOT / "ab" / (tag + ".o")
    cmd = [b.nvcc_path()] + b.COMPILE_FLAGS + flags + ["-c", str(b.CSRC / "yart_device.cu"), "-o", str(obj)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    (ROOT / "ab" / (tag + ".log")).write_text(" ".join(cmd) + "\n" + r.stdout + r.stderr)
    if r.returncode:
        return tag, "COMPILE FAILED\n" + r.stderr[-2000:]
    others = [str(b.OBJ_DIR / (s.replace(".", "_") + ".o")) for s in b.SOURCES if s != "yart_device.cu"]
    lib = ROOT / "ab" / (tag + ".so")
    r2 = subprocess.run([b.nvcc_path()] + b.LINK_FLAGS + ["-o", str(lib), str(obj)] + others, capture_output=True, text=True)
    if r2.returncode:
        return tag, "LINK FAILED\n" + r2.stderr[-2000:]
    obj.unlink()
    text = r.stdout + r.stderr
    info = []
    lines = text.splitlines()
    for i, ln in enumerate(lines):
        if "Compiling entry function" in ln and ("k_traverseILb0ELb0ELi32E" in ln or "k_shade" in ln):
            name = "k_shade" if "k_shade" in ln else "k_traverse<reference>"
            info.append("%s: %s | %s" % (name, lines[i + 2].strip() if i + 2 < len(lines) else "", lines[i + 3].strip() if i + 3 < len(lines) else ""))
    return tag, "\n  ".join(info)


if __name__ == "__main__":
    (ROOT / "ab").mkdir(exist_ok=True)
    b.build()
    with ThreadPoolExecutor(max_workers=4) as ex:
        for tag, info in ex.map(one, sys.argv[1:]):
            print(tag + ":\n  " + info)

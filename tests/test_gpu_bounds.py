"""Memory-safety run: every kernel and scene feature through the bounds-checked library.

compute-sanitizer is not offered on the GPU pool, so `build.py --bounds-check` compiles the same sources with
-DYART_BOUNDS_CHECK: every index into the tree, the triangle records, the traversal stack, the ray / hit
arrays and the path queues is checked on the device and a violation traps (the process then fails)."""
import os
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
CHECKED = ROOT / "yet-another-raytracer_b200" / "libyart_b200_checked.so"


def test_checked_library_contains_the_checks():
    if not CHECKED.exists():
        pytest.skip("bounds-checked library not built (python yet-another-raytracer_b200/build.py --bounds-check)")
    assert b"YART_CHECK failed" in CHECKED.read_bytes()
    assert b"cur < P.n_nodes" in CHECKED.read_bytes()  # the traversal's node-index check
    assert b"YART_CHECK failed" not in (CHECKED.parent / "libyart_b200.so").read_bytes()


@pytest.mark.gpu
def test_every_kernel_under_bounds_checks():
    assert CHECKED.exists(), "run __graft_entry__.build() first"
    env = dict(os.environ, YART_LIB_PATH=str(CHECKED))
    res = subprocess.run([sys.executable, str(ROOT / "tools" / "exercise_kernels.py")], env=env, capture_output=True,
                         text=True, timeout=600)
    out = res.stdout + res.stderr
    assert "YART_CHECK failed" not in out, out[-2000:]
    assert res.returncode == 0, out[-2000:]
    assert "exercise done" in out

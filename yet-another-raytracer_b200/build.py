"""Builds libyart_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python yet-another-raytracer_b200/build.py [--force] [--verbose]
    python yet-another-raytracer_b200/build.py --bounds-check    (-> libyart_b200_checked.so, see below)

Flags that matter:
  -gencode arch=compute_100a,code=sm_100a   B200 only, no PTX for other archs
  -fmad=false                               the reference is f64 Rust without FMA contraction;
                                            bit-exact closest-hit parity needs the same roundings
  -Xcompiler -ffp-contract=off              same for the host-side QBVH build / camera maths
  -lineinfo                                 so ncu's source page maps SASS back to these files

Every source is compiled to its own object (in parallel, cached under build/ by a digest of the source, the headers
and the flags) and the objects are linked into the shared library; `build.log` keeps the ptxas -v output of all of them.

--bounds-check builds a second library with -DYART_BOUNDS_CHECK: every index the kernels form (tree nodes,
triangle records, traversal stack, ray / hit / queue slots) is checked and a violation traps.  It stands in
for compute-sanitizer, which the GPU pool does not offer; run it with
YART_LIB_PATH=yet-another-raytracer_b200/libyart_b200_checked.so (tests/test_gpu_bounds.py does).
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
ROOT = PKG.parent
LIB = PKG / "libyart_b200.so"
LIB_CHECKED = PKG / "libyart_b200_checked.so"
HOST_EXE = PKG / "yart"  # the native command-line host (host/yart_main.cpp): the reference's flags on the C ABI
OBJ_DIR = PKG / "build"

SOURCES = ["host_obj.cpp", "host_qbvh.cpp", "host_presets.cpp", "host_api.cpp", "yart_device.cu", "device_trace_lean.cu",
           "device_build.cu", "device_comm.cu", "device_occlude.cu"]
HEADERS = ["host_common.h", "device_common.cuh", "device_trace.cuh", "device_shade.cuh", "device_build.h", "device_occlude.h"]
INCLUDES = ["yart.h", "yart_rng.h", "yart_spectral_tables.h"]

COMPILE_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo", "-fmad=false",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math,-Wall",
    "-Xptxas", "-v",
]
LINK_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "--shared", "-cudart", "shared", "-ldl"]
# tuning knobs: resident blocks per SM / CTA sizes the kernels are compiled for
for knob in ("YART_TRAVERSE_MIN_BLOCKS", "YART_SHADE_MIN_BLOCKS", "YART_TRACE_THREADS", "YART_SHADE_THREADS"):
    if os.environ.get(knob):
        COMPILE_FLAGS += ["-D%s=%s" % (knob, os.environ[knob])]
for extra in os.environ.get("YART_NVCC_EXTRA", "").split():
    COMPILE_FLAGS.append(extra)


def _digest(source, extra):
    h = hashlib.sha256()
    for f in [CSRC / source] + [CSRC / s for s in HEADERS] + [ROOT / "include" / i for i in INCLUDES] + [Path(__file__)]:
        h.update(f.read_bytes())
    h.update(" ".join(COMPILE_FLAGS + extra).encode())
    return h.hexdigest()


def nvcc_path():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _compile(source, extra, tag, force):
    obj = OBJ_DIR / ("%s%s.o" % (source.replace(".", "_"), tag))
    stamp = obj.with_suffix(".digest")
    log = obj.with_suffix(".log")
    digest = _digest(source, extra)
    if not force and obj.exists() and stamp.exists() and log.exists() and stamp.read_text().strip() == digest:
        return obj, log.read_text(), 0
    cmd = [nvcc_path()] + COMPILE_FLAGS + extra + ["-c", str(CSRC / source), "-o", str(obj)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    text = " ".join(cmd) + "\n" + res.stdout + res.stderr
    log.write_text(text)
    if res.returncode == 0:
        stamp.write_text(digest)
    return obj, text, res.returncode


def build(force=False, verbose=False, bounds_check=False):
    lib = LIB_CHECKED if bounds_check else LIB
    tag = "_checked" if bounds_check else ""
    extra = ["-DYART_BOUNDS_CHECK"] if bounds_check else []
    OBJ_DIR.mkdir(exist_ok=True)
    lib_stamp = PKG / (".build_stamp_checked" if bounds_check else ".build_stamp")
    total = hashlib.sha256("".join(_digest(s, extra) for s in SOURCES).encode()).hexdigest()
    if not force and lib.exists() and lib_stamp.exists() and lib_stamp.read_text().strip() == total:
        if not bounds_check:
            build_host()
        return str(lib)
    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as ex:
        results = list(ex.map(lambda s: _compile(s, extra, tag, force), SOURCES))
    logs = "".join(r[1] for r in results)
    log_path = PKG / ("build_checked.log" if bounds_check else "build.log")
    if any(r[2] for r in results):
        log_path.write_text(logs)
        sys.stderr.write("".join(r[1] for r in results if r[2]))
        raise RuntimeError("nvcc failed (see %s)" % log_path)
    cmd = [nvcc_path()] + LINK_FLAGS + ["-o", str(lib)] + [str(r[0]) for r in results]
    res = subprocess.run(cmd, capture_output=True, text=True)
    logs += " ".join(cmd) + "\n" + res.stdout + res.stderr
    log_path.write_text(logs)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("link failed (see %s)" % log_path)
    if verbose:
        print(logs)
    lib_stamp.write_text(total)
    if not bounds_check:
        build_host(force=True)
    return str(lib)


def build_host(force=False):
    """g++ (no nvcc, no CUDA headers): host/yart_main.cpp needs nothing but include/yart.h and the shared library."""
    src = PKG / "host" / "yart_main.cpp"
    stamp = PKG / ".build_stamp_host"
    digest = hashlib.sha256(src.read_bytes() + (ROOT / "include" / "yart.h").read_bytes()).hexdigest()
    if not force and HOST_EXE.exists() and stamp.exists() and stamp.read_text().strip() == digest:
        return str(HOST_EXE)
    cmd = [os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-Wall", "-Wextra", "-I", str(ROOT / "include"), str(src), "-o", str(HOST_EXE),
           "-L", str(PKG), "-lyart_b200", "-Wl,-rpath,$ORIGIN", "-pthread"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("host program build failed")
    stamp.write_text(digest)
    return str(HOST_EXE)


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, bounds_check="--bounds-check" in sys.argv))

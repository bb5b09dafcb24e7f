#!/usr/bin/env python3
"""What the compiler made of k_shade, from a build of libyart_b200.so (needs no GPU):

    python tools/shade_sass.py [--lib LIB] [--log BUILD_LOG]

Per k_shade instance: ptxas's stack frame and spill bytes (from the build log), the SASS counts of local-memory
accesses (STL / LDL), subroutine calls (CALL; most go to the f64 division slow path every inlined `/` carries), block
barriers (BAR) and the size of the kernel body (up to its first unpredicated EXIT; the called subroutines follow it).
Then one SHA-256 per traversal kernel over its SASS, so that two builds can be checked instruction-identical there."""
import argparse
import collections
import hashlib
import re
import subprocess
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "yet-another-raytracer_b200"
SHADE = [("k_shade<false>", "_ZN4yart7k_shadeILb0EEEvNS_12RenderParamsEPKjS3_PjS4_jNS_8NeeStateE"),
         ("k_shade<true>", "_ZN4yart7k_shadeILb1EEEvNS_12RenderParamsEPKjS3_PjS4_jNS_8NeeStateE")]
TRAVERSAL = re.compile(r"_ZN4yart(10k_traverse|15k_traverse_lean|9k_occlude)I")
INSN = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(@!?U?P[T\d]+\s+)?([A-Z0-9_.]+)([^;]*);")


def functions(lib):
    """{symbol: [(offset, predicate, opcode, operands)]} of every kernel in the library."""
    out = subprocess.run(["cuobjdump", "-sass", str(lib)], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for ln in out.splitlines():
        m = re.search(r"Function : (\S+)", ln)
        if m:
            cur = funcs.setdefault(m.group(1), [])
            continue
        m = INSN.search(ln)
        if m and cur is not None:
            cur.append((int(m.group(1), 16), (m.group(2) or "").strip(), m.group(3), m.group(4).strip()))
    return funcs


def ptxas_lines(log, sym):
    lines = log.splitlines()
    for i, ln in enumerate(lines):
        if "Compiling entry function '%s'" % sym in ln:
            return lines[i + 2].strip(), lines[i + 3].strip()
    return "(not in the build log)", ""


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=str(PKG / "libyart_b200.so"))
    ap.add_argument("--log", default=str(PKG / "build" / "yart_device_cu.log"))
    a = ap.parse_args()
    funcs = functions(a.lib)
    log = Path(a.log).read_text() if Path(a.log).exists() else ""
    for name, sym in SHADE:
        insns = funcs[sym]
        ops = collections.Counter(op.split(".")[0] for _, _, op, _ in insns)
        body = next((off + 16 for off, pred, op, _ in insns if op == "EXIT" and not pred), None)
        calls = collections.Counter(arg for _, _, op, arg in insns if op.startswith("CALL"))
        frame, regs = ptxas_lines(log, sym)
        print("%s\n  ptxas: %s | %s" % (name, frame, regs))
        print("  STL %d  LDL %d  CALL %d (%d to the most-called target)  BAR %d  body %d instructions (%d B)"
              % (ops["STL"], ops["LDL"], sum(calls.values()), max(calls.values(), default=0), ops["BAR"],
                 body // 16, body))
    print("traversal kernels (SHA-256 of the SASS):")
    for sym in sorted(s for s in funcs if TRAVERSAL.match(s)):
        text = "\n".join("%x %s %s %s" % i for i in funcs[sym])
        print("  %s  %s" % (hashlib.sha256(text.encode()).hexdigest()[:16], sym))


if __name__ == "__main__":
    main()

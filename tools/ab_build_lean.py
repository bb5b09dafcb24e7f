#!/usr/bin/env python3
"""A/B build of the lean traversal kernel's translation unit with extra -D flags into ab/<tag>.so (the other objects
come from the regular build):   python tools/ab_build_lean.py <tag> [-DFOO=1 ...]   then YART_LIB_PATH=ab/<tag>.so."""
import importlib, subprocess, sys
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
b = importlib.import_module("yet-another-raytracer_b200.build")
b.build()
(ROOT/'ab').mkdir(exist_ok=True)
tag, flags = sys.argv[1], sys.argv[2:]
obj = ROOT/'ab'/(tag+'_lean.o')
cmd=[b.nvcc_path()]+b.COMPILE_FLAGS+flags+['-Xptxas','-v','-c',str(b.CSRC/'device_trace_lean.cu'),'-o',str(obj)]
r=subprocess.run(cmd,capture_output=True,text=True)
if r.returncode: print(r.stderr[-2000:]); sys.exit(1)
txt=r.stdout+r.stderr
lines=txt.splitlines()
for i,l in enumerate(lines):
    if 'k_traverse_leanILi24E' in l and 'Compiling' in l: print(lines[i+2].strip(), '|', lines[i+3].strip())
others=[str(b.OBJ_DIR/(s.replace('.','_')+'.o')) for s in b.SOURCES if s!='device_trace_lean.cu']
lib=ROOT/'ab'/(tag+'.so')
r2=subprocess.run([b.nvcc_path()]+b.LINK_FLAGS+['-o',str(lib),str(obj)]+others,capture_output=True,text=True)
print('link', r2.returncode, r2.stderr[-500:]); obj.unlink()

"""Build the A/B variants of the library (compile-time experiments, DESIGN.md section 7) into ab/ -- run HERE, before a
gpurun call (ab/ is git-ignored but travels to the GPU box); select one with IEVM_LIB_PATH=ab/lib_<name>.so.
    python scripts/build_ab.py [name ...]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ievm_b200 import _lib

VARIANTS = {"halfk": ["IEVM_EXP_HALFK"], "interleave": ["IEVM_EXP_INTERLEAVE"],
            "interleave_halfk": ["IEVM_EXP_INTERLEAVE", "IEVM_EXP_HALFK"], "scalar_epi": ["IEVM_EXP_SCALAR_EPI"]}
os.makedirs(os.path.join(_lib.ROOT, "ab"), exist_ok=True)
for name in (sys.argv[1:] or VARIANTS):
    print(_lib.build(defines=VARIANTS[name], out=os.path.join(_lib.ROOT, "ab", f"lib_{name}.so")))

"""Build an A/B variant of libabcgpt.so: extra nvcc flags (usually -D switches) for selected sources, output next to the
product library as libabcgpt_<name>.so.  Select it at run time with ABCGPT_LIB=<path> (ai_music_generation_b200/_C.py).

    python tools/build_variant.py NAME "-DABCGPT_NO_PDL" gemm.cu [attn.cu ...]
"""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ai_music_generation_b200 import build as B  # noqa: E402

name, flags, srcs = sys.argv[1], sys.argv[2].split(), sys.argv[3:]
B.build()  # product objects are up to date
out_dir = os.path.join(B.OBJ_DIR, "variant_" + name)
os.makedirs(out_dir, exist_ok=True)
objs = []
for src in B.SOURCES:
    if src in srcs:
        obj = os.path.join(out_dir, src.replace(".cu", ".o"))
        cmd = [B._nvcc(), *[f for f in B.NVCC_FLAGS if f not in ("-Xptxas", "-v")], *flags, "-c", os.path.join(B.CSRC, src), "-o", obj]
        subprocess.run(cmd, check=True)
    else:
        obj = os.path.join(B.OBJ_DIR, src.replace(".cu", ".o"))
    objs.append(obj)
path = os.path.join(B.HERE, f"libabcgpt_{name}.so")
subprocess.run([B._nvcc(), "-shared", "-o", path, *objs, "-lcudart"], check=True)
print(path)

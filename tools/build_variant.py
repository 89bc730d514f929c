"""Build a timing / A-B variant of libriser_b200.so with extra nvcc flags into build_ab/ (git-ignored).  Select it at
run time with RISER_B200_LIB=build_ab/<name>.so.  Run in a checkout of another commit, it builds that commit's
library, which can then be copied into this tree's build_ab/ and timed against it, alternating RISER_B200_LIB.

  python tools/build_variant.py parent                 (the sources of this checkout, default flags)
  python tools/build_variant.py maxreg -maxrregcount=128
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from riser_b200 import build as b  # noqa: E402


def main():
    name, flags = sys.argv[1], sys.argv[2:]
    out_dir = os.path.join(ROOT, "build_ab")
    os.makedirs(out_dir, exist_ok=True)
    objs = []
    procs = []
    for src in b.SOURCES:
        o = os.path.join(out_dir, f"{name}_{src.replace('.cu', '.o')}")
        procs.append(subprocess.Popen(["nvcc"] + b.NVCC_FLAGS + flags + ["-c", os.path.join(b.CSRC, src), "-o", o]))
        objs.append(o)
    for p in procs:
        if p.wait():
            raise SystemExit("nvcc failed")
    lib = os.path.join(out_dir, f"{name}.so")
    subprocess.run(["nvcc"] + b.NVCC_FLAGS + ["-shared", "-o", lib] + objs + ["-lrt", "-ldl", "-lpthread"], check=True)
    for o in objs:
        os.remove(o)
    print(lib)


if __name__ == "__main__":
    main()

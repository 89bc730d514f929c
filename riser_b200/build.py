"""Build libriser_b200.so (the C-ABI library, include/riser_b200.h) in-tree with nvcc
for sm_100a.  No torch headers, no JIT: the .so travels to the GPU box with the repo
snapshot.  ``python -m riser_b200.build`` or ``riser_b200.build.build()``."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libriser_b200.so")
SOURCES = ["preprocess.cu", "normalise_f32.cu", "normalise_long.cu", "polya_f32.cu", "convnet.cu", "resnet.cu", "resnet_tc.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-cudart", "static"]


def _newer(target, deps):
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(d) <= t for d in deps)


def build_hostpack(force=False):
    """gcc -> riser_b200/_hostpack<EXT_SUFFIX>: the CPython module that gathers a poll's read prefixes into the
    pinned staging buffer (csrc/hostpack.c; buffer protocol + pthreads, no third-party headers)."""
    import sysconfig
    src = os.path.join(CSRC, "hostpack.c")
    out = os.path.join(HERE, "_hostpack" + sysconfig.get_config_var("EXT_SUFFIX"))
    if force or not _newer(out, [src]):
        subprocess.run([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-pthread", "-I",
                        sysconfig.get_paths()["include"], src, "-o", out], check=True)
    return out


def build(force=False, verbose=False):
    build_hostpack(force)
    nvcc = os.environ.get("NVCC", "nvcc")
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "riser_b200.h"))
    objs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        if not os.path.exists(s):
            continue
        o = os.path.join(CSRC, src.replace(".cu", ".o"))
        if force or not _newer(o, [s] + headers):
            cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            subprocess.run(cmd, check=True)
        objs.append(o)
    if force or not _newer(LIB, objs):
        subprocess.run([nvcc] + NVCC_FLAGS + ["-shared", "-o", LIB] + objs + ["-lrt", "-ldl", "-lpthread"],
                       check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

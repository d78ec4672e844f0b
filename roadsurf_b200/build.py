"""Builds libroadsurf_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, os.environ.get("ROADSURF_B200_LIBNAME", "libroadsurf_b200.so"))
SOURCES = ("rs_kernel.cu", "rs_host.cu", "rs_ensemble.cu", "rs_model.cpp")

# -fmad=false: no FMA contraction, like a generic x86-64 gfortran build of the reference, so that
# threshold decisions (freeze/melt limits, minimum storages) are taken on identically rounded values.
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-fmad=false", "-Xcompiler", "-fPIC,-ffp-contract=off", "-shared", "-cudart", "static"]


def nvcc_path():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(HERE, "..", "include", "roadsurf_b200.h"))
    deps.append(os.path.abspath(__file__))
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False):
    """Compile every CUDA source of the package into roadsurf_b200/libroadsurf_b200.so."""
    if not force and not needs_build():
        return LIB
    cmd = [nvcc_path()] + NVCC_FLAGS + os.environ.get("ROADSURF_B200_NVCC_EXTRA", "").split()
    if verbose:
        cmd += ["-Xptxas", "-v"]
    cmd += ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stdout + r.stderr)
    return LIB


if __name__ == "__main__":
    import sys
    print(build_library(force=True, verbose="-v" in sys.argv))

"""Build the in-tree native libraries with nvcc for sm_100a (no JIT cache: the .so files travel with the tree)."""
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libh2v.so")
HOSTCHECK = os.path.join(PKG, "libh2v_hostcheck.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _sources():
    out = [os.path.join(ROOT, "include", "h2v.h")]
    for f in sorted(os.listdir(CSRC)):
        if f.endswith((".cu", ".cuh", ".h", ".hpp")):
            out.append(os.path.join(CSRC, f))
    return out


def build(force=False, verbose=False):
    srcs = _sources()
    nvcc = os.environ.get("NVCC", "nvcc")
    if force or _newer(LIB, srcs):
        # the translation units (kernels + ABI, prover, circuit builder, mock prover, witness generation) compiled side by side; -split-compile 0: ptxas works on the
        # kernels of one unit in parallel (4.5 min -> 2 min on 8 cores), same code
        common = [nvcc, "-Xcompiler", "-fPIC", "-O3", "-std=c++17", "-lineinfo", "-split-compile", "0", *ARCH,
                  "-I" + os.path.join(ROOT, "include"), "-I" + CSRC]
        if verbose:
            common.insert(1, "-Xptxas=-v")
        os.makedirs(os.path.join(PKG, "build"), exist_ok=True)
        procs, objs = [], []
        for unit in ("h2v", "prover", "circuit", "mock", "witness"):
            src, obj = os.path.join(CSRC, unit + ".cu"), os.path.join(PKG, "build", unit + ".o")
            objs.append(obj)
            deps = [s_ for s_ in srcs if not s_.endswith(".cu")] + [src]
            if force or _newer(obj, deps):
                cmd = common + ["-c", "-o", obj, src]
                if verbose:
                    print(" ".join(cmd))
                procs.append((cmd, subprocess.Popen(cmd)))
        for cmd, p in procs:
            if p.wait() != 0:
                raise subprocess.CalledProcessError(p.returncode, cmd)
        subprocess.check_call([nvcc, "-shared", *ARCH, "-o", LIB, *objs])
    if force or _newer(HOSTCHECK, srcs):
        cmd = [nvcc, "-shared", "-Xcompiler", "-fPIC", "-O2", "-std=c++17", "-Wno-deprecated-gpu-targets",
               "-I" + CSRC, "-o", HOSTCHECK, os.path.join(CSRC, "hostcheck.cu")]
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(LIB)

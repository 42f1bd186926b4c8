"""In-tree build of the CUDA extension (sm_100a only)."""
import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
INCLUDE = os.path.join(os.path.dirname(PKG_DIR), "include")
LIB = os.path.join(CSRC, "libpve_mcc.so")
SOURCES = [os.path.join(CSRC, "pve_mcc.cu"), os.path.join(CSRC, "scene_step.cuh"), os.path.join(CSRC, "scene_step4.cuh"), os.path.join(CSRC, "actor.cuh"),
           os.path.join(CSRC, "actor_mma.cuh"), os.path.join(CSRC, "nstep.cuh"), os.path.join(CSRC, "critic_mma.cuh"), os.path.join(CSRC, "mlp_tc5.cuh"), os.path.join(CSRC, "arrivals.cuh"),
           os.path.join(INCLUDE, "pve_mcc.h")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              # float64 state must follow the reference's two-rounding a*b+c (no FMA contraction)
              "-fmad=false",
              "-shared", "-Xcompiler", "-fPIC"]


def find_nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def build_cuda(force=False, verbose=False):
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> csrc/libpve_mcc.so"""
    if (not force and os.path.exists(LIB)
            and os.path.getmtime(LIB) >= max(os.path.getmtime(f) for f in SOURCES)):
        return LIB
    cmd = [find_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          ["-I", INCLUDE, "-I", CSRC, SOURCES[0], "-o", LIB]
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout)
    if verbose:
        print(res.stdout)
    return LIB

"""TEST INFRASTRUCTURE: compiles ngp_oracle.c with gcc into oracle/_build/libngp_oracle.so."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "ngp_oracle.c")
OUT_DIR = os.path.join(HERE, "_build")
LIB = os.path.join(OUT_DIR, "libngp_oracle.so")

# -ffp-contract=off: the oracle spells out every fused multiply-add the device performs with fmaf().
CFLAGS = ["-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-fno-fast-math"]


def build(force=False):
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= os.path.getmtime(SRC):
        return LIB
    os.makedirs(OUT_DIR, exist_ok=True)
    subprocess.check_call(["gcc"] + CFLAGS + ["-o", LIB, SRC, "-lm"])
    return LIB


# the reference kernels a host cannot reproduce (device intrinsics), each with the flags its comment gives
CUDA_SRCS = {"ref_freq.cu": ["--use_fast_math"], "ref_raymarching.cu": ["-fmad=false"]}
CUDA_LIB = os.path.join(OUT_DIR, "libngp_ref_device.so")
CUDA_ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def build_cuda(force=False):
    """ref_freq.cu and ref_raymarching.cu with nvcc into oracle/_build/libngp_ref_device.so."""
    srcs = [os.path.join(HERE, s) for s in CUDA_SRCS]
    if not force and os.path.exists(CUDA_LIB) and os.path.getmtime(CUDA_LIB) >= max(os.path.getmtime(s) for s in srcs):
        return CUDA_LIB
    os.makedirs(OUT_DIR, exist_ok=True)
    objs = []
    for src, flags in zip(srcs, CUDA_SRCS.values()):
        obj = os.path.join(OUT_DIR, os.path.basename(src) + ".o")
        subprocess.check_call(["nvcc", "-c", "-O3", "-Xcompiler", "-fPIC", "-o", obj, src] + CUDA_ARCH + flags)
        objs.append(obj)
    subprocess.check_call(["nvcc", "-shared", "-o", CUDA_LIB] + objs + CUDA_ARCH)
    return CUDA_LIB

"""Build libtdsfs.so (hand-written CUDA for sm_100a) in-tree with nvcc.

The shared library is the product's only compute path; it travels to the GPU box with the
repository snapshot (git-ignored, not gpurun-ignored)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "lib", "libtdsfs.so")
PACKER = os.path.join(HERE, "lib", "libtdsfs_pack.so")
DICTCONV = os.path.join(HERE, "lib", "libtdsfs_dictconv.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-shared",
              "-Xcompiler", "-fPIC", "-diag-suppress", "1886"]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def build(force=False, verbose=False):
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    cuda_src = [os.path.join(SRC, "tdsfs.cu"), os.path.join(SRC, "tdsfs_kernels.cuh"), os.path.join(SRC, "tdsfs_fused.cuh"),
                os.path.join(SRC, "tdsfs_diversity.cuh"), os.path.join(SRC, "tdsfs_ld.cuh"),
                os.path.join(HERE, "..", "include", "tdsfs.h")]
    if force or _newer(LIB, cuda_src):
        nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB, cuda_src[0]]
        subprocess.check_call(cmd)
    pack_src = os.path.join(SRC, "vcf_pack.cpp")
    if os.path.exists(pack_src) and (force or _newer(PACKER, [pack_src])):
        subprocess.check_call(["g++", "-O3", "-std=c++17", "-shared", "-fPIC", "-pthread", "-o", PACKER, pack_src, "-lz"])
    conv_src = os.path.join(SRC, "dictconv.c")
    if os.path.exists(conv_src) and (force or _newer(DICTCONV, [conv_src])):
        import sysconfig
        subprocess.check_call(["gcc", "-O2", "-shared", "-fPIC", "-I" + sysconfig.get_paths()["include"], "-o", DICTCONV, conv_src])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

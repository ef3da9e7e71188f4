"""Build libcgl_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python ecen743-project-cgol_b200/build.py [--force] [--verbose]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libcgl_b200.so")
SOURCES = ["cgl_api.cu", "cgl_env.cu", "cgl_env_run.cu", "cgl_env_lookahead.cu", "cgl_sim1.cu", "cgl_rollout.cu", "cgl_life.cu", "cgl_life_tb.cu"]
HEADERS = ["cgl_bits.cuh", "cgl_internal.cuh", os.path.join("..", "..", "include", "cgl_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--use_fast_math", "-Xcompiler", "-fPIC", "-shared", "-cudart", "static"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    deps += [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + srcs
    env = dict(os.environ)
    env.pop("CC", None), env.pop("CXX", None)      # the image's default CC has no libstdc++ headers for nvcc
    r = subprocess.run(cmd, capture_output=True, text=True, env=env)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building libcgl_b200.so")
    if verbose:
        sys.stderr.write(r.stdout + r.stderr)
    return LIB


EXT_SRC = os.path.join(HERE, "csrc_ext", "cgl_torch_ext.cpp")
EXT_LIB = os.path.join(HERE, "cgl_b200", "_cgl_ext.so")


def build_ext(force=False):
    """The thin PyTorch C++ extension (csrc_ext/cgl_torch_ext.cpp -> cgl_b200/_cgl_ext.so): g++ against torch's
    headers, linked to libcgl_b200.so through an $ORIGIN rpath.  In-tree, so it travels with the gpurun snapshot."""
    import sysconfig
    build()
    deps = [EXT_SRC, os.path.join(HERE, "..", "include", "cgl_b200.h"), os.path.abspath(__file__)]
    if not force and os.path.exists(EXT_LIB) and all(os.path.getmtime(d) <= os.path.getmtime(EXT_LIB) for d in deps):
        return EXT_LIB
    import torch
    from torch.utils import cpp_extension as ce
    inc = ce.include_paths() + [sysconfig.get_paths()["include"], "/usr/local/cuda/include"]
    libdir = ce.library_paths()[0]
    abi = int(torch._C._GLIBCXX_USE_CXX11_ABI)
    cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-DTORCH_EXTENSION_NAME=_cgl_ext", "-DTORCH_API_INCLUDE_EXTENSION_H",
           f"-D_GLIBCXX_USE_CXX11_ABI={abi}", "-Wno-deprecated-declarations"]
    cmd += [f"-I{i}" for i in inc] + [EXT_SRC, "-o", EXT_LIB, f"-L{libdir}", f"-L{HERE}", "-lcgl_b200", "-ltorch_python",
                                     "-ltorch", "-ltorch_cpu", "-lc10", "-lc10_cuda",
                                     "-Wl,-rpath,$ORIGIN/..", f"-Wl,-rpath,{libdir}"]
    env = dict(os.environ)
    env.pop("CC", None), env.pop("CXX", None)
    r = subprocess.run(cmd, capture_output=True, text=True, env=env)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("g++ failed building cgl_b200/_cgl_ext.so")
    return EXT_LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
    if "--ext" in sys.argv:
        print(build_ext(force="--force" in sys.argv))

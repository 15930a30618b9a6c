"""Compile libcube_b200.so for sm_100a with nvcc (in-tree, so it travels to the GPU box).

    python rubiks_cube_solver_b200/csrc/build.py [--force] [--verbose]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
LIB = os.path.join(PKG, "libcube_b200.so")
SOURCES = ["scramble.cu", "prefix.cu", "walk.cu", "launch.cu", "expand.cu", "leaf.cu", "decode.cu", "adi.cu", "seeds.cu", "mcts.cu", "pipeline.cu", "envhost.cu", "peer.cu", "distance.cu", "abi.cu"]
HEADERS = ["cube_common.cuh", "cube_threads.cuh", "cube_bulk.cuh", "cube_sched.cuh", "cube_launch.cuh", "cube_tables.cuh", "cube_distance.cuh", "cube_seeds.cuh", "cube_kernels.h", os.path.join("..", "..", "include", "cube_b200.h")]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-shared"]


def nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(HERE, f)) > t
               for f in SOURCES + HEADERS if os.path.exists(os.path.join(HERE, f)))


def build(force=False, verbose=False):
    """One object per source (compiled in parallel, rebuilt only when the source or a header is newer),
    then one link.  Objects live in csrc/build/ (git-ignored)."""
    from concurrent.futures import ThreadPoolExecutor
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(HERE, s))]
    if not force and not stale():
        return LIB
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    hdr_t = max(os.path.getmtime(os.path.join(HERE, h)) for h in HEADERS + ["build.py"] if os.path.exists(os.path.join(HERE, h)))
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"] + (["-Xptxas", "-v"] if verbose else [])

    def compile_one(src):
        obj = os.path.join(objdir, src[:-3] + ".o")
        if not force and os.path.exists(obj) and os.path.getmtime(obj) > max(hdr_t, os.path.getmtime(os.path.join(HERE, src))):
            return obj
        tmp_o = obj + ".tmp%d" % os.getpid()
        try:
            subprocess.check_call([nvcc()] + compile_flags + ["-c", "-o", tmp_o, src], cwd=HERE)
            os.replace(tmp_o, obj)
        finally:
            if os.path.exists(tmp_o):
                os.remove(tmp_o)
        return obj

    with ThreadPoolExecutor(max_workers=min(len(srcs), os.cpu_count() or 4)) as pool:
        objs = list(pool.map(compile_one, srcs))
    tmp = LIB + ".tmp%d" % os.getpid()                     # never leave a half-written library in the tree
    try:
        subprocess.check_call([nvcc()] + NVCC_FLAGS + ["-o", tmp] + objs, cwd=HERE)
        os.replace(tmp, LIB)
    finally:
        if os.path.exists(tmp):
            os.remove(tmp)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))

"""Builds the CUDA extension in-tree: predpreygrass_b200/libppg_b200.so (sm_100a only).

nvcc cross-compiles without a GPU; the .so is git-ignored but travels with the tree to the GPU box.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libppg_b200.so")
SOURCES = ["ppg_base.cu", "ppg_eco.cu", "ppg_stag.cu", "ppg_obs.cu", "ppg_world.cu", "ppg_returns.cu", "ppg_api.cu"]
HEADERS = ["ppg_device.cuh", "ppg_step_common.cuh", os.path.join("..", "..", "include", "ppg.h"), os.path.join("..", "..", "include", "ppg_philox.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "--fmad=false",
]


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    from concurrent.futures import ThreadPoolExecutor

    def compile_one(src):
        obj = os.path.join(CSRC, src[:-3] + ".o")
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        subprocess.check_call(cmd)
        return obj

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as ex:  # one nvcc per translation unit
        objs = list(ex.map(compile_one, SOURCES))
    subprocess.check_call([nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

"""Build the in-tree libraries (git-ignored, but they travel to the GPU box):

  liblfr_b200.so  the product: CUDA kernels + the C ABI of include/lfr.h      (nvcc, sm_100a; cross-compiles without a GPU)
  liblfr_host.so  CPU-only host utilities behind include/lfr_wire.h and include/lfr_host.h
                  (protobuf wire codec, host graph stage) — no CUDA dependency, so the
                  reference arm of bench.py and the tests can use them without mapping the product library
  multi-view-refinement/build/solve_native
                  the native drop-in executable (lfr_solve_main.cc), linked against the two libraries
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "liblfr_b200.so")
OUT_HOST = os.path.join(HERE, "liblfr_host.so")
SOURCES = ["lfr_capi.cu"]
HOST_SOURCES = ["lfr_wire.cc", "lfr_host.cc"]
EXE_SOURCE = "lfr_solve_main.cc"
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT_EXE = os.path.join(ROOT, "multi-view-refinement", "build", "solve_native")
INC = os.path.join("..", "..", "include")
DEPS = SOURCES + ["lfr_solve_warp.cuh", "lfr_solve_warp2.cuh", "lfr_solve_cta.cuh", "lfr_solve_tile.cuh", "lfr_math.cuh",
                  os.path.join(INC, "lfr.h")]
HOST_DEPS = HOST_SOURCES + ["lfr_cut.h", os.path.join(INC, "lfr.h"), os.path.join(INC, "lfr_wire.h"),
                            os.path.join(INC, "lfr_host.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "-cudart", "shared"]


def _stale(out, deps):
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(os.path.join(HERE, d)) > t for d in deps)


def build_host(force: bool = False) -> str:
    if force or _stale(OUT_HOST, HOST_DEPS):
        subprocess.check_call(["g++", "-std=c++17", "-O3", "-fPIC", "-shared", "-pthread", "-Wall", "-o", OUT_HOST] +
                              [os.path.join(HERE, s) for s in HOST_SOURCES])
    return OUT_HOST


def build_exe(force: bool = False, out: str = OUT_EXE, solve_lib_dir: str = HERE, solve_lib: str = "lfr_b200") -> str:
    """The native `solve`.  The product links csrc/liblfr_b200.so; tests/ link the same source against the
    CPU checker (oracle/liblfr_ref.so exports the same C ABI) to compare it with the reference binary."""
    deps = [EXE_SOURCE, os.path.join(INC, "lfr.h"), os.path.join(INC, "lfr_wire.h"), os.path.join(INC, "lfr_host.h")]
    if force or _stale(out, deps) or not os.path.exists(out):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-o", out, os.path.join(HERE, EXE_SOURCE),
                               "-L" + solve_lib_dir, "-l" + solve_lib, "-L" + HERE, "-llfr_host",
                               # found next to the checkout wherever it is mounted, then by absolute path
                               "-Wl,-rpath,$ORIGIN/../../local-feature-refinement_b200/csrc",
                               "-Wl,-rpath," + solve_lib_dir, "-Wl,-rpath," + HERE])
    return out


def build(force: bool = False, verbose: bool = False) -> str:
    build_host(force)
    _build_cuda(force, verbose)
    build_exe(force)
    return OUT


def _build_cuda(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale(OUT, DEPS):
        return OUT
    cmd = [NVCC] + NVCC_FLAGS + ["-o", OUT] + [os.path.join(HERE, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

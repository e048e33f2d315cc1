"""Builds the CUDA extension in-tree: stratego_env_b200/csrc/libstratego_b200.so (sm_100a only)."""
import os
import shutil
import subprocess

CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc")
LIB_PATH = os.path.join(CSRC, "libstratego_b200.so")
SOURCES = ["sx_kernels.cu", "sx_policy.cu", "sx_alloc.cu", "sx_hidden.cu", "sx_expand.cu", "sx_playout.cu", "sx_keys.cu", "sx_search.cu",
           "sx_guided.cu"]
HEADERS = ["sx_device.cuh", "sx_toy.cuh", os.path.join("..", "..", "include", "stratego_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the B200 Stratego engine has no CPU fallback and cannot be built")


def dependencies():
    """every file the library is built from: the listed ones plus anything else matching csrc/*.cu* (so a new header
    can never be forgotten here)"""
    import glob
    deps = {os.path.normpath(os.path.join(CSRC, f)) for f in SOURCES + HEADERS}
    deps.update(os.path.normpath(f) for f in glob.glob(os.path.join(CSRC, "*.cu*")))
    return sorted(deps)


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(d) > built for d in dependencies())


def build_extension(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB_PATH
    tmp = LIB_PATH + ".tmp.%d" % os.getpid()
    cmd = [_nvcc(), *NVCC_FLAGS, *(["-Xptxas", "-v"] if verbose else []), "-o", tmp,
           *[os.path.join(CSRC, s) for s in SOURCES]]
    subprocess.run(cmd, check=True, cwd=CSRC)
    os.replace(tmp, LIB_PATH)
    return LIB_PATH


if __name__ == "__main__":
    print(build_extension(force=True, verbose=True))

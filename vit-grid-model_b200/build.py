"""Build libvitgrid.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

nvcc cross-compiles without a GPU, so this runs in the CPU-only build container; the resulting .so is
git-ignored but travels to the GPU box with the repository snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(HERE, "libvitgrid.so")
SOURCES = ["vg_api.cu", "vg_gemm.cu", "vg_mem.cu", "vg_attn.cu", "vg_attn_fused2.cu", "vg_attn_bwd_tc.cu", "vg_wgrad.cu", "vg_bwd.cu", "vg_bwd_vit.cu", "vg_eval.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libvitgrid.so cannot be built (there is no CPU fallback)")


def have_nvcc() -> bool:
    try:
        _nvcc()
        return True
    except RuntimeError:
        return False


def _newest_source_mtime() -> float:
    files = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "vitgrid.h")]
    return max(os.path.getmtime(f) for f in files if os.path.isfile(f))


def is_stale() -> bool:
    return not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < _newest_source_mtime()


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB_PATH
    nvcc = _nvcc()
    import fcntl
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    with open(os.path.join(HERE, "build", ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)                # one builder at a time (torchrun ranks share the tree)
        if not force and not is_stale():                # another process built it while this one waited
            return LIB_PATH
        return _build_locked(nvcc, verbose)


def _build_locked(nvcc: str, verbose: bool) -> str:
    objdir = os.path.join(HERE, "build", f"obj.{os.getpid()}")
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src: str) -> str:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    tmp = f"{LIB_PATH}.{os.getpid()}.tmp"
    r = subprocess.run([nvcc, "-shared", "-o", tmp, *objs, "-cudart", "static"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, LIB_PATH)
    shutil.rmtree(objdir, ignore_errors=True)
    return LIB_PATH


if __name__ == "__main__":
    import sys
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))

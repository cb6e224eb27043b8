"""Builds libdisenlink_b200.so in-tree with nvcc for sm_100a (no torch headers involved).

    python -m disenlink_b200.build [--force] [--verbose]
    python -m disenlink_b200.build --variant NAME SRC.cu -DFOO=1 ...   (-> _variants/lib_NAME.so)

The library is plain CUDA behind a C ABI (include/disenlink_b200.h); Python reaches it with ctypes.
The .so is git-ignored but travels to the GPU box with the working tree.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ_DIR = os.path.join(HERE, "_obj")
LIB = os.path.join(HERE, "libdisenlink_b200.so")
VARIANT_DIR = os.path.join(HERE, "_variants")
SOURCES = ["graph_build.cu", "factor_fwd.cu", "attn_stream.cu", "attn_fl.cu", "attn_sym.cu", "gather_stream.cu", "bwd_stream.cu", "bwd_fl.cu", "bwd_sym.cu", "slice_gather.cu", "factor_bwd.cu", "bwd_dir.cu",
           "pair_score.cu", "pair_stream.cu", "link_loss.cu", "eval_metrics.cu", "sampling.cu", "peer_copy.cu", "dense_compat.cu", "feat_proj.cu"]
HEADERS = [os.path.join(CSRC, h) for h in ("dl_common.cuh", "dl_dispatch.cuh", "dl_stream.cuh", "dl_fl.cuh", "dl_prims.cuh")] + [
    os.path.join(os.path.dirname(HERE), "include", "disenlink_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--fmad=false", "-Xptxas", "-v", "-Wno-deprecated-declarations"]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found; libdisenlink_b200.so cannot be built")


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _ccbin():
    # pin the system host compiler when present (CC/CXX may name wrappers nvcc cannot use as host compiler)
    return ["-ccbin", "/usr/bin/g++"] if os.path.exists("/usr/bin/g++") else []


def _compile(nvcc, src, obj, log, extra=(), verbose=False):
    cmd = [nvcc] + _ccbin() + NVCC_FLAGS + list(extra) + ["-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    with open(log, "w") as f:
        f.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
    if verbose:
        print(r.stderr)


def _link(nvcc, out, objs):
    cmd = [nvcc] + _ccbin() + ["-shared", "-o", out] + objs + ["-lcudart", "-Xlinker", "-z", "-Xlinker", "defs"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        if force or _stale(obj, [os.path.join(CSRC, src)] + HEADERS):
            _compile(nvcc, src, obj, os.path.join(OBJ_DIR, src.replace(".cu", ".ptxas.log")), verbose=verbose)
        return obj

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or _stale(LIB, objs):
        _link(nvcc, LIB, objs)
    return LIB


def build_variant(name: str, src: str, defines, force: bool = False) -> str:
    """_variants/lib_NAME.so: the regular objects with SRC recompiled under extra -D flags (A/B experiments,
    debug builds).  Load it with DL_LIB_PATH or ctypes; requires build() first."""
    nvcc = _nvcc()
    os.makedirs(VARIANT_DIR, exist_ok=True)
    stem = src.replace(".cu", "")
    obj = os.path.join(VARIANT_DIR, f"{name}_{stem}.o")
    lib = os.path.join(VARIANT_DIR, f"lib_{name}.so")
    stamp = obj + ".flags"                     # the -D flags the object was compiled with
    flags = " ".join(defines)
    same_flags = os.path.exists(stamp) and open(stamp).read() == flags
    if force or not same_flags or _stale(obj, [os.path.join(CSRC, src)] + HEADERS):
        _compile(nvcc, src, obj, os.path.join(VARIANT_DIR, f"{name}.ptxas.log"), extra=defines)
        with open(stamp, "w") as f:
            f.write(flags)
    objs = [obj] + [os.path.join(OBJ_DIR, s.replace(".cu", ".o")) for s in SOURCES if s != src]
    if force or _stale(lib, objs):
        _link(nvcc, lib, objs)
    return lib


if __name__ == "__main__":
    if len(sys.argv) > 3 and sys.argv[1] == "--variant":
        build()
        print(build_variant(sys.argv[2], sys.argv[3], sys.argv[4:], force=True))
    else:
        print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))

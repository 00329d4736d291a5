"""Build the CUDA C-ABI library in-tree with nvcc for sm_100a (no torch in the link).

    python -m brl_b200.build            # -> brl_b200/lib/libbrl_b200.so

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIB_DIR, "libbrl_b200.so")
SOURCES = ["brl_env.cu", "brl_algo.cu", "brl_mlp.cu", "brl_mlp_train.cu", "brl_ppo.cu", "brl_eval.cu", "brl_sl.cu", "brl_cv.cu", "brl_match.cu", "brl_posterior.cu", "brl_host.cu", "xla_ffi_shim.cc"]
NVCC_FLAGS = [
    "-std=c++17", "-O3", "-lineinfo",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-Xcompiler", "-fPIC,-O3,-Wall",
    "-cudart", "static",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; cannot build brl_b200 (there is no CPU fallback)")


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "brl_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.isfile(d))


def _xla_ffi_include():
    """-I for the typed XLA FFI handlers, if jaxlib happens to be installed (it is not in this image)."""
    try:
        import jaxlib  # noqa: F401
        inc = os.path.join(os.path.dirname(jaxlib.__file__), "include")
        if os.path.exists(os.path.join(inc, "xla", "ffi", "api", "ffi.h")):
            return ["-I", inc]
    except Exception:
        pass
    return []


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile and link in-tree.  Concurrent callers (torchrun ranks that all see a stale library) are serialised by
    an exclusive file lock: the first one builds, the others wake up to a fresh library and return.  Objects go to a
    per-process directory and the library is moved into place with os.replace, so nobody ever dlopens a half-written file."""
    if not force and not _stale():
        return LIB
    os.makedirs(LIB_DIR, exist_ok=True)
    import fcntl
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not _stale():
                return LIB
            return _build_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose: bool) -> str:
    nvcc = _nvcc()
    objs = []
    procs = []
    obj_dir = os.path.join(LIB_DIR, f"obj.{os.getpid()}")
    os.makedirs(obj_dir, exist_ok=True)
    tmp_lib = os.path.join(obj_dir, "libbrl_b200.so")
    try:
        return _compile_and_link(nvcc, obj_dir, tmp_lib, objs, procs, verbose)
    finally:
        shutil.rmtree(obj_dir, ignore_errors=True)


def _compile_and_link(nvcc, obj_dir, tmp_lib, objs, procs, verbose):
    for src in SOURCES:
        obj = os.path.join(obj_dir, os.path.splitext(src)[0] + ".o")
        cmd = [nvcc, *NVCC_FLAGS, *_xla_ffi_include(), "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose:
            print(out)
    link = [nvcc, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp_lib, *objs]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    os.replace(tmp_lib, LIB)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

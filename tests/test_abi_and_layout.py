"""CPU: the C-ABI library loads and exports every symbol include/brl_b200.h declares
(no compute calls without a GPU); the product never imports the oracle; product ops
fail loudly without CUDA."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "brl_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(brl_[a-z0-9_]+)\s*\(", hdr)) - {"brl_op_fn"})


def test_header_symbols_are_all_exported():
    from brl_b200 import _lib
    L = _lib.load()
    names = _declared_symbols()
    assert len(names) >= 20
    for name in names:
        assert hasattr(L, name), f"{name} declared in include/brl_b200.h but not exported"
    assert set(_lib.ALL_SYMBOLS) == set(names)
    assert L.brl_abi_version() == _lib.ABI_VERSION == 3


def test_params_struct_matches_header():
    from brl_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "brl_b200.h")).read()
    body = re.search(r"typedef struct BrlParams \{(.*?)\} BrlParams;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = re.findall(r"\b(\w+);", body)
    assert fields == [f[0] for f in _lib.BrlParams._fields_]
    assert ctypes.sizeof(_lib.BrlParams) == 64


def test_usage_errors_are_reported_without_a_gpu():
    """Argument validation happens before any CUDA call, so it is testable here."""
    from brl_b200 import _lib
    L = _lib.load()
    p = _lib.BrlParams(4, 0, 4, 0, 10, 0, 0, 0, -1.0, 1.0, 0.0, 0.0)
    bufs = (ctypes.c_void_p * 10)()
    rc = L.brl_step(None, bufs, ctypes.byref(p), ctypes.sizeof(p))
    assert rc == -2 and b"NULL" in L.brl_last_error()
    rc = L.brl_step(None, bufs, ctypes.byref(p), 12)
    assert rc == -1 and b"BrlParams" in L.brl_last_error()
    with pytest.raises(_lib.BrlError):
        _lib.call("brl_gae", 0, [None] * 6, p)


def test_ppo_update_ops_validate_their_arguments_without_a_gpu():
    """brl_ppo_grad / brl_mlp_adam_step / brl_mlp_pack_train reject bad calls before any CUDA work; the size queries are
    pure host arithmetic."""
    from brl_b200 import _lib
    L = _lib.load()
    n = L.brl_mlp_num_params()
    assert n == 480 * 1024 + 1024 + 3 * (1024 * 1024 + 1024) + 1024 * 38 + 38 + 1024 + 1 == 3681319
    # per layer W[in, out_pad] as bf16 hi + lo, fp32 bias, 256-byte aligned sections
    assert L.brl_mlp_train_blob_bytes() == sum(((2 * k * m * 2 + 4 * m + 255) // 256) * 256
                                               for k, m in ((480, 1024), (1024, 1024), (1024, 1024), (1024, 1024), (1024, 64)))
    assert L.brl_mlp_train_scratch_bytes(0) == 0
    assert 0 < L.brl_mlp_train_scratch_bytes(64) < L.brl_mlp_train_scratch_bytes(1024) < L.brl_mlp_train_scratch_bytes(4096)
    assert 0 < L.brl_mlp_train_trace_offset(1024) < L.brl_mlp_train_scratch_bytes(1024)
    bufs = (ctypes.c_void_p * 13)()
    pp = _lib.BrlPpoParams(1024, 4096, 0.2, 0.01, 0.5, 0.0, _lib.PPO_VALUE_CLIPPING, 0)
    assert L.brl_ppo_grad(None, bufs, ctypes.byref(pp), ctypes.sizeof(pp)) == -2 and b"'obs' is NULL" in L.brl_last_error()
    assert L.brl_ppo_grad(None, bufs, ctypes.byref(pp), 8) == -1 and b"BrlPpoParams" in L.brl_last_error()
    pp.batch = 0
    assert L.brl_ppo_grad(None, bufs, ctypes.byref(pp), ctypes.sizeof(pp)) == -1 and b"batch" in L.brl_last_error()
    ap = _lib.BrlAdamParams(n, 1, 1e-3, 0.9, 0.999, 1e-5, 0.5)
    assert L.brl_mlp_adam_step(None, bufs, ctypes.byref(ap), ctypes.sizeof(ap)) == -2 and b"'params' is NULL" in L.brl_last_error()
    fake = (ctypes.c_void_p * 6)(*[ctypes.c_void_p(4096)] * 6)   # never dereferenced: the size check fails first
    ap.n = 12345
    assert L.brl_mlp_adam_step(None, fake, ctypes.byref(ap), ctypes.sizeof(ap)) == -1 and b"brl_mlp_num_params" in L.brl_last_error()
    bp = _lib.BrlParams(0, 0, 0, 0, 0, 0, 0, 0, 0.0, 0.0, 0.0, 0.0)
    assert L.brl_mlp_pack_train(None, bufs, ctypes.byref(bp), ctypes.sizeof(bp)) == -2 and b"params" in L.brl_last_error()


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "brl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cc")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f"{f} imports the oracle"
                assert "brl_oracle" not in src, f"{f} references the oracle"


def test_ops_refuse_cpu_tensors():
    import torch
    from brl_b200 import _lib, ops
    with pytest.raises(_lib.BrlError, match="CUDA"):
        ops.legal_mask(torch.zeros((5, 4, 4), dtype=torch.int32), torch.zeros((4, 38), dtype=torch.uint8))
    from brl_b200 import BridgeBidding
    with pytest.raises(RuntimeError, match="CUDA"):
        BridgeBidding(table=np.zeros((1, 48), np.uint8), device="cpu")


def test_typed_ffi_half_of_the_xla_shim_compiles_against_an_api_stub(tmp_path):
    """The typed-FFI handlers (`<op>_ffi`) are compiled only when XLA's `xla/ffi/api/ffi.h` is on the include path, which it
    never is in this image (no jaxlib).  tests/ffi_stub holds a minimal stand-in for the API surface the shim uses, so the
    typed half is at least compiled -- one handler per op of the table -- instead of rotting unseen.  (It says nothing
    about behaviour inside XLA; INTEGRATION.md states that this half has never run.)"""
    import shutil
    import subprocess
    from brl_b200 import _lib
    gxx = shutil.which("g++")
    assert gxx, "g++ is part of the image"
    obj = tmp_path / "shim.o"
    subprocess.run([gxx, "-std=c++17", "-c", "-I", os.path.join(ROOT, "tests", "ffi_stub"),
                    os.path.join(ROOT, "brl_b200", "csrc", "xla_ffi_shim.cc"), "-o", str(obj)], check=True)
    syms = subprocess.run(["nm", "--defined-only", str(obj)], check=True, capture_output=True, text=True).stdout
    defined = {line.split()[-1] for line in syms.splitlines() if line.strip()}
    for op in _lib.OPS:
        assert op + "_ffi" in defined, f"no typed-FFI handler for {op}"
        assert op + "_xla" in defined

"""ctypes binding of the C-ABI library (include/brl_b200.h).

There is NO CPU fallback: if the CUDA library is missing or fails to load, every
op raises.  The library is built in-tree by `python -m brl_b200.build`.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

# Supervised-learning and league ops, bound on their first call() instead of in load(): a process that never uses them (the
# rollout and PPO loops, bench.py) then creates exactly the Python objects it created before they existed.  Binding them
# eagerly moved the interpreter's garbage-collection schedule in bench.py so that its rollout leg measured 8 % slower on a
# B200 (1000 W), with identical device code and identical timings under gc.disable().
LAZY_OPS = ("brl_sl_examples", "brl_sl_grad", "brl_sl_eval", "brl_model_rows", "brl_policy_act_grouped", "brl_match_stats_ranges",
            "brl_duplicate_match", "brl_evaluate_match", "brl_ppo_grad_grouped", "brl_mlp_adam_step_grouped",
            "brl_ppo_grad_anchored", "brl_ppo_grad_grouped_anchored", "brl_par", "brl_gather_reward_par", "brl_par_stats",
            "brl_system_stats", "brl_system_stats_auctions", "brl_call_values", "brl_cv_grad", "brl_cv_eval",
            "brl_hand_posterior", "brl_hand_posterior_smc")
OPS = (
    "brl_make_keys", "brl_init", "brl_reset_fields", "brl_step", "brl_duplicate_step", "brl_duplicate_init",
    "brl_observe", "brl_legal_mask", "brl_rollout_random", "brl_imp_reward", "brl_gae", "brl_categorical",
    "brl_match_stats", "brl_state_fields", "brl_gather_reward", "brl_team_rows", "brl_mlp_pack", "brl_obs_to_bf16", "brl_mlp_forward", "brl_policy_act",
    "brl_policy_act_rows",
    "brl_ppo_loss", "brl_adam_clip", "brl_adam_apply", "brl_gather_rows", "brl_eval_act_log", "brl_eval_summary", "brl_mlp_pack_train", "brl_mlp_adam_step", "brl_ppo_grad",
) + LAZY_OPS
HOST_API = ("brl_env_create", "brl_env_destroy", "brl_env_init_host", "brl_env_step_host", "brl_env_rollout_host",
            "brl_env_rollout_host_async", "brl_env_wait", "brl_env_trajectory", "brl_env_rollout_host_compact_async",
            "brl_env_rollout_host_compact", "brl_result16_decode", "brl_alloc_compressible", "brl_free_compressible",
            "brl_compressible_granularity", "brl_round_up_granularity")
MISC = ("brl_last_error", "brl_abi_version", "brl_mlp_packed_bytes", "brl_mlp_scratch_bytes", "brl_mlp_rows_scratch_bytes",
        "brl_xla_layout", "brl_xla_unreported_failures", "brl_eval_num_sums",
        "brl_mlp_num_params", "brl_mlp_train_blob_bytes", "brl_mlp_train_scratch_bytes", "brl_mlp_train_trace_offset",
        "brl_mlp_pool_stride", "brl_model_rows_capacity", "brl_policy_grouped_scratch_bytes",
        "brl_duplicate_match_scratch_bytes", "brl_duplicate_match_graph_builds", "brl_evaluate_match_scratch_bytes",
        "brl_evaluate_match_partner_scratch_bytes",
        "brl_ppo_grad_grouped_scratch_bytes", "brl_mlp_param_stride", "brl_call_values_scratch_bytes",
        "brl_hand_posterior_scratch_bytes", "brl_hand_posterior_smc_scratch_bytes")
XLA_LEGACY = tuple(op + "_xla" for op in OPS)  # legacy XLA GPU custom-call targets (csrc/xla_ffi_shim.cc)
ALL_SYMBOLS = OPS + HOST_API + MISC + XLA_LEGACY

# flags (include/brl_b200.h)
F_AUTORESET = 0x0001
F_RANDOM_ACTION = 0x0002
F_ACCUMULATE = 0x0004
F_OBS_U8 = 0x0010
F_OBS_BF16 = 0x0020
F_SAMPLE = 0x0040
F_SL_CHECK = 0x0080
F_QUAD_LAST = 0x0100
F_MLP_BF16 = 0x0200
F_EVAL_INDICATOR_BIDS = 0x0400
F_HOST_STAGED = 0x0800
F_RESULT_I16 = 0x1000
F_UNIFORM_U16 = 0x2000
F_SEED_SALT = 0x4000
F_COUNT_DONE = 0x8000
ABI_VERSION = 3  # include/brl_b200.h BRL_ABI_VERSION; load() refuses a library built from other headers
EVAL_ACC_COLS = 76
MATCH_MAX_STEPS = 638  # brl_duplicate_match's bound on forwards (BRL_MATCH_MAX_STEPS)
MATCH_OK, MATCH_BAD_MODEL, MATCH_STEP_BOUND, MATCH_RECORD_CAPACITY = 0, 1, 2, 3  # its status codes (BRL_MATCH_*)
F_TUNE_MLP_LAYERS, F_TUNE_MLP_FUSED = 1 << 29, 1 << 30  # pin the policy forward's path (BRL_F_TUNE_MLP_*)
EVAL_MATCH_DUPLICATE, EVAL_MATCH_SINGLE, EVAL_MATCH_SIMPLE = 1, 2, 3  # brl_evaluate_match's modes (BRL_EVAL_MATCH_*)
F_EVAL_FREE_RUN = 0x0008  # brl_evaluate_match: team 2 always passes (BRL_F_EVAL_FREE_RUN)
F_EVAL_PARTNER = 1 << 25  # brl_evaluate_match: a 3-net pool, net 2 the actor's partner (BRL_F_EVAL_PARTNER)
F_PLAYER_MODELS = 1 << 24  # brl_model_rows / brl_duplicate_match: env_models[n, 4] by player id (BRL_F_PLAYER_MODELS)
SYS_CONTEXTS, SYS_COLS = 75, 96  # the bidding-system histogram hist[M, 75, 38, 96] (BRL_SYS_*)
# brl_hand_posterior's per-query status codes (BRL_POST_*) and its Philox stream tag
POST_OK, POST_ILLEGAL, POST_SHORT, POST_BAD_NET, POST_BAD_QUERY, POST_CAPACITY = 0, 1, 2, 3, 4, 5
POST_STAGES = 6  # brl_hand_posterior_smc: the prefix is longer than the stage bound
POST_TAG = 0x484E4430
SMC_TAG, SMC_MAX_MOVES, SMC_MAX_STAGES = 0x534D0000, 64, 320  # brl_hand_posterior_smc (BRL_SMC_*)
POST_FEATURES = 95


def f_eval_match(mode: int) -> int:
    """BRL_F_EVAL_MATCH(mode): the flag bits naming brl_evaluate_match's mode"""
    return mode << 27


def tune(epw: int = 0, wpb: int = 0, classic_rollout: bool = False, writers: int = 0, balanced=None) -> int:
    """flag bits: envs-per-warp of the tile kernels / envs-per-block of the warp-specialised
    rollout (8/16/32), warps-per-block of the tile kernels (1/2/4/8), classic_rollout = the
    tile-per-warp rollout instead of the warp-specialised one, writers = writer warps of the
    warp-specialised rollout (1..7).  0 = automatic everywhere."""
    return (({0: 0, 8: 1, 16: 2, 32: 3}[epw] << 16) | ({0: 0, 1: 1, 2: 2, 4: 3, 8: 3 | (1 << 8)}[wpb] << 18) |
            ((1 << 20) if classic_rollout else 0) | ((writers & 7) << 21) |
            (0 if balanced is None else ((1 << 24) if balanced else (1 << 25))))


class BrlParams(C.Structure):
    _fields_ = [
        ("n_envs", C.c_int64), ("env_offset", C.c_int64), ("state_stride", C.c_int64), ("seed", C.c_uint64),
        ("n_deals", C.c_int32), ("flags", C.c_int32), ("step", C.c_uint32), ("k_steps", C.c_int32),
        ("illegal_penalty", C.c_float), ("illegal_bonus", C.c_float), ("gamma", C.c_float), ("gae_lambda", C.c_float),
    ]


class BrlSmcParams(C.Structure):
    _fields_ = [("post", BrlParams), ("ess_threshold", C.c_float), ("moves", C.c_int32), ("stages", C.c_int32),
                ("reserved", C.c_int32)]


class BrlPpoParams(C.Structure):
    _fields_ = [("batch", C.c_int64), ("total", C.c_int64), ("clip_eps", C.c_float), ("ent_coef", C.c_float),
                ("vf_coef", C.c_float), ("illegal_l2_coef", C.c_float), ("flags", C.c_int32), ("reserved", C.c_int32)]


class BrlAdamParams(C.Structure):
    _fields_ = [("n", C.c_int64), ("step", C.c_int32), ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float),
                ("eps", C.c_float), ("max_grad_norm", C.c_float)]


class BrlPpoGroupedParams(C.Structure):
    _fields_ = [("batch", C.c_int64), ("n_learners", C.c_int32), ("flags", C.c_int32), ("reserved", C.c_int32), ("pad", C.c_int32)]


MAX_LEARNERS = 64  # include/brl_b200.h BRL_MAX_LEARNERS


class BrlSlParams(C.Structure):
    _fields_ = [("batch", C.c_int64), ("ent_coef", C.c_float), ("flags", C.c_int32)]


SL_ACC_BYTES = 128  # include/brl_b200.h BRL_SL_ACC_BYTES
SL_OK, SL_ILLEGAL, SL_EARLY_END, SL_NOT_ENDED = 0, 1, 2, 3  # brl_sl_examples check status (BRL_SL_*)


PPO_VALUE_CLIPPING, PPO_REWARD_SCALING, PPO_UNMASKED_POLICY, PPO_ILLEGAL_STAT = 1, 2, 4, 8
PPO_OBS_U8, PPO_OBS_BF16 = 0x10, 0x20
PPO_SCRATCH_BYTES = 188416  # include/brl_b200.h BRL_PPO_SCRATCH_BYTES


class BrlError(RuntimeError):
    pass


_LIB = None


def lib_path() -> str:
    return _build.LIB


def load():
    """Load (building first if sources are newer) the CUDA C-ABI library; raises if impossible."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = _build.LIB
    override = os.environ.get("BRL_B200_LIB")  # debug builds (e.g. -DBRL_GRAM_TIMING, -DBRL_ROLE_TIMING) of the same sources
    if override:
        path = override
    elif not os.path.exists(path) or _build._stale():
        try:
            path = _build.build()  # serialised across processes by a file lock, installed with os.replace
        except Exception as exc:  # no nvcc on this box and no prebuilt library
            if not os.path.exists(_build.LIB):
                raise BrlError(f"libbrl_b200.so is missing and cannot be built ({exc}); there is no CPU fallback") from exc
            import warnings
            warnings.warn(f"brl_b200: sources are newer than {_build.LIB} and the rebuild failed ({exc}); loading the "
                          "existing library (its ABI version is checked below)", RuntimeWarning)
            path = _build.LIB
    try:
        L = C.CDLL(path)
    except OSError as exc:
        raise BrlError(f"cannot load {path}: {exc}; there is no CPU fallback") from exc
    for name in OPS:
        if name in LAZY_OPS:
            continue
        fn = getattr(L, name)
        fn.restype = C.c_int32
        fn.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p, C.c_size_t]
    L.brl_last_error.restype = C.c_char_p
    L.brl_abi_version.restype = C.c_int32
    if L.brl_abi_version() != ABI_VERSION:
        raise BrlError(f"{path} reports ABI version {L.brl_abi_version()}, this package expects {ABI_VERSION}: "
                       "rebuild with `python -m brl_b200.build --force`")
    L.brl_mlp_packed_bytes.restype = C.c_int64
    L.brl_mlp_scratch_bytes.restype = C.c_int64
    L.brl_mlp_scratch_bytes.argtypes = [C.c_int64]
    L.brl_mlp_rows_scratch_bytes.restype = C.c_int64
    L.brl_mlp_rows_scratch_bytes.argtypes = [C.c_int64]
    L.brl_xla_layout.restype = C.c_char_p
    L.brl_xla_layout.argtypes = [C.c_char_p]
    L.brl_xla_unreported_failures.restype = C.c_longlong
    for name in XLA_LEGACY:
        if name[:-4] in LAZY_OPS:
            continue
        fn = getattr(L, name)
        fn.restype = None
        fn.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_char_p, C.c_size_t, C.c_void_p]
    L.brl_mlp_num_params.restype = C.c_int64
    L.brl_mlp_train_blob_bytes.restype = C.c_int64
    L.brl_mlp_train_scratch_bytes.restype = C.c_int64
    L.brl_mlp_train_scratch_bytes.argtypes = [C.c_int64]
    L.brl_mlp_train_trace_offset.restype = C.c_int64
    L.brl_mlp_train_trace_offset.argtypes = [C.c_int64]
    L.brl_env_create.restype = C.c_void_p
    L.brl_env_create.argtypes = [C.c_int64, C.c_int64, C.c_void_p, C.c_int32, C.c_uint64, C.c_int32]
    L.brl_env_destroy.restype = None
    L.brl_env_destroy.argtypes = [C.c_void_p]
    L.brl_env_init_host.restype = C.c_int32
    L.brl_env_init_host.argtypes = [C.c_void_p] * 6
    L.brl_env_step_host.restype = C.c_int32
    L.brl_env_step_host.argtypes = [C.c_void_p] * 7
    L.brl_env_rollout_host.restype = C.c_int32
    L.brl_env_rollout_host.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.brl_env_rollout_host_async.restype = C.c_int64
    L.brl_env_rollout_host_async.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.brl_env_wait.restype = C.c_int32
    L.brl_env_wait.argtypes = [C.c_void_p, C.c_int64]
    L.brl_env_rollout_host_compact_async.restype = C.c_int64
    L.brl_env_rollout_host_compact_async.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    L.brl_env_rollout_host_compact.restype = C.c_int32
    L.brl_env_rollout_host_compact.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    L.brl_result16_decode.restype = None
    L.brl_result16_decode.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.brl_env_trajectory.restype = C.c_int32
    L.brl_env_trajectory.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.brl_alloc_compressible.restype = C.c_void_p
    L.brl_alloc_compressible.argtypes = [C.c_size_t, C.c_int32, C.POINTER(C.c_int32)]
    L.brl_free_compressible.restype = None
    L.brl_free_compressible.argtypes = [C.c_void_p]
    L.brl_compressible_granularity.restype = C.c_int64
    L.brl_compressible_granularity.argtypes = [C.c_int32]
    L.brl_round_up_granularity.restype = C.c_size_t
    L.brl_round_up_granularity.argtypes = [C.c_size_t, C.c_size_t]
    _LIB = L
    return L


class CompressibleBuffer:
    """`nbytes` of device memory from brl_alloc_compressible (compressible where the device supports it), freed with the
    object.  torch sees it as u8[nbytes] through __cuda_array_interface__ and keeps it alive as long as a view of it lives."""

    def __init__(self, nbytes: int, device: int):
        L = load()
        self.ptr = None  # __del__ of a failed allocation
        granted = C.c_int32(0)
        ptr = L.brl_alloc_compressible(nbytes, device, C.byref(granted))
        if not ptr:
            raise BrlError(f"brl_alloc_compressible({nbytes}) failed: {L.brl_last_error().decode()}")
        self.ptr, self.nbytes, self.granted = ptr, nbytes, bool(granted.value)
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "strides": None,
                                         "version": 3, "stream": None}

    def __del__(self):
        if self.ptr and _LIB is not None:
            _LIB.brl_free_compressible(self.ptr)


def call(name: str, stream: int, buffers, params) -> None:
    """Invoke one stream-first op: buffers = iterable of device addresses (int) or None."""
    L = load()
    fn = getattr(L, name)
    if fn.argtypes is None:  # one of LAZY_OPS, first call: bind it and its XLA symbol
        fn.restype = C.c_int32
        fn.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p, C.c_size_t]
        xla = getattr(L, name + "_xla")
        xla.restype = None
        xla.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_char_p, C.c_size_t, C.c_void_p]
    arr = (C.c_void_p * len(buffers))(*[C.c_void_p(b) if b else None for b in buffers])
    rc = fn(C.c_void_p(stream), arr, C.byref(params), C.sizeof(params))
    if rc != 0:
        raise BrlError(f"{name} failed ({rc}): {L.brl_last_error().decode()}")

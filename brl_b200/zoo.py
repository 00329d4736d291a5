"""The fictitious self-play model zoo (ppo.py:351-362 / :392-470) kept packed in HBM.

ppo.py keeps past models on disk and the host path keeps them as NumPy dicts, so every PFSP probe copied each model to the
device and packed it again.  `ModelZoo` holds them as packed blobs in one contiguous device pool, u8[1 + capacity,
brl_mlp_pool_stride()] -- the pool layout brl_duplicate_match and brl_policy_act_grouped read -- so the whole probe is one
match call over the pool (evaluation.make_device_pfsp_probe) and choosing an opponent is one device-to-device copy.
"""
from __future__ import annotations

import torch

from . import dist as bdist
from . import ops
from .models import PackedParams, make_forward_pass

LEARNER_SLOT = 0  # re-packed with the learner's current parameters for each probe


def device_zoo_bytes(capacity: int, probe_envs: int, max_envs: int = 1 << 20) -> int:
    """device memory of a `capacity`-model zoo and of what its PFSP probe (evaluation.make_device_pfsp_probe at `probe_envs`
    boards per model and `max_envs`; `probe_envs` = 0: no probe) holds on each rank: the pool plus the probe's one buffer set,
    sized for the largest chunk over all 1 + capacity nets (evaluation.pfsp_probe_bytes)"""
    from .evaluation import pfsp_probe_bytes
    probe = pfsp_probe_bytes(capacity, probe_envs, max_envs, bdist.rank_world()[1]) if probe_envs else 0
    return (1 + capacity) * ops.mlp_pool_stride() + probe


def device_zoo_fits(capacity: int, probe_envs: int, device, reserve_bytes: int = 16 << 30) -> bool:
    """Whether a `capacity`-model zoo and its probe (device_zoo_bytes) fit in the device's free memory with `reserve_bytes`
    left for the run's own buffers (rollout, update, evaluation matches).  Both are allocated when the zoo is made
    (ModelZoo, probe.reserve), so this one check at the start covers the whole run."""
    free, _ = torch.cuda.mem_get_info(torch.device(device))
    return device_zoo_bytes(capacity, probe_envs) + reserve_bytes <= free


class ModelZoo:
    """The newest `capacity` appended models, packed in HBM.  Logical index k (0 = oldest) names the same model as `zoo[k]`
    of a host list trimmed by `zoo[:] = zoo[-capacity:]` after each append; the models sit in a ring over slots 1..capacity
    and `slot(k)` maps one to the other.  The pool is allocated once, so its address never changes (the match's graph cache
    keys on buffer addresses)."""

    def __init__(self, capacity: int, device):
        if capacity < 0:
            raise ValueError("ModelZoo capacity must be >= 0")
        self.capacity = capacity
        self.pool = torch.zeros((1 + capacity, ops.mlp_pool_stride()), dtype=torch.uint8, device=device)
        self._blob_bytes = ops._lib.load().brl_mlp_packed_bytes()
        self._pack_into = make_forward_pass().pack_into   # the blob layout is the same for both precisions
        self._slots = []                                   # logical index -> pool slot, oldest first

    def __len__(self) -> int:
        return len(self._slots)

    def slot(self, k: int) -> int:
        """pool row of logical model k"""
        return self._slots[k]

    def blob(self, slot: int) -> torch.Tensor:
        """the packed blob of pool row `slot` (a view)"""
        return self.pool[slot, :self._blob_bytes]

    def append(self, params) -> None:
        """pack `params` (device fp32 tensors) straight into a slot; past `capacity` models the oldest one's slot is reused"""
        if self.capacity == 0:
            return
        slot = 1 + len(self._slots) if len(self._slots) < self.capacity else self._slots.pop(0)
        self._pack_into(params, self.blob(slot))
        self._slots.append(slot)

    def set_learner(self, params) -> None:
        """re-pack the learner's current parameters into slot 0"""
        self._pack_into(params, self.blob(LEARNER_SLOT))

    def opponent(self, k: int) -> PackedParams:
        """logical model k as an opponent: a copy of its blob, so later appends that reuse its slot do not change it"""
        return PackedParams(self.blob(self.slot(k)).clone())

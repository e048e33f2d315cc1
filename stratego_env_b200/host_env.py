"""``HostBufferEnv``: the batched engine for callers that keep actions and observations in HOST memory.

Thin wrapper of the C ABI's ``sx_host_env_*`` object (include/stratego_b200.h): the library owns the device
state and output buffers and, per step, pipelines H2D(actions) -> fused kernel -> D2H(outputs) in chunks over
internal streams.  Pass pinned tensors; this path is PCIe-bound (~30.5 KB of outputs per 10x10 game and step, ~17 KB
with an engine built with ``obs_dtype=torch.bfloat16``: the observation buffers follow the engine's dtype) and is what
``bench.py`` reports as ``e2e``.
"""
import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _lib
from .engine import StrategoEngine


class HostBufferEnv:
    def __init__(self, engine: StrategoEngine, num_envs: int, setups: Optional[np.ndarray] = None, seed: int = 0,
                 env_base: int = 0, partial: bool = True, full: bool = False, mask: bool = True,
                 auto_reset: bool = True, sample_actions: bool = True, n_chunks: int = 16, copy_obs: bool = True):
        self.engine, self.num_envs = engine, int(num_envs)
        self._setups = None if setups is None else np.ascontiguousarray(setups, dtype=np.uint8)
        flags = ((_lib.SX_AUTO_RESET if auto_reset else 0) | (_lib.SX_SAMPLE_NEXT if sample_actions else 0) |
                 (_lib.SX_RESET_RANDOM_SHUFFLE if setups is None else 0))
        obs_mask = (_lib.OBS_PO if partial else 0) | (_lib.OBS_FO if full else 0) | (_lib.OBS_MASK if mask else 0)
        self._handle = C.c_void_p()
        with torch.cuda.device(engine.device):
            _lib.check(engine.lib.sx_host_env_create(
                engine._cfg, self.num_envs, int(env_base), obs_mask, flags,
                None if self._setups is None else self._setups.ctypes.data,
                0 if self._setups is None else self._setups.shape[0], int(seed) & (2 ** 64 - 1), int(n_chunks),
                C.byref(self._handle)), "sx_host_env_create")
        R, Cc, A = engine.spatial_action_size
        B = self.num_envs

        def pinned(shape, dtype):
            return torch.empty(shape, dtype=dtype, pin_memory=True)

        self.host = {"reward": pinned((B,), torch.float32), "done": pinned((B,), torch.uint8),
                     "winner": pinned((B,), torch.int8), "ending_invalid": pinned((B,), torch.uint8),
                     "illegal": pinned((B,), torch.uint8), "player": pinned((B,), torch.int8),
                     "next_action": pinned((B,), torch.int32)}
        if copy_obs:  # copy_obs=False: observations and mask stay on the device (scalars only cross PCIe)
            if partial:
                self.host["partial_obs"] = pinned((B, R, Cc, engine.po_channels), engine.obs_dtype)
            if full:
                self.host["full_obs"] = pinned((B, R, Cc, engine.fo_channels), engine.obs_dtype)
            if mask:
                self.host["valid_mask"] = pinned((B, R, Cc, A), torch.uint8)
        self._out = _lib.SxOutputs()
        for k, t in self.host.items():
            setattr(self._out, k, t.data_ptr())
        self.actions = pinned((B,), torch.int32)

    @property
    def d2h_bytes_per_step(self) -> int:
        return sum(t.numel() * t.element_size() for t in self.host.values())

    @property
    def h2d_bytes_per_step(self) -> int:
        return self.actions.numel() * self.actions.element_size()

    def reset(self) -> dict:
        with torch.cuda.device(self.engine.device):
            _lib.check(self.engine.lib.sx_host_env_reset(self._handle, self._out), "sx_host_env_reset")
        return self.host

    def step(self, actions: Optional[torch.Tensor] = None) -> dict:
        """actions: int32 host tensor (default: self.actions); returns the pinned host output tensors (synchronous)"""
        if actions is not None and actions.data_ptr() != self.actions.data_ptr():
            self.actions.copy_(actions)
        with torch.cuda.device(self.engine.device):
            _lib.check(self.engine.lib.sx_host_env_step(self._handle, self.actions.data_ptr(), self._out),
                       "sx_host_env_step")
        return self.host

    def step_ex(self, one_d: bool = False, flags: int = 0) -> dict:
        """one step of self.actions with an explicit action format / per-call flags (used by the one-game API)"""
        with torch.cuda.device(self.engine.device):
            _lib.check(self.engine.lib.sx_host_env_step_ex(
                self._handle, self.actions.data_ptr(), _lib.SX_ACTION_1D if one_d else _lib.SX_ACTION_SPATIAL,
                int(flags), self._out), "sx_host_env_step_ex")
        return self.host

    def device_state(self) -> "RawDeviceState":
        """the object's device-resident state, usable with StrategoEngine.reset / import / export / observe"""
        st = _lib.SxState()
        _lib.check(self.engine.lib.sx_host_env_state(self._handle, C.byref(st), None), "sx_host_env_state")
        return RawDeviceState(st, self.num_envs, self)

    def close(self):
        if self._handle:
            self.engine.lib.sx_host_env_destroy(self._handle)
            self._handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass


class RawDeviceState:
    """state tensors owned by the library (sx_host_env), addressed by raw device pointers"""

    def __init__(self, struct, num_envs, owner):
        self._struct, self.num_envs, self._owner = struct, int(num_envs), owner  # owner keeps the buffers alive

    def as_struct(self):
        return self._struct

"""Batched device-resident CleanupFeatures / HarvestFeatures (+ fused subgame contract wrapper).

Reference: environments/cleanup_features.py:48-336, environments/harvest_features.py:60-364,
contract/contract_list.py:7-54, environments/two_stage_train.py:62-121,159-187.  Eight lanes per env, one launch per
step; observations are float64 feature vectors [E, n, F], or the policy's flat rows (flat_policy.py).
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .batched import HostResultMixin
from .checkpoint import CheckpointMixin
from .episodes import EpisodeLogMixin
from .flat_policy import FlatPolicyMixin
from .maps import CLEANUP_MAP, HARVEST_MAP

_DEFAULT_HIGH = {"CleanupContract": 0.2, "HarvestFeaturemodLocalContract": 10.0}


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


class BatchedFeatureEnv(HostResultMixin, FlatPolicyMixin, CheckpointMixin, EpisodeLogMixin):
    """kind: 'cleanup' | 'harvest' (the reference's `environment` strings for the feature envs).

    policy_dtype: None (float64 `obs` [E, n, F]), or torch.float32 / float16 / bfloat16: the env writes the policy's flat
    rows `policy_obs` T [E*n, policy_width] instead (features ++ [theta, 0] with a contract, policy_width = F + 2; the
    features alone without one) and `obs` is None; reset / step / step_host_async return `policy_obs` in its place.  The
    mode is fixed for the env's lifetime.  (`W` is the map width.)"""

    def __init__(self, kind, num_envs, num_agents, ascii_map=None, horizon=1000, contract=None, theta_low=0.0,
                 theta_high=None, null_prob=0.0, seed=73907, first_env_id=0, device=None, policy_dtype=None):
        if kind not in ("cleanup", "harvest"):
            raise ValueError("BatchedFeatureEnv kind must be cleanup or harvest, got %r" % (kind,))
        if not torch.cuda.is_available():
            raise _lib.SsdError("CUDA device required: contracts_b200 has no CPU fallback")
        self.lib = _lib.load()
        self.kind, self.E, self.n = kind, int(num_envs), int(num_agents)
        self.device = _lib.resolve_device(device)
        self.ascii_map = list(ascii_map) if ascii_map is not None else (CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP)
        self.H, self.W = len(self.ascii_map), len(self.ascii_map[0])
        self.horizon, self.contract = int(horizon), contract
        if theta_high is None:
            theta_high = _DEFAULT_HIGH.get(contract, 0.0)
        self._flat = "".join(self.ascii_map).encode("ascii")
        self.seed, self.first_env_id = int(seed) & 0xFFFFFFFF, int(first_env_id) & 0xFFFFFFFF
        cfg = _lib.make_config(
            env_kind=_lib.ENV_KIND[kind], num_envs=self.E, num_agents=self.n,
            map_h=self.H, map_w=self.W, ascii_map=self._flat, horizon=self.horizon,
            contract_kind=_lib.CONTRACT_KIND[contract], theta_low=float(np.float32(theta_low)),
            theta_high=float(np.float32(theta_high)), null_prob=float(null_prob), seed=int(seed) & 0xFFFFFFFF,
            first_env_id=int(first_env_id) & 0xFFFFFFFF, device=self.device.index, flags=0)
        h = ctypes.c_void_p()
        _lib.check(None, self.lib.ssd_create(ctypes.byref(cfg), ctypes.byref(h)))
        self._h = h
        self.F = self.lib.ssd_feature_dim(self._h)
        E, n, dev = self.E, self.n, self.device
        f64 = torch.float64
        self.obs = None if self._init_policy_output(policy_dtype, self.F) else torch.zeros((E, n, self.F), dtype=f64, device=dev)
        self.rew = torch.zeros((E, n), dtype=f64, device=dev)
        self.base_rew = torch.zeros((E, n), dtype=f64, device=dev)
        self.transfers = torch.zeros((E, n), dtype=f64, device=dev)
        self.info = torch.zeros((E, n, 4), dtype=torch.uint8, device=dev)
        self.done = torch.zeros((E,), dtype=torch.uint8, device=dev)
        self._io = _lib.ssd_feat_io()

    def close(self):
        if getattr(self, "_h", None):
            self.lib.ssd_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def reset(self, mask=None):
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        _lib.check(self._h, self.lib.ssd_feat_reset(self._h, _ptr(mask), _ptr(self.obs), self._stream()))
        return self.observation

    def step(self, actions, extras=True, auto_reset=False):
        """actions: uint8 CUDA tensor [E, n].  Returns (obs [E, n, F] or policy_obs, rew, done [E], info [E, n, 4])."""
        if actions.dtype != torch.uint8 or actions.device != self.device or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=torch.uint8).contiguous()
        io = self._io
        io.actions_dev, io.obs_dev, io.rew_dev = actions.data_ptr(), _ptr(self.obs), self.rew.data_ptr()
        io.base_rew_dev = self.base_rew.data_ptr() if extras else None
        io.transfers_dev = self.transfers.data_ptr() if extras else None
        io.info_dev = self.info.data_ptr()
        io.done_dev = self.done.data_ptr()
        io.auto_reset = 1 if auto_reset else 0       # next-step auto-reset: finished envs restart in the following step
        _lib.check(self._h, self.lib.ssd_feat_step(self._h, ctypes.byref(io), self._stream()))
        return self.observation, self.rew, self.done, self.info

    def step_host_async(self, actions_host, result, dense_rewards=False, auto_reset=False):
        """Submit one step with HOST actions (pinned uint8 [E, n]); returns a ticket without synchronising.  The compact
        result block (int8 rewards + exact float64 records + dones) lands in `result` (a HostResult from new_host_result());
        `step_host_wait(ticket)` makes it valid.  At most two steps in flight; observations stay in self.obs (policy_obs)."""
        if actions_host.device.type != "cpu" or actions_host.dtype != torch.uint8 or not actions_host.is_contiguous():
            raise ValueError("step_host_async needs a contiguous CPU uint8 tensor [E, n] (pinned for an asynchronous copy)")
        io = self._io
        io.actions_dev, io.obs_dev = None, _ptr(self.obs)
        io.rew_dev = self.rew.data_ptr() if dense_rewards else None
        io.base_rew_dev = io.transfers_dev = None
        io.info_dev = self.info.data_ptr()
        io.done_dev = self.done.data_ptr()
        io.auto_reset = 1 if auto_reset else 0
        ticket = ctypes.c_int64(-1)
        _lib.check(self._h, self.lib.ssd_feat_step_host_async(self._h, ctypes.byref(io), ctypes.c_void_p(actions_host.data_ptr()),
                                                              ctypes.c_void_p(result.block.data_ptr()), ctypes.byref(ticket), self._stream()))
        return ticket.value

    def random_actions(self, step_index, num_actions, out=None):
        if step_index is None:
            step_index = 0xFFFFFFFF
        if out is None:
            out = torch.empty((self.E, self.n), dtype=torch.uint8, device=self.device)
        _lib.check(self._h, self.lib.ssd_random_actions(self._h, int(step_index), int(num_actions), _ptr(out), self._stream()))
        return out

    def set_contract_params(self, theta):
        theta = torch.as_tensor(theta, dtype=torch.float64, device=self.device).expand(self.E).contiguous()
        _lib.check(self._h, self.lib.ssd_set_contract_params(self._h, _ptr(theta), self._stream()))

    def get_state(self):
        E, n, dev = self.E, self.n, self.device
        st = {"pos": torch.empty((E, n, 2), dtype=torch.int32, device=dev), "ori": torch.empty((E, n), dtype=torch.int32, device=dev),
              "cells": torch.empty((E, self.H, self.W), dtype=torch.uint8, device=dev),
              "theta": torch.empty((E,), dtype=torch.float64, device=dev), "t": torch.empty((E,), dtype=torch.int32, device=dev)}
        _lib.check(self._h, self.lib.ssd_feat_get_state(self._h, _ptr(st["pos"]), _ptr(st["ori"]), _ptr(st["cells"]),
                                                        _ptr(st["theta"]), _ptr(st["t"]), self._stream()))
        return st

    def metrics_raw(self):
        out = torch.empty((self.E, 40), dtype=torch.float64, device=self.device)
        _lib.check(self._h, self.lib.ssd_feat_get_metrics(self._h, _ptr(out), self._stream()))
        return out

    @property
    def kernel_launches(self):
        return int(self.lib.ssd_kernel_launches(self._h))

"""Batched device-resident SelfAcceleratingCarEnv (+ fused SelfdriveContractDistprop subgame wrapper).

Reference: environments/self_driving_car_accelerate.py:18-250, contract/contract_list.py:56-102,
environments/two_stage_train.py:62-121,159-187.  One kernel launch steps E envs; all values are float64 (observations:
or the policy's flat rows, flat_policy.py).
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .batched import HostResultMixin
from .checkpoint import CheckpointMixin
from .episodes import EpisodeLogMixin
from .flat_policy import FlatPolicyMixin


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


class BatchedCarEnv(HostResultMixin, FlatPolicyMixin, CheckpointMixin, EpisodeLogMixin):
    """policy_dtype: None (float64 `obs` [E, n, D]), or torch.float32 / float16 / bfloat16: the env writes the policy's
    flat rows `policy_obs` T [E*n, policy_width] instead (each car's D values ++ [theta, 0] with a contract,
    policy_width = D + 2; the D values alone without one) and `obs` is None; reset / step / step_host_async return
    `policy_obs` in its place.  The mode is fixed for the env's lifetime."""
    kind = "selfdrive"

    def __init__(self, num_envs, num_agents, contract=None, low_bound=-10.0, high_bound=10.0, start_vel=0.2,
                 start_vel_ambulance=0.8, theta_low=0.0, theta_high=100.0, null_prob=0.0, seed=73907, first_env_id=0,
                 device=None, policy_dtype=None):
        if contract not in (None, "SelfdriveContractDistprop"):
            raise ValueError("selfdrive supports contract None or 'SelfdriveContractDistprop', got %r" % (contract,))
        if not torch.cuda.is_available():
            raise _lib.SsdError("CUDA device required: contracts_b200 has no CPU fallback")
        self.lib = _lib.load()
        self.E, self.n = int(num_envs), int(num_agents)
        self.device = _lib.resolve_device(device)
        self.contract = contract
        self.seed, self.first_env_id = int(seed) & 0xFFFFFFFF, int(first_env_id) & 0xFFFFFFFF
        cfg = _lib.make_config(
            env_kind=_lib.ENV_KIND["selfdrive"], num_envs=self.E, num_agents=self.n,
            map_h=0, map_w=0, ascii_map=None, horizon=0, contract_kind=_lib.CONTRACT_KIND[contract],
            theta_low=float(np.float32(theta_low)), theta_high=float(np.float32(theta_high)), null_prob=float(null_prob),
            seed=int(seed) & 0xFFFFFFFF, first_env_id=int(first_env_id) & 0xFFFFFFFF, device=self.device.index, flags=0)
        cfg.env_params[0], cfg.env_params[1] = float(low_bound), float(high_bound)
        cfg.env_params[2], cfg.env_params[3] = float(start_vel), float(start_vel_ambulance)
        h = ctypes.c_void_p()
        _lib.check(None, self.lib.ssd_create(ctypes.byref(cfg), ctypes.byref(h)))
        self._h = h
        self.D = self.lib.ssd_feature_dim(self._h)
        E, n, dev = self.E, self.n, self.device
        f64 = torch.float64
        self.obs = None if self._init_policy_output(policy_dtype, self.D) else torch.zeros((E, n, self.D), dtype=f64, device=dev)
        self.rew = torch.zeros((E, n), dtype=f64, device=dev)
        self.base_rew = torch.zeros((E, n), dtype=f64, device=dev)
        self.transfers = torch.zeros((E, n), dtype=f64, device=dev)
        self.info = torch.zeros((E, n, 4), dtype=f64, device=dev)
        self.done = torch.zeros((E, n + 1), dtype=torch.uint8, device=dev)
        self._io = _lib.ssd_selfdrive_io()

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
        _lib.check(self._h, self.lib.ssd_selfdrive_reset(self._h, _ptr(mask), _ptr(self.obs), self._stream()))
        return self.observation

    def step(self, actions, extras=True, auto_reset=False):
        """actions: float32 CUDA tensor [E, n].  Returns (obs or policy_obs, rew, done [E, n+1], info [E, n, 4])."""
        if actions.dtype != torch.float32 or actions.device != self.device or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=torch.float32).contiguous()
        io = self._io
        io.actions_dev, io.obs_dev, io.rew_dev = actions.data_ptr(), _ptr(self.obs), self.rew.data_ptr()
        io.base_rew_dev = self.base_rew.data_ptr() if extras else None
        io.transfers_dev = self.transfers.data_ptr() if extras else None
        io.info_dev = self.info.data_ptr() if extras else None
        io.done_dev = self.done.data_ptr()
        io.auto_reset = 1 if auto_reset else 0       # next-step auto-reset: finished envs restart in the following step
        _lib.check(self._h, self.lib.ssd_selfdrive_step(self._h, ctypes.byref(io), self._stream()))
        return self.observation, self.rew, self.done, self.info

    @property
    def host_done_shape(self):
        return (self.E, self.n + 1)

    def step_host_async(self, actions_host, result, dense_rewards=False, auto_reset=False):
        """Submit one step with HOST actions (pinned float32 [E, n]); returns a ticket without synchronising.  The compact
        result block (int8 rewards + exact float64 records + dones [E, n+1]) lands in `result` (a HostResult from
        new_host_result()); `step_host_wait(ticket)` makes it valid.  At most two steps in flight."""
        if actions_host.device.type != "cpu" or actions_host.dtype != torch.float32 or not actions_host.is_contiguous():
            raise ValueError("step_host_async needs a contiguous CPU float32 tensor [E, n] (pinned for an asynchronous copy)")
        io = self._io
        io.actions_dev, io.obs_dev = None, _ptr(self.obs)
        io.rew_dev = self.rew.data_ptr() if dense_rewards else None
        io.base_rew_dev = io.transfers_dev = io.info_dev = None
        io.done_dev = self.done.data_ptr()
        io.auto_reset = 1 if auto_reset else 0
        ticket = ctypes.c_int64(-1)
        _lib.check(self._h, self.lib.ssd_selfdrive_step_host_async(self._h, ctypes.byref(io), ctypes.c_void_p(actions_host.data_ptr()),
                                                                   ctypes.c_void_p(result.block.data_ptr()), ctypes.byref(ticket), self._stream()))
        return ticket.value

    def random_actions(self, step_index, lo=-0.1, hi=0.1, out=None):
        if step_index is None:
            step_index = 0xFFFFFFFF
        if out is None:
            out = torch.empty((self.E, self.n), dtype=torch.float32, device=self.device)
        _lib.check(self._h, self.lib.ssd_selfdrive_random_actions(self._h, int(step_index), float(lo), float(hi), _ptr(out),
                                                                  self._stream()))
        return out

    def set_contract_params(self, theta):
        theta = torch.as_tensor(theta, dtype=torch.float64, device=self.device).expand(self.E).contiguous()
        _lib.check(self._h, self.lib.ssd_set_contract_params(self._h, _ptr(theta), self._stream()))

    def get_state(self):
        E, n, dev = self.E, self.n, self.device
        st = {"pos": torch.empty((E, n), dtype=torch.float64, device=dev), "vel": torch.empty((E, n), dtype=torch.float64, device=dev),
              "theta": torch.empty((E,), dtype=torch.float64, device=dev),
              "transfers": torch.empty((E,), dtype=torch.float64, device=dev), "t": torch.empty((E,), dtype=torch.int32, device=dev)}
        _lib.check(self._h, self.lib.ssd_selfdrive_get_state(self._h, _ptr(st["pos"]), _ptr(st["vel"]), _ptr(st["theta"]),
                                                             _ptr(st["transfers"]), _ptr(st["t"]), self._stream()))
        return st

    @property
    def kernel_launches(self):
        return int(self.lib.ssd_kernel_launches(self._h))

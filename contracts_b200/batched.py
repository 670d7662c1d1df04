"""Batched device-resident environments: the fast path behind the drop-in API.

`BatchedGridEnv` owns E independent cleanup_new / harvest_new environments (optionally with
the subgame contract wrapper fused in) on one GPU.  All I/O is torch CUDA tensors; the step
is one kernel launch through the C ABI (`ssd_step`).  PyTorch is used only for device
memory and streams.

Reference classes covered (paths relative to the reference root):
  environments/cleanup_new.py CleanupEnv, environments/harvest_new.py HarvestEnv,
  environments/two_stage_train.py SeparateContractEnv.step :62-121 and
  SeparateContractSubgameStage.reset :159-187, contract/contract_list.py.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .checkpoint import CheckpointMixin
from .episodes import EpisodeLogMixin
from .maps import CLEANUP_MAP, HARVEST_MAP

_DEFAULT_HIGH = {"CleanupContract": 0.2, "HarvestFeaturemodLocalContract": 10.0}


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def negotiate(batch, proposals, accept, mask=None, out=None):
    """Agreement stage of SeparateContractNegotiateStage.step (two_stage_train.py:266-281) for every env of `batch` (any
    Batched*Env): proposals [E], accept [E, n] float64.  Sets each env's contract parameter; returns uint8 [E].
    mask (uint8 [E], optional): only the envs with mask != 0 negotiate (the ones that were just reset); the decision
    bytes of the others are left as they are in `out`."""
    def ready(x, shape):                                  # the hot caller passes tensors that need no conversion
        return torch.is_tensor(x) and x.dtype == torch.float64 and x.device == batch.device and tuple(x.shape) == shape \
            and x.is_contiguous()
    if not ready(proposals, (batch.E,)):
        proposals = torch.as_tensor(proposals, dtype=torch.float64, device=batch.device).expand(batch.E).contiguous()
    if not ready(accept, (batch.E, batch.n)):
        accept = torch.as_tensor(accept, dtype=torch.float64, device=batch.device).expand(batch.E, batch.n).contiguous()
    if mask is not None and (mask.dtype != torch.uint8 or mask.device != batch.device or not mask.is_contiguous()):
        mask = mask.to(device=batch.device, dtype=torch.uint8).contiguous()
    dec = out if out is not None else (torch.empty if mask is None else torch.zeros)((batch.E,), dtype=torch.uint8, device=batch.device)
    stream = ctypes.c_void_p(torch.cuda.current_stream(batch.device).cuda_stream)
    _lib.check(batch._h, batch.lib.ssd_negotiate(batch._h, _ptr(mask), _ptr(proposals), _ptr(accept), _ptr(dec), stream))
    return dec


def solver_sample(batch, num_samples):
    """Candidate contracts of NegotiationSolver.negotiate (two_stage_train.py:705-746) for every env of `batch` (any
    Batched*Env): float64 [E, 1 + num_samples], column 0 = the null contract, the others float32-valued samples."""
    params = torch.empty((batch.E, num_samples + 1), dtype=torch.float64, device=batch.device)
    stream = ctypes.c_void_p(torch.cuda.current_stream(batch.device).cuda_stream)
    _lib.check(batch._h, batch.lib.ssd_solver_sample(batch._h, int(num_samples), _ptr(params), stream))
    return params


def solver_choose(batch, params, vals, rule="majority"):
    """compute_best_param (two_stage_train.py:748-776): vals float64 [E, 1 + S, n] = the caller's value function for
    every candidate and agent.  Sets each env's contract parameter; returns (theta [E], chosen index [E])."""
    E, S1 = params.shape
    vals = torch.as_tensor(vals, dtype=torch.float64, device=batch.device).contiguous()
    if tuple(vals.shape) != (E, S1, batch.n):
        raise ValueError("vals must be [E, 1 + S, n] = %r, got %r" % ((E, S1, batch.n), tuple(vals.shape)))
    params = params.to(device=batch.device, dtype=torch.float64).contiguous()
    best = torch.empty((E,), dtype=torch.float64, device=batch.device)
    idx = torch.empty((E,), dtype=torch.int32, device=batch.device)
    stream = ctypes.c_void_p(torch.cuda.current_stream(batch.device).cuda_stream)
    _lib.check(batch._h, batch.lib.ssd_solver_choose(batch._h, S1 - 1, _lib.SOLVER_RULE[rule], _ptr(params), _ptr(vals),
                                                     _ptr(best), _ptr(idx), stream))
    return best, idx


class HostResult:
    """One pinned result block of `ssd_step_host_async` with numpy views of its fields (valid after step_host_wait):
    count (records in use), done uint8 [E] ([E, n + 1] for selfdrive), rew_i8 int8 [E, n], rec_env int32 [E],
    rec_rew float64 [E, n].  `batch` is any of the batched envs (grid, feature, selfdrive)."""

    def __init__(self, batch):
        lay = batch.host_result_layout()
        self.batch, self.lay = batch, lay
        self.block = torch.zeros((lay.total_bytes,), dtype=torch.uint8).pin_memory()
        b = self.block.numpy()
        E, n = batch.E, batch.n
        self._count = b[lay.count_offset:lay.count_offset + 4].view(np.uint32)
        dshape = getattr(batch, "host_done_shape", (E,))          # selfdrive: [E, n + 1] (per-car dones, then '__all__')
        self.done = b[lay.done_offset:lay.done_offset + int(np.prod(dshape))].reshape(dshape)
        self.rew_i8 = b[lay.rew_i8_offset:lay.rew_i8_offset + E * n].view(np.int8).reshape(E, n)
        rec = b[lay.records_offset:lay.records_offset + E * lay.record_bytes].reshape(E, lay.record_bytes)
        self.rec_env = rec[:, 0:4].view(np.int32).reshape(E)
        self.rec_rew = rec[:, 8:].view(np.float64).reshape(E, n)

    @property
    def count(self):
        return int(self._count[0])

    def rewards(self, out=None):
        """dense float64 [E, n] (ssd_host_result_expand: int8 rewards widened, the exact records on top)"""
        if out is None:
            out = np.empty((self.batch.E, self.batch.n), dtype=np.float64)
        _lib.check(self.batch._h, self.batch.lib.ssd_host_result_expand(self.batch._h, ctypes.c_void_p(self.block.data_ptr()),
                                                                         out.ctypes.data_as(ctypes.c_void_p)))
        return out


class HostResultMixin:
    """host_result_layout / new_host_result / step_host_wait shared by the batched envs (ssd_host_result_layout,
    ssd_step_host_wait serve every env kind)."""

    def host_result_layout(self):
        lay = _lib.ssd_host_layout()
        _lib.check(self._h, self.lib.ssd_host_result_layout(self._h, ctypes.byref(lay)))
        return lay

    def new_host_result(self):
        """A pinned host block for step_host_async + numpy views of its fields (`HostResult`)."""
        return HostResult(self)

    def step_host_wait(self, ticket):
        _lib.check(self._h, self.lib.ssd_step_host_wait(self._h, int(ticket)))


class BatchedGridEnv(HostResultMixin, CheckpointMixin, EpisodeLogMixin):
    """E environments of one kind on one device.

    kind: 'cleanup_new' | 'harvest_new' (the reference's `environment` strings,
    utils/env_creator_functions.py:47-60).  contract: None or the class name from
    contract/contract_list.py.  theta_low/high default to the contract's gym Box bounds, which
    gym stores as float32 (contract_list.py:20,43) — the float32 rounding is part of parity.

    policy_dtype: None (uint8 windows in `obs`, the reference's observation), or torch.float32 / float16 / bfloat16: the
    env writes the policy's input tensors itself (ssd_set_policy_output) — `policy_image` T [E*n, 3, 15, 15], the value
    `policy_inputs(T)` would make of the windows, and `policy_contract` T [E*n, 10] (None without a contract) — and keeps
    no uint8 windows (`obs` is None).  reset / step / step_host return `policy_image` in place of `obs`.  The mode is fixed
    for the env's lifetime; the methods that read the uint8 windows (host_snapshot(obs=True), concatenated_obs,
    policy_inputs) raise ValueError in it.

    image_obs=False: the observation is the feature vector (image_obs=False of the reference, cleanup_new.py:193-202,243-254,
    harvest_new.py:160-168,212-222), written by the device at every step and reset (ssd_set_feature_output) — the same
    interface as BatchedFeatureEnv: `obs` float64 [E, n, F], or with policy_dtype T the policy's flat rows `policy_obs`
    T [E*n, policy_width] (features ++ [theta, 0] under a contract, policy_width = F + 2; the features alone without one)
    and `obs` None.  No uint8 windows are kept: step(want_features=True) and the methods that read windows raise
    ValueError.

    global_obs=True: the observation is JointEnv's global view (global_obs=True of the reference, two_stage_train.py:572-617:
    get_global_obs() = global_view() / 255, cleanup_new.py:299-300), written by the device at every step and reset
    (ssd_set_global_output): `obs` uint8 [E, H, W, 3], what global_view() returns, or with policy_dtype T `policy_obs`
    T [E, 3, H, W] = (u8 / 255).float().permute(0, 3, 1, 2).to(T) — VisionNetwork.forward's input — and `obs` None.  No
    contract (JointEnv wraps the bare base env) and image_obs=True.  No uint8 windows are kept: step(want_features=True)
    and the methods that read windows raise ValueError; global_view() and render() still work.
    (The concatenated JointEnv variant needs no form of its own: `policy_image.view(E, 3 n, 15, 15)` of a policy_dtype env
    without a contract is (concatenated_obs() / 255).float().permute(0, 3, 1, 2), the channel index 3 a + c being
    agent-major.)
    """

    def __init__(self, kind, num_envs, num_agents, ascii_map=None, horizon=1000, contract=None,
                 theta_low=0.0, theta_high=None, null_prob=0.0, seed=73907, first_env_id=0,
                 device=None, padded_obs=False,
                 use_collective_reward=False, inequity_averse_reward=False, alpha=0.0, beta=0.0, policy_dtype=None,
                 image_obs=True, global_obs=False):
        if kind not in ("cleanup_new", "harvest_new"):
            raise ValueError("BatchedGridEnv kind must be cleanup_new or harvest_new, got %r" % (kind,))
        if global_obs and not image_obs:
            raise ValueError("global_obs=True observes the colour map: it does not go with image_obs=False")
        if global_obs and contract is not None:
            raise ValueError("global_obs=True is JointEnv's observation of the bare base env: no contract (got %r)" % (contract,))
        if not torch.cuda.is_available():
            raise _lib.SsdError("CUDA device required: contracts_b200 has no CPU fallback")
        self.lib = _lib.load()
        self.kind, self.E, self.n = kind, int(num_envs), int(num_agents)
        self.device = _lib.resolve_device(device)
        self.ascii_map = list(ascii_map) if ascii_map is not None else (
            CLEANUP_MAP if kind == "cleanup_new" else HARVEST_MAP)
        self.H, self.W = len(self.ascii_map), len(self.ascii_map[0])
        if any(len(r) != self.W for r in self.ascii_map):
            raise ValueError("ascii_map rows must have equal length")
        self.horizon = int(horizon)
        self.contract = contract
        self.inequity_averse_reward = bool(inequity_averse_reward)     # env rewards are float64 (map_env.py:293-300)
        if theta_high is None:
            theta_high = _DEFAULT_HIGH.get(contract, 0.0)
        self.theta_low = float(np.float32(theta_low))
        self.theta_high = float(np.float32(theta_high))
        self.seed, self.first_env_id = int(seed) & 0xFFFFFFFF, int(first_env_id) & 0xFFFFFFFF
        self._flat = "".join(self.ascii_map).encode("ascii")
        cfg = _lib.make_config(
            env_kind=_lib.ENV_KIND[kind], num_envs=self.E, num_agents=self.n,
            map_h=self.H, map_w=self.W, ascii_map=self._flat, horizon=self.horizon,
            contract_kind=_lib.CONTRACT_KIND[contract], theta_low=self.theta_low, theta_high=self.theta_high,
            null_prob=float(null_prob), seed=self.seed, first_env_id=self.first_env_id,
            device=self.device.index,
            # MapEnv reward shaping kwargs (map_env.py:69-72,289-301)
            flags=(_lib.FLAG_COLLECTIVE_REWARD if use_collective_reward else 0)
            | (_lib.FLAG_INEQUITY_AVERSE if inequity_averse_reward else 0))
        cfg.env_params[0], cfg.env_params[1] = float(alpha), float(beta)
        h = ctypes.c_void_p()
        _lib.check(None, self.lib.ssd_create(ctypes.byref(cfg), ctypes.byref(h)))
        self._h = h
        self.F = self.lib.ssd_feature_dim(self._h)
        E, n, dev = self.E, self.n, self.device
        self.policy_dtype, self.policy_image, self.policy_contract = policy_dtype, None, None
        self.image_obs, self.policy_obs, self.policy_width = bool(image_obs), None, None
        self.global_obs = bool(global_obs)
        if not self.image_obs:
            self._init_feature_output(policy_dtype)
        elif self.global_obs:
            self._init_global_output(policy_dtype)
        elif policy_dtype is not None:
            try:
                code = _lib.policy_dtype_code(policy_dtype)
            except ValueError:
                self.close()
                raise
            self.policy_image = torch.zeros((E * n, 3, 15, 15), dtype=policy_dtype, device=dev)
            if contract is not None:
                self.policy_contract = torch.zeros((E * n, 10), dtype=policy_dtype, device=dev)
            out = _lib.ssd_policy_out(struct_size=ctypes.sizeof(_lib.ssd_policy_out), dtype=code,
                                      image_dev=self.policy_image.data_ptr(),
                                      contract_dev=None if self.policy_contract is None else self.policy_contract.data_ptr())
            _lib.check(self._h, self.lib.ssd_set_policy_output(self._h, ctypes.byref(out)))
            self.obs_stride, self._obs_buf, self.obs = 0, None, None
        else:
            # observation batch tensor: dense [E, n, 15, 15, 3], or env stride padded to 16 B
            dense = n * _lib.OBS_BYTES_PER_AGENT
            self.obs_stride = (dense + 15) // 16 * 16 if padded_obs else dense
            self._obs_buf = torch.zeros((E, self.obs_stride), dtype=torch.uint8, device=dev)
            self.obs = self._obs_buf[:, :dense].view(E, n, 15, 15, 3) if padded_obs else self._obs_buf.view(E, n, 15, 15, 3)
        self.rew = torch.zeros((E, n), dtype=torch.float64, device=dev)
        self.base_rew = torch.zeros((E, n), dtype=torch.float64, device=dev)
        self.transfers = torch.zeros((E, n), dtype=torch.float64, device=dev)
        self.info = torch.zeros((E, n, 4), dtype=torch.uint8, device=dev)
        self.done = torch.zeros((E,), dtype=torch.uint8, device=dev)
        self.feature_obs = None
        self._host_actions_dev = None
        self._io = _lib.ssd_step_io()

    # ------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self.lib.ssd_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _init_feature_output(self, policy_dtype):
        """image_obs=False: the handle writes float64 feature rows to `obs`, or the policy's flat rows to `policy_obs`"""
        E, n = self.E, self.n
        try:
            code = _lib.FEATURE_F64 if policy_dtype is None else _lib.policy_dtype_code(policy_dtype)
        except ValueError:
            self.close()
            raise
        self.policy_width = self.F + (2 if self.contract is not None else 0)
        if policy_dtype is None:
            self.obs = torch.zeros((E, n, self.F), dtype=torch.float64, device=self.device)
            rows = self.obs
        else:
            self.obs = None
            self.policy_obs = rows = torch.zeros((E * n, self.policy_width), dtype=policy_dtype, device=self.device)
        out = _lib.ssd_feature_out(struct_size=ctypes.sizeof(_lib.ssd_feature_out), dtype=code, obs_dev=rows.data_ptr())
        _lib.check(self._h, self.lib.ssd_set_feature_output(self._h, ctypes.byref(out)))
        self.obs_stride, self._obs_buf = 0, None

    def _init_global_output(self, policy_dtype):
        """global_obs=True: the handle writes the global view uint8 [E, H, W, 3] to `obs`, or T [E, 3, H, W] to `policy_obs`"""
        try:
            code = _lib.GLOBAL_U8 if policy_dtype is None else _lib.policy_dtype_code(policy_dtype)
        except ValueError:
            self.close()
            raise
        if policy_dtype is None:
            self.obs = rows = torch.zeros((self.E, self.H, self.W, 3), dtype=torch.uint8, device=self.device)
        else:
            self.obs = None
            self.policy_obs = rows = torch.zeros((self.E, 3, self.H, self.W), dtype=policy_dtype, device=self.device)
        out = _lib.ssd_global_out(struct_size=ctypes.sizeof(_lib.ssd_global_out), dtype=code, obs_dev=rows.data_ptr())
        _lib.check(self._h, self.lib.ssd_set_global_output(self._h, ctypes.byref(out)))
        self.obs_stride, self._obs_buf = 0, None

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def observation(self):
        """what reset / step return: `obs`, or `policy_image` when the env writes the policy's tensors (`policy_obs` with
        image_obs=False or global_obs=True)"""
        if not self.image_obs or self.global_obs:
            return self.obs if self.policy_dtype is None else self.policy_obs
        return self.obs if self.policy_dtype is None else self.policy_image

    def _no_feature_copy(self, want_features):
        if want_features and not self.image_obs:
            raise ValueError("want_features: with image_obs=False the observation already is the feature rows (`obs` / policy_obs)")
        if want_features and self.global_obs:
            raise ValueError("want_features: a global_obs=True env writes the global view and no feature rows")

    def _need_windows(self, what):
        if not self.image_obs:
            raise ValueError("%s needs the uint8 observation windows; this env observes feature vectors (image_obs=False)" % what)
        if self.global_obs:
            raise ValueError("%s needs the uint8 observation windows; this env observes the global view (global_obs=True)" % what)
        if self.policy_dtype is not None:
            raise ValueError("%s needs the uint8 observation windows; this env writes the policy's tensors instead "
                             "(policy_dtype=%s)" % (what, self.policy_dtype))

    def _obs_rows(self):
        """the observation rows checkpoint / restore carry: uint8 [E, n, 15, 15, 3], or T [E, n, 3, 15, 15] in policy mode;
        with image_obs=False float64 [E, n, F], or T [E, n, policy_width]; with global_obs=True uint8 [E, H, W, 3], or
        T [E, 3, H, W]"""
        if not self.image_obs:
            return self.obs if self.policy_dtype is None else self.policy_obs.view(self.E, self.n, self.policy_width)
        if self.global_obs:
            return self.obs if self.policy_dtype is None else self.policy_obs
        return self.obs if self.policy_dtype is None else self.policy_image.view(self.E, self.n, 3, 15, 15)

    def reset(self, mask=None):
        """Reset all envs (mask None) or those with mask != 0 (uint8 CUDA tensor [E]).  Returns obs (policy_image in
        policy mode)."""
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        _lib.check(self._h, self.lib.ssd_reset(self._h, _ptr(mask), _ptr(self._obs_buf), self.obs_stride, self._stream()))
        return self.observation

    def _auto_reset_io(self, io, auto_reset, negotiation):
        """vectorised-sampler mode of a step: finished envs restart inside the step (+ negotiate, given the policy's
        negotiation outputs (proposals [E], accept [E, n], decisions uint8 [E] or None) as float64 CUDA tensors)"""
        io.auto_reset = 1 if auto_reset else 0
        io.neg_proposals_dev = io.neg_accept_dev = io.neg_decision_dev = None
        if auto_reset and negotiation is not None:
            prop, acc, dec = negotiation
            for x, shape in ((prop, (self.E,)), (acc, (self.E, self.n))):
                if x.dtype != torch.float64 or x.device != self.device or tuple(x.shape) != shape or not x.is_contiguous():
                    raise ValueError("negotiation tensors must be contiguous float64 CUDA tensors [E] and [E, n]")
            io.neg_proposals_dev, io.neg_accept_dev = prop.data_ptr(), acc.data_ptr()
            io.neg_decision_dev = dec.data_ptr() if dec is not None else None

    def step(self, actions, want_features=False, extras=True, auto_reset=False, negotiation=None):
        """actions: uint8 CUDA tensor [E, n].  Returns (obs, rew, done, info) device tensors.

        The same output tensors are reused every step.  extras=False skips base_rew/transfers.
        auto_reset=True: envs that finish in this step are reset by the step itself (their observation is the reset
        observation; rewards / done / info are the final step's) and, with negotiation=(proposals, accept, decisions),
        negotiate their next contract — what `reset(done)` + `negotiate(..., mask=done)` would do, without the launches.
        """
        if actions.dtype != torch.uint8 or actions.device != self.device or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=torch.uint8).contiguous()
        self._no_feature_copy(want_features)
        if want_features and self.feature_obs is None:
            self.feature_obs = torch.zeros((self.E, self.n, self.F), dtype=torch.float64, device=self.device)
        io = self._io
        io.actions_dev = actions.data_ptr()
        io.obs_dev = None if self._obs_buf is None else self._obs_buf.data_ptr()
        io.obs_env_stride = self.obs_stride
        io.rew_dev = self.rew.data_ptr()
        io.base_rew_dev = self.base_rew.data_ptr() if extras else None
        io.transfers_dev = self.transfers.data_ptr() if extras else None
        io.info_dev = self.info.data_ptr()
        io.feature_obs_dev = self.feature_obs.data_ptr() if want_features else None
        io.done_dev = self.done.data_ptr()
        self._auto_reset_io(io, auto_reset, negotiation)
        _lib.check(self._h, self.lib.ssd_step(self._h, ctypes.byref(io), self._stream()))
        return self.observation, self.rew, self.done, self.info

    def step_host(self, actions_host, rew_host, done_host=None, want_features=False):
        """One step for a caller holding HOST tensors (pinned for asynchronous copies): uint8 actions [E, n] in,
        float64 rewards [E, n] (and uint8 dones [E]) out, valid on return.  The rewards travel back while the
        observe kernel still runs; the observations stay on the device in `self.obs`."""
        for t, dt in ((actions_host, torch.uint8), (rew_host, torch.float64)) + (((done_host, torch.uint8),) if done_host is not None else ()):
            if t.device.type != "cpu" or t.dtype != dt or not t.is_contiguous():
                raise ValueError("step_host needs contiguous CPU tensors: uint8 actions, float64 rewards, uint8 dones")
        if self._host_actions_dev is None:
            self._host_actions_dev = torch.empty((self.E, self.n), dtype=torch.uint8, device=self.device)
        self._no_feature_copy(want_features)
        if want_features and self.feature_obs is None:
            self.feature_obs = torch.zeros((self.E, self.n, self.F), dtype=torch.float64, device=self.device)
        io = self._io
        io.actions_dev = self._host_actions_dev.data_ptr()
        io.obs_dev = None if self._obs_buf is None else self._obs_buf.data_ptr()
        io.obs_env_stride = self.obs_stride
        io.rew_dev = self.rew.data_ptr()
        io.base_rew_dev = None
        io.transfers_dev = None
        io.info_dev = self.info.data_ptr()
        io.feature_obs_dev = self.feature_obs.data_ptr() if want_features else None
        io.done_dev = self.done.data_ptr()
        self._auto_reset_io(io, False, None)
        _lib.check(self._h, self.lib.ssd_step_host(self._h, ctypes.byref(io), ctypes.c_void_p(actions_host.data_ptr()),
                                                   ctypes.c_void_p(rew_host.data_ptr()),
                                                   ctypes.c_void_p(done_host.data_ptr()) if done_host is not None else None,
                                                   self._stream()))
        return self.observation, rew_host, done_host

    # ---- pipelined host-buffer step (RLlib BaseEnv send_actions / poll shape) ---------------------------------
    def step_host_async(self, actions_host, result, want_features=False, dense_rewards=False, auto_reset=False, negotiation=None):
        """Submit one step with HOST actions (pinned uint8 [E, n]); returns a ticket without synchronising.  The
        compact result block (int8 rewards + exact float64 records + dones) is copied into `result` (a HostResult)
        while the observe kernel runs; `step_host_wait(ticket)` makes it valid.  At most two steps in flight.
        dense_rewards=True also writes the float64 [E, n] matrix to self.rew on the device."""
        if actions_host.device.type != "cpu" or actions_host.dtype != torch.uint8 or not actions_host.is_contiguous():
            raise ValueError("step_host_async needs a contiguous CPU uint8 tensor [E, n] (pinned for an asynchronous copy)")
        self._no_feature_copy(want_features)
        if want_features and self.feature_obs is None:
            self.feature_obs = torch.zeros((self.E, self.n, self.F), dtype=torch.float64, device=self.device)
        io = self._io
        io.actions_dev = None
        io.obs_dev = None if self._obs_buf is None else self._obs_buf.data_ptr()
        io.obs_env_stride = self.obs_stride
        io.rew_dev = self.rew.data_ptr() if dense_rewards else None
        io.base_rew_dev = None
        io.transfers_dev = None
        io.info_dev = self.info.data_ptr()
        io.feature_obs_dev = self.feature_obs.data_ptr() if want_features else None
        io.done_dev = self.done.data_ptr()
        self._auto_reset_io(io, auto_reset, negotiation)
        ticket = ctypes.c_int64(-1)
        _lib.check(self._h, self.lib.ssd_step_host_async(self._h, ctypes.byref(io), ctypes.c_void_p(actions_host.data_ptr()),
                                                         ctypes.c_void_p(result.block.data_ptr()), ctypes.byref(ticket), self._stream()))
        return ticket.value

    # ---- packed host snapshots (dict façade, vector adapter): ONE device -> host copy per call ----------------
    def host_snapshot(self, index=None, features=False, extras=True, obs=True):
        """Everything a dict API returns for env `index` (None: every env), gathered into one device byte buffer and
        copied to the host with ONE transfer + ONE synchronisation.  Returns numpy views:
        obs uint8 [.., n, 15, 15, 3], rew / base_rew / transfers float64 [.., n], info uint8 [.., n, 4], done uint8 [..],
        feat float64 [.., n, F] (when `features`)."""
        if obs:
            self._need_windows("host_snapshot(obs=True)")
        sel = slice(None) if index is None else slice(index, index + 1)
        E = self.E if index is None else 1
        parts = [("rew", self.rew[sel], np.float64, (E, self.n)), ("info", self.info[sel], np.uint8, (E, self.n, 4)),
                 ("done", self.done[sel], np.uint8, (E,))]
        if obs:
            parts.append(("obs", self.obs[sel], np.uint8, (E, self.n, 15, 15, 3)))
        if extras:
            parts += [("base_rew", self.base_rew[sel], np.float64, (E, self.n)), ("transfers", self.transfers[sel], np.float64, (E, self.n))]
        if features and self.feature_obs is not None:
            parts.append(("feat", self.feature_obs[sel], np.float64, (E, self.n, self.F)))
        # float64 fields first: every field starts 8-byte aligned in the packed buffer
        parts.sort(key=lambda x: -np.dtype(x[2]).itemsize)
        flat = [t.reshape(-1).view(torch.uint8) if t.dtype != torch.uint8 else t.reshape(-1) for _, t, _, _ in parts]
        packed = torch.cat(flat)
        key = int(packed.numel())
        host = self._snap_host.get(key) if hasattr(self, "_snap_host") else None
        if host is None:
            if not hasattr(self, "_snap_host"):
                self._snap_host = {}
            host = self._snap_host[key] = torch.empty((key,), dtype=torch.uint8).pin_memory()
        host.copy_(packed, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        buf, out, off = host.numpy(), {}, 0
        for (name, _, dt, shape), f in zip(parts, flat):
            nb = int(f.numel())
            a = buf[off:off + nb].view(dt).reshape(shape)
            out[name] = a[0] if index is not None else a
            off += nb
        return out

    def random_actions(self, step_index, num_actions, out=None):
        """Uniform random actions; step_index=None uses the handle's device-side counter (CUDA-graph friendly)."""
        if step_index is None:
            step_index = 0xFFFFFFFF
        if out is None:
            out = torch.empty((self.E, self.n), dtype=torch.uint8, device=self.device)
        _lib.check(self._h, self.lib.ssd_random_actions(self._h, int(step_index), int(num_actions), _ptr(out), self._stream()))
        return out

    # ------------------------------------------------------------------------------------------
    def set_contract_params(self, theta):
        theta = torch.as_tensor(theta, dtype=torch.float64, device=self.device).expand(self.E).contiguous()
        _lib.check(self._h, self.lib.ssd_set_contract_params(self._h, _ptr(theta), self._stream()))

    def negotiate(self, proposals, accept, mask=None, out=None):
        """Agreement stage (two_stage_train.py:266-281).  proposals [E], accept [E, n] float64.  Returns uint8 [E]."""
        return negotiate(self, proposals, accept, mask, out)

    def set_episode_stats(self, stats):
        """stats: float64 CUDA tensor [8] (zeroed by the caller) or None.  While set, every reset() adds the accumulators
        of the finished episodes it replaces: apples_eaten, raw_env_rewards, transfers, dirt_cleaned, sum of transferred
        rewards, sum of raw rewards, episodes, max err_flags (sharding.STAT_FIELDS with `envs` = episodes)."""
        if stats is not None and (stats.dtype != torch.float64 or stats.device != self.device or stats.numel() != _lib.STATS_LEN
                                  or not stats.is_contiguous()):
            raise ValueError("stats must be a contiguous float64 CUDA tensor of %d elements on %s" % (_lib.STATS_LEN, self.device))
        self._stats = stats                              # keep it alive while the library holds its address
        _lib.check(self._h, self.lib.ssd_set_episode_stats(self._h, _ptr(stats)))

    # ---- JointEnv output layouts (two_stage_train.py:476-617) ---------------------------------------
    def global_view(self, out=None):
        """MapEnv.global_view() of every env (map_env.py:394-395): uint8 [E, H, W, 3]; `global_obs` is this / 255."""
        if out is None:
            out = torch.empty((self.E, self.H, self.W, 3), dtype=torch.uint8, device=self.device)
        _lib.check(self._h, self.lib.ssd_global_view(self._h, _ptr(out), self._stream()))
        return out

    def record_beams(self, on=True):
        """Keep the cells crossed by the beams of each step (MapEnv.beam_pos) so that `render()` can draw them."""
        _lib.check(self._h, self.lib.ssd_record_beams(self._h, 1 if on else 0))

    def render(self, out=None):
        """MapEnv.full_map_to_colors() of every env (map_env.py:389-392): uint8 [E, H, W, 3], beams included when recorded."""
        if out is None:
            out = torch.empty((self.E, self.H, self.W, 3), dtype=torch.uint8, device=self.device)
        _lib.check(self._h, self.lib.ssd_render(self._h, _ptr(out), self._stream()))
        return out

    def concatenated_obs(self, out=None):
        """The agents' windows concatenated along the channel axis (two_stage_train.py:527-533): uint8 [E, 15, 15, 3 n]."""
        self._need_windows("concatenated_obs")
        if out is None:
            out = torch.empty((self.E, 15, 15, 3 * self.n), dtype=torch.uint8, device=self.device)
        _lib.check(self._h, self.lib.ssd_concat_obs(self._h, _ptr(self._obs_buf), self.obs_stride, _ptr(out), self._stream()))
        return out

    # ---- policy-side consumer (environments/Networks/vision_net.py:150-181) -----------------------------
    def policy_inputs(self, dtype=torch.float32, with_contract=True, image=None, contract=None):
        """The current observations as VisionNetwork.forward feeds its convolutions: image [E*n, 3, 15, 15] =
        (`curr_obs / 255`).float().permute(0, 3, 1, 2), contract [E*n, 10] = (theta, 0) repeated 5 times.
        (With policy_dtype set the env writes these itself: policy_image / policy_contract.)"""
        self._need_windows("policy_inputs")
        B = self.E * self.n
        if image is None:
            image = torch.empty((B, 3, 15, 15), dtype=dtype, device=self.device)
        if with_contract and contract is None:
            contract = torch.empty((B, 10), dtype=dtype, device=self.device)
        _lib.check(self._h, self.lib.ssd_policy_inputs(self._h, _ptr(self._obs_buf), self.obs_stride, _lib.policy_dtype_code(dtype),
                                                       _ptr(image), _ptr(contract) if with_contract else None, self._stream()))
        return (image, contract) if with_contract else image

    # ---- NegotiationSolver (two_stage_train.py:619-776) ---------------------------------------------
    def solver_sample(self, num_samples):
        return solver_sample(self, num_samples)

    def solver_choose(self, params, vals, rule="majority"):
        return solver_choose(self, params, vals, rule)

    def get_state(self):
        E, n, dev = self.E, self.n, self.device
        st = {"map": torch.empty((E, self.H, self.W), dtype=torch.uint8, device=dev),
              "pos": torch.empty((E, n, 2), dtype=torch.int32, device=dev),
              "ori": torch.empty((E, n), dtype=torch.int32, device=dev),
              "t": torch.empty((E,), dtype=torch.int32, device=dev),
              "theta": torch.empty((E,), dtype=torch.float64, device=dev)}
        _lib.check(self._h, self.lib.ssd_get_state(self._h, _ptr(st["map"]), _ptr(st["pos"]), _ptr(st["ori"]),
                                                   _ptr(st["t"]), _ptr(st["theta"]), self._stream()))
        return st

    def set_state(self, map=None, pos=None, ori=None, t=None, theta=None):
        def prep(x, dt, shape):
            if x is None:
                return None
            return torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x).to(device=self.device, dtype=dt).expand(shape).contiguous()
        E, n = self.E, self.n
        m, p, o = prep(map, torch.uint8, (E, self.H, self.W)), prep(pos, torch.int32, (E, n, 2)), prep(ori, torch.int32, (E, n))
        tt, th = prep(t, torch.int32, (E,)), prep(theta, torch.float64, (E,))
        _lib.check(self._h, self.lib.ssd_set_state(self._h, _ptr(m), _ptr(p), _ptr(o), _ptr(tt), _ptr(th), self._stream()))

    def metrics_raw(self):
        out = torch.empty((self.E, _lib.METRIC_STRIDE), dtype=torch.float64, device=self.device)
        _lib.check(self._h, self.lib.ssd_get_metrics(self._h, _ptr(out), self._stream()))
        return out

    @property
    def kernel_launches(self):
        return int(self.lib.ssd_kernel_launches(self._h))

    def enable_timing(self, on=True):
        """bracket the step's kernels with CUDA events (measurement only; not graph-capturable)"""
        _lib.check(self._h, self.lib.ssd_enable_timing(self._h, 1 if on else 0))

    def step_times_ms(self):
        """(logic kernel ms, observe kernel ms) of the last step taken with timing enabled"""
        out = (ctypes.c_double * 2)()
        _lib.check(self._h, self.lib.ssd_get_step_times(self._h, out))
        return float(out[0]), float(out[1])

    @property
    def state_map_bytes(self):
        """bytes of the compact map inside an env record (rows padded to 4 cells, total to 16 bytes)"""
        return ((self.H * ((self.W + 3) // 4 * 4)) + 15) // 16 * 16

    @property
    def state_bytes_per_env(self):
        return int(self.lib.ssd_state_bytes_per_env(self._h))

"""The NegotiationSolver inside a vectorised sampler: each restarted env's contract chosen on the device.

In the reference every env is its own NegotiationSolver (two_stage_train.py:619-776): each reset samples 1 + S candidate
contracts, queries the frozen policy's value function for every candidate and agent, and installs the winner.  In a batch
stepped with auto_reset only the envs that were just reset need that.  A `SolverQueue` finds them on the device (an env
is *pending* at t == 0 of an episode whose contract the solver has not chosen) and serves them in windows of at most
`capacity` envs in env order (ssd_solver_rows / ssd_solver_resolve, include/ssd_b200.h):

    q = SolverQueue(batch, num_samples=50, capacity=256)     # capacity >= the envs that restart in one step
    ... per step, inside a CUDA graph if wished:
    batch.step(actions, auto_reset=True)
    rows, env, count = q.rows()[:3]         # value-query rows [C, 1 + S, n, W] of the window (zeros beyond it)
    theta, index = q.resolve(value_fn(rows))   # float64 [C, 1 + S, n] -> each window env's contract

After a full reset every env is pending at once: `q.run(value_fn)` loops windows until none is left.  Each env ends with
what `solver_sample` + `solver_choose` would give it on the same values.

Rows by the batch's observation form (W = the last dimension):
  - flat forms (BatchedFeatureEnv, BatchedCarEnv, BatchedGridEnv(image_obs=False)): obs ++ [param, 0], W = F + 2, float64
    (what NegotiationSolver._obs_with builds) or the policy dtype (the policy rows' feature columns, bit for bit);
  - image forms (BatchedGridEnv): the contract part alone, float64 (param, 0) with uint8 windows (W = 2), or the policy
    dtype (param, 0) x 5 with a policy image (W = 10).  The image is the same for every candidate: rows() also returns
    `image_index` [C * n], the rows of `obs.view(E * n, ...)` / `policy_image` to gather (env ids beyond the window read
    row 0..n-1 of env 0).
"""
import ctypes

import torch

from . import _lib


class SolverQueue:
    """The solver queue of one batch (any Batched*Env with a contract; one queue per batch)."""

    def __init__(self, env, num_samples=50, capacity=None, rule="majority"):
        if env.contract is None:
            raise ValueError("SolverQueue needs a batch with a contract")
        if rule not in _lib.SOLVER_RULE:
            raise ValueError("rule must be 'max' or 'majority', got %r" % (rule,))
        capacity = env.E if capacity is None else int(capacity)
        if not 1 <= capacity <= env.E:
            raise ValueError("capacity must be in [1, E = %d], got %d" % (env.E, capacity))
        self.batch, self.S, self.C, self.rule = env, int(num_samples), capacity, rule
        if self.S < 0:
            raise ValueError("num_samples must be >= 0")
        n, dev, C, S1 = env.n, env.device, capacity, self.S + 1
        self.image = False
        self.obs_required = False
        if hasattr(env, "image_obs") and env.image_obs:          # grid world, image forms: the contract part alone
            self.image = True
            self.width, self.dtype = (2, torch.float64) if env.policy_dtype is None else (10, env.policy_dtype)
        else:
            F = env.F if hasattr(env, "F") else env.D
            self.width = F + 2
            self.dtype = torch.float64 if env.policy_dtype is None else env.policy_dtype
            self.obs_required = env.policy_dtype is None and not hasattr(env, "image_obs")
        self.env = torch.full((C,), -1, dtype=torch.int32, device=dev)
        self.episode = torch.zeros((C,), dtype=torch.int32, device=dev)       # uint32 bits
        self.count = torch.zeros((2,), dtype=torch.int32, device=dev)          # uint32 bits: in window, pending in total
        self.params = torch.zeros((C, S1), dtype=torch.float64, device=dev)
        self.query_rows = torch.zeros((C, S1, n, self.width), dtype=self.dtype, device=dev)
        self.theta = torch.zeros((C,), dtype=torch.float64, device=dev)
        self.index = torch.full((C,), -1, dtype=torch.int32, device=dev)
        self.stale = torch.zeros((1,), dtype=torch.int32, device=dev)
        self._agent = torch.arange(n, dtype=torch.int64, device=dev)
        self._win = self._window(C, self.S, self.env, self.episode, self.count, self.params, self.query_rows)
        # pending(): a one-env window of its own, so that counting leaves the queue's window as it is
        self._probe = [torch.zeros((1,), dtype=torch.int32, device=dev), torch.zeros((1,), dtype=torch.int32, device=dev),
                       torch.zeros((2,), dtype=torch.int32, device=dev), torch.zeros((1, 1), dtype=torch.float64, device=dev),
                       torch.zeros((1, 1, n, self.width), dtype=self.dtype, device=dev)]
        self._probe_win = self._window(1, 0, *self._probe)
        _lib.check(env._h, env.lib.ssd_solver_enable(env._h, 1))
        env._solver_queue = self                  # the handle holds one record of resolved episodes

    @staticmethod
    def _window(C, S, env, episode, count, params, rows):
        return _lib.ssd_solver_window(struct_size=ctypes.sizeof(_lib.ssd_solver_window), num_samples=S, capacity=C,
                                      env_dev=env.data_ptr(), episode_dev=episode.data_ptr(), count_dev=count.data_ptr(),
                                      params_dev=params.data_ptr(), rows_dev=rows.data_ptr())

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.batch.device).cuda_stream)

    def _obs_ptr(self, obs):
        if obs is None and self.obs_required:
            obs = self.batch.obs
        return None if obs is None else ctypes.c_void_p(obs.data_ptr())

    def rows(self, obs=None):
        """Find the window, sample its candidates and write its value-query rows.  Returns (rows [C, 1 + S, n, W], env
        int32 [C] (-1 beyond the window), count int32 [2] (envs in the window, pending envs in total); device tensors,
        no synchronisation), plus image_index int64 [C * n] for the image forms.  obs: the float64 observation of a
        feature-env / selfdrive batch (default: batch.obs); None for every other form."""
        b = self.batch
        _lib.check(b._h, b.lib.ssd_solver_rows(b._h, ctypes.byref(self._win), self._obs_ptr(obs), self._stream()))
        if not self.image:
            return self.query_rows, self.env, self.count
        image_index = (self.env.clamp(min=0).to(torch.int64)[:, None] * b.n + self._agent).reshape(-1)
        return self.query_rows, self.env, self.count, image_index

    def resolve(self, vals):
        """vals float64 [C, 1 + S, n]: the value of every window row.  Installs each window env's contract; returns
        (theta float64 [C], index int32 [C]): the chosen parameter and candidate index, index -1 for an env that was
        stepped or reset since rows() (left unchanged; `stale` counts them) and for the slots beyond the window."""
        b = self.batch
        shape = (self.C, self.S + 1, b.n)
        if not (torch.is_tensor(vals) and vals.dtype == torch.float64 and vals.device == b.device and vals.is_contiguous()):
            vals = torch.as_tensor(vals, dtype=torch.float64, device=b.device).contiguous()
        if tuple(vals.shape) != shape:
            raise ValueError("vals must be [C, 1 + S, n] = %r, got %r" % (shape, tuple(vals.shape)))
        _lib.check(b._h, b.lib.ssd_solver_resolve(b._h, ctypes.byref(self._win), _lib.SOLVER_RULE[self.rule],
                                                  ctypes.c_void_p(vals.data_ptr()), ctypes.c_void_p(self.theta.data_ptr()),
                                                  ctypes.c_void_p(self.index.data_ptr()), ctypes.c_void_p(self.stale.data_ptr()),
                                                  self._stream()))
        return self.theta, self.index

    def pending(self):
        """The number of pending envs now (one synchronisation)."""
        b = self.batch
        obs = self._obs_ptr(None)
        _lib.check(b._h, b.lib.ssd_solver_rows(b._h, ctypes.byref(self._probe_win), obs, self._stream()))
        return int(self._probe[2][1].item())

    def run(self, value_fn, obs=None):
        """Resolve every pending env, one window after the other (after a full reset every env is pending).
        value_fn(*rows()) -> float64 [C, 1 + S, n].  Returns the number of envs resolved (one synchronisation per
        window)."""
        done = 0
        while True:
            out = self.rows(obs)
            self.resolve(value_fn(*out))
            cnt = self.count.tolist()
            done += cnt[0] - int(self.stale.item())
            if cnt[0] == 0 or cnt[1] <= cnt[0]:
                return done

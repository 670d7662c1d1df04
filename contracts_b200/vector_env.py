"""A vectorised, RLlib-`BaseEnv`-shaped adapter over a device batch: E environments behind ONE rollout worker.

The reference hands RLlib one Python env per rollout worker (`utils/ray_config_utils.py:140` `num_workers`,
`run_training.py:68`); RLlib's sampler talks to envs through `BaseEnv.poll()` / `send_actions()` / `try_reset()`
(ray/rllib/env/base_env.py).  `SSDVectorEnv` exposes E device-resident envs through exactly those three calls, with
the dict conventions of the reference's wrappers (`{env_id: {agent_id: ...}}`; observations as
`SeparateContractEnv._with_contract` builds them, two_stage_train.py:104-121; `dones[env_id]['__all__']`), and
  * ONE host -> device copy per `send_actions` (the action matrix) and ONE device -> host copy per `poll` (a packed
    snapshot of observations, rewards, dones, infos of all E envs: `BatchedGridEnv.host_snapshot`);
  * finished envs are reset by `try_reset(env_id)` (RLlib calls it after `dones['__all__']`), batched: the resets
    requested between two polls run as one masked device reset.
Arrays are also available without the dict building through `poll_arrays()` — for samplers that batch the policy
forward themselves the dict layer is pure overhead (INTEGRATION.md §2b has the measured rates).

The envs live on the device, so `get_sub_environments()` has no Python envs to offer an RLlib callback; the metrics the
reference's MetricsCallback (utils/logger_utils.py:126-151) reads from each env come from `episode_metrics()` instead:
every adapter keeps an episode log (contracts_b200/episodes.py) and drains it there.
"""
import numpy as np
import torch

from .batched import BatchedGridEnv
from .episodes import EpisodeLog


def _upload(v, actions_host):
    """one asynchronous host -> device copy of the action matrix; an event marks when the pinned staging buffer may be
    rewritten (two sends without a poll between them must not race with the copy still reading it)"""
    v._actions_dev.copy_(actions_host, non_blocking=True)
    if actions_host is v._actions_host:
        if v._uploaded is None:
            v._uploaded = torch.cuda.Event()
        v._uploaded.record(torch.cuda.current_stream(v.batch.device))


def _staging_free(v):
    if v._uploaded is not None:
        v._uploaded.synchronize()


def _open_episode_log(v, capacity):
    """the adapter's episode log (capacity None: 2 E records; 0: none)"""
    v._episode_log = None
    if capacity is None or capacity > 0:
        v._episode_log = EpisodeLog(v.batch, capacity)
        v.batch.set_episode_log(v._episode_log)


class _EpisodeMetricsMixin:
    def episode_metrics(self):
        """The metrics of every episode that ended since the last call (a reset of a finished or unfinished env ends it),
        sorted by (env_id, episode): per episode the dict the drop-in class's `metrics` returns at its last step, plus
        `env_id` (global) and `episode`.  One device -> host copy and synchronisation; what an RLlib callback calls in
        place of reading `get_sub_environments()`."""
        log = self._episode_log
        if log is None:
            raise ValueError("this adapter was created with episode_log_capacity=0")
        rec = log.drain()
        return [dict(m, env_id=int(e), episode=int(k)) for m, e, k in zip(log.metrics(rec), rec["env_id"], rec["episode"])]


class SSDVectorEnv(_EpisodeMetricsMixin):
    def __init__(self, kind, num_envs, num_agents, contract=None, horizon=1000, seed=73907, first_env_id=0, device=None,
                 ascii_map=None, one_hot_id=False, episode_log_capacity=None, **batch_kwargs):
        self.batch = BatchedGridEnv(kind, num_envs, num_agents, ascii_map=ascii_map, horizon=horizon, contract=contract,
                                    seed=seed, first_env_id=first_env_id, device=device, **batch_kwargs)
        _open_episode_log(self, episode_log_capacity)
        self.num_envs, self.num_agents, self.contract = int(num_envs), int(num_agents), contract
        self.agent_ids = ["a%d" % i for i in range(self.num_agents)]
        self.one_hot_id = one_hot_id
        self._actions_host = torch.full((self.num_envs, self.num_agents), 4, dtype=torch.uint8).pin_memory()
        self._actions_dev = torch.empty_like(self._actions_host, device=self.batch.device)
        self._uploaded = None         # event behind the last asynchronous upload out of _actions_host
        self._pending_reset = np.zeros(self.num_envs, dtype=np.uint8)
        self._fresh = None            # envs whose next poll() returns a reset observation (no reward / done yet)
        self._stepped = False
        self.batch.reset()
        self._theta = self.batch.get_state()["theta"].cpu().numpy() if contract else None
        self._fresh = np.ones(self.num_envs, dtype=bool)

    # ---- BaseEnv ---------------------------------------------------------------------------------------
    def send_actions(self, action_dict):
        """{env_id: {agent_id: action}}; agents that are absent stay put (action 4), as in the drop-in classes."""
        _staging_free(self)
        a = self._actions_host.numpy()
        a[:] = 4
        for e, acts in action_dict.items():
            for k, v in acts.items():
                a[e, int(k[1:])] = int(v)
        self.send_action_array(self._actions_host)

    def send_action_array(self, actions_host):
        """uint8 [E, n] pinned host tensor (or numpy array): one host -> device copy, then the step is enqueued."""
        if not torch.is_tensor(actions_host):
            _staging_free(self)
            self._actions_host.numpy()[:] = actions_host
            actions_host = self._actions_host
        self._flush_resets()
        _upload(self, actions_host)
        self.batch.step(self._actions_dev, extras=False)
        self._stepped = True
        self._fresh[:] = False

    def try_reset(self, env_id):
        """Queue env_id for reset; the observation arrives with the next poll() (RLlib accepts that: ASYNC_RESET_RETURN)."""
        self._pending_reset[env_id] = 1
        return None

    def _flush_resets(self):
        if self._pending_reset.any():
            mask = torch.from_numpy(self._pending_reset).to(self.batch.device, non_blocking=False)
            self.batch.reset(mask)
            if self.contract:
                self._theta = self.batch.get_state()["theta"].cpu().numpy()
            self._fresh = self._pending_reset.astype(bool)
            self._pending_reset[:] = 0
            self._stepped = False

    def poll_arrays(self):
        """-> dict of numpy arrays for all E envs from ONE device -> host copy: obs uint8 [E, n, 15, 15, 3], rew float64
        [E, n], done uint8 [E], info uint8 [E, n, 4] (+ `fresh` bool [E]: the env was just reset, rew / done are void)."""
        self._flush_resets()
        snap = self.batch.host_snapshot(index=None, extras=False)
        snap["fresh"] = self._fresh.copy()
        if not self._stepped:
            snap["rew"] = np.zeros_like(snap["rew"]); snap["done"] = np.zeros_like(snap["done"])
        return snap

    def poll(self):
        """-> (obs, rewards, dones, infos, off_policy_actions), each {env_id: {agent_id: value}} (BaseEnv.poll)."""
        s = self.poll_arrays()
        obs, rews, dones, infos = {}, {}, {}, {}
        img = s["obs"].astype(np.float64) / 255                    # `curr_obs / 255` (cleanup_new.py:204,258)
        cleanup = self.batch.kind == "cleanup_new"
        for e in range(self.num_envs):
            if not self._stepped and not s["fresh"][e]:            # nothing new for this env since the last poll
                continue
            o = {}
            for i, k in enumerate(self.agent_ids):
                d = {"image": img[e, i]}
                if self.one_hot_id:
                    v = np.zeros(self.num_agents); v[i] = 1; d["features"] = v
                if self.contract:                                  # SeparateContractEnv._with_contract (two_stage_train.py:104-111)
                    d["contract"] = np.array([self._theta[e], 0.0])
                o[k] = d
            obs[e] = o
            if s["fresh"][e]:
                continue
            rews[e] = {k: np.float64(s["rew"][e, i]) for i, k in enumerate(self.agent_ids)}
            dn = bool(s["done"][e])
            dones[e] = {"__all__": dn, "a0": dn, "a1": dn}         # the keys the reference hard-codes (cleanup_new.py:242)
            infos[e] = {k: ({"eaten_apples": int(s["info"][e, i, 0]), "cleaned_squares": int(s["info"][e, i, 1])} if cleanup else
                            {"eaten_apples": int(s["info"][e, i, 0]), "eaten_close_apples": int(s["info"][e, i, 1])})
                        for i, k in enumerate(self.agent_ids)}
        return obs, rews, dones, infos, {}

    def get_sub_environments(self):
        return []

    def stop(self):
        self.batch.close()


class _ArrayVectorEnv(_EpisodeMetricsMixin):
    """poll_arrays() / send_action_array() / try_reset() over a feature-env or selfdrive batch (same contract as
    `SSDVectorEnv`: one host -> device copy per send, one packed device -> host copy per poll, resets requested between two
    polls run as one masked device reset and show up as `fresh` envs in the next poll)."""

    def _setup(self, batch, action_dtype, idle_action, episode_log_capacity):
        self.batch = batch
        _open_episode_log(self, episode_log_capacity)
        self.num_envs, self.num_agents = batch.E, batch.n
        self.agent_ids = ["a%d" % i for i in range(self.num_agents)]
        self._idle = idle_action
        self._actions_host = torch.full((self.num_envs, self.num_agents), idle_action, dtype=action_dtype).pin_memory()
        self._actions_dev = torch.empty_like(self._actions_host, device=batch.device)
        self._uploaded = None
        self._pending_reset = np.zeros(self.num_envs, dtype=np.uint8)
        self._stepped = False
        batch.reset()
        self._fresh = np.ones(self.num_envs, dtype=bool)
        self._fields = [("obs", batch.obs), ("rew", batch.rew), ("done", batch.done)]
        self._packed = torch.empty((sum(t.numel() * t.element_size() for _, t in self._fields) + 8 * self.num_envs,),
                                   dtype=torch.uint8).pin_memory()

    def send_action_array(self, actions_host):
        if not torch.is_tensor(actions_host):
            _staging_free(self)
            self._actions_host.numpy()[:] = actions_host
            actions_host = self._actions_host
        self._flush_resets()
        _upload(self, actions_host)
        self.batch.step(self._actions_dev, extras=False)
        self._stepped = True
        self._fresh[:] = False

    def try_reset(self, env_id):
        self._pending_reset[env_id] = 1
        return None

    def _flush_resets(self):
        if self._pending_reset.any():
            self.batch.reset(torch.from_numpy(self._pending_reset).to(self.batch.device))
            self._fresh = self._pending_reset.astype(bool)
            self._pending_reset[:] = 0
            self._stepped = False

    def poll_arrays(self):
        """-> numpy arrays of all E envs from ONE device -> host copy: obs float64 [E, n, F], rew float64 [E, n], done uint8
        (features: [E]; selfdrive: [E, n + 1]), theta float64 [E], fresh bool [E] (just reset: rew / done are void)."""
        self._flush_resets()
        theta = self.batch.get_state()["theta"]
        parts = [t.reshape(-1).view(torch.uint8) for _, t in self._fields] + [theta.reshape(-1).view(torch.uint8)]
        self._packed.copy_(torch.cat(parts), non_blocking=False)
        buf, off, out = self._packed.numpy(), 0, {}
        for name, t in self._fields + [("theta", theta)]:
            nbytes = t.numel() * t.element_size()
            dt = {torch.float64: np.float64, torch.uint8: np.uint8}[t.dtype]
            out[name] = buf[off:off + nbytes].view(dt).reshape(tuple(t.shape)).copy()
            off += nbytes
        out["fresh"] = self._fresh.copy()
        if not self._stepped:
            out["rew"] = np.zeros_like(out["rew"]); out["done"] = np.zeros_like(out["done"])
        return out

    def get_sub_environments(self):
        return []

    def stop(self):
        self.batch.close()


class SSDFeatureVectorEnv(_ArrayVectorEnv):
    """E CleanupFeatures / HarvestFeatures envs ('cleanup' / 'harvest') behind one rollout worker; `poll()` returns the flat
    observations of the non-convolutional wrapper, features ++ [theta, 0] (two_stage_train.py:104-121)."""

    def __init__(self, kind, num_envs, num_agents, contract=None, horizon=1000, seed=73907, first_env_id=0, device=None,
                 ascii_map=None, episode_log_capacity=None):
        from .features import BatchedFeatureEnv
        self.contract = contract
        self._setup(BatchedFeatureEnv(kind, num_envs, num_agents, ascii_map=ascii_map, horizon=horizon, contract=contract,
                                      seed=seed, first_env_id=first_env_id, device=device), torch.uint8, 4, episode_log_capacity)

    def send_actions(self, action_dict):
        _staging_free(self)
        a = self._actions_host.numpy()
        a[:] = self._idle
        for e, acts in action_dict.items():
            for k, v in acts.items():
                a[e, int(k[1:])] = int(v)
        self.send_action_array(self._actions_host)

    def poll(self):
        s = self.poll_arrays()
        obs, rews, dones, infos = {}, {}, {}, {}
        for e in range(self.num_envs):
            if not self._stepped and not s["fresh"][e]:
                continue
            tail = np.array([s["theta"][e], 0.0])
            obs[e] = {k: (np.concatenate((s["obs"][e, i], tail)) if self.contract else s["obs"][e, i].copy()) for i, k in enumerate(self.agent_ids)}
            if s["fresh"][e]:
                continue
            rews[e] = {k: np.float64(s["rew"][e, i]) for i, k in enumerate(self.agent_ids)}
            dn = bool(s["done"][e])
            dones[e] = {"__all__": dn, "a0": dn, "a1": dn}
            infos[e] = {k: {} for k in self.agent_ids}
        return obs, rews, dones, infos, {}


class SSDCarVectorEnv(_ArrayVectorEnv):
    """E SelfAcceleratingCarEnv envs behind one rollout worker (arrays only: float32 accelerations [E, n] in; cars that are
    done are flagged in done[:, k] and their actions are ignored)."""

    def __init__(self, num_envs, num_agents, contract=None, seed=73907, first_env_id=0, device=None, episode_log_capacity=None,
                 **batch_kwargs):
        from .selfdrive import BatchedCarEnv
        self.contract = contract
        self._setup(BatchedCarEnv(num_envs, num_agents, contract=contract, seed=seed, first_env_id=first_env_id, device=device,
                                  **batch_kwargs), torch.float32, 0.0, episode_log_capacity)

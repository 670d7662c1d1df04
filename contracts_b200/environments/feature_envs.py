"""`CleanupFeatures` / `HarvestFeatures` with the reference's constructor and dict API
(environments/cleanup_features.py:48-336, environments/harvest_features.py:60-364), stepping on the GPU.

`image_obs=True` (HarvestFeatures' un-rotated colour window, unused by every shipped config) is rejected.  Randomness is
the counter-based Philox stream (kwargs `seed`, `env_id`).
"""
import numpy as np
import torch

from .. import spaces
from ..features import BatchedFeatureEnv
from ..maps import CLEANUP_MAP, HARVEST_MAP
from .gridworld import _num, equality, sustainability


class _FeatureEnv:
    KIND, MAP = None, None

    def __init__(self, num_agents=2, horizon=1000, image_obs=False, num_envs=1, seed=73907, env_id=0, device=None, **kwargs):
        if image_obs:
            raise NotImplementedError("image_obs=True is not part of the accelerated feature envs")
        self.map = self.MAP
        self.num_agents, self.horizon, self.image_obs = int(num_agents), int(horizon), image_obs
        self.num_envs, self.seed, self.env_id, self.device = int(num_envs), int(seed), int(env_id), device
        self.timesteps = 0
        self.agent_ids = ["a%d" % i for i in range(self.num_agents)]
        self._make_spaces()
        self._contract = None
        self._batch = None
        self._last = None

    @property
    def batch(self):
        if self._batch is None:
            c = self._contract or (None, 0.0, 0.0, 0.0)
            self._batch = BatchedFeatureEnv(self.KIND, self.num_envs, self.num_agents, self.map, horizon=self.horizon,
                                            contract=c[0], theta_low=c[1], theta_high=c[2], null_prob=c[3], seed=self.seed,
                                            first_env_id=self.env_id, device=self.device)
        return self._batch

    def _bind_contract(self, name, low, high, null_prob):
        if self._batch is not None:
            self._batch.close()
            self._batch = None
        self._contract = (name, float(low), float(high), float(null_prob))

    def reset(self):
        obs = self.batch.reset()[0].cpu().numpy()
        self.timesteps = 0
        return {k: obs[i].copy() for i, k in enumerate(self.agent_ids)}

    def step(self, acts):
        b = self.batch
        a = np.full((self.num_envs, self.num_agents), 4, dtype=np.uint8)
        for k, v in acts.items():
            a[0, int(k[1:])] = int(v)
        obs, rew, done, info = b.step(torch.from_numpy(a).to(b.device))
        self.timesteps += 1
        L = {"obs": obs[0].cpu().numpy(), "rew": rew[0].cpu().numpy(), "base_rew": b.base_rew[0].cpu().numpy(),
             "transfers": b.transfers[0].cpu().numpy(), "info": info[0].cpu().numpy(), "done": bool(done[0].item())}
        self._last = L
        d = L["done"]
        dones = {"__all__": d, "a0": d, "a1": d}
        obs_d = {k: self._step_obs(L["obs"][i]) for i, k in enumerate(self.agent_ids)}
        rews = {k: float(L["base_rew"][i]) for i, k in enumerate(self.agent_ids)}
        infos = {k: self._agent_info(L["info"][i], L["obs"][i]) for i, k in enumerate(self.agent_ids)}
        return obs_d, rews, dones, infos

    @property
    def metrics(self):
        raw = self.batch.metrics_raw()[0].cpu().numpy()
        return feature_metrics(self.KIND, raw, self.num_agents, self.timesteps == self.horizon,
                               contract=self._contract is not None and self._contract[0] is not None)

    def compute_equality(self, reward_dict):
        return equality([sum(v) for v in reward_dict.values()])

    def compute_sustainability(self, reward_dict):
        return sustainability([sum(v) for v in reward_dict.values()], [sum(t * r for t, r in enumerate(v)) for v in reward_dict.values()])

    def render(self):
        pass

    def close(self):
        if self._batch is not None:
            self._batch.close()
            self._batch = None


class CleanupFeatures(_FeatureEnv):
    """environments/cleanup_features.py CleanupFeatures ('Cleanup')."""
    KIND, MAP = "cleanup", CLEANUP_MAP

    def _make_spaces(self):
        n, H, W = self.num_agents, len(self.map), len(self.map[0])
        flat = "".join(self.map)
        self.observation_space = spaces.Box(
            low=np.array([0.0] * (12 + n)),
            high=np.array([H, W, 4, H, W, 4, H, W, H, W, flat.count("B") + 1, flat.count("H") + flat.count("R") + 1] + [np.inf] * n))
        self.action_space = spaces.Discrete(8)
        self.continuous_action_space = spaces.Box(low=-10.0, high=10.0, shape=(8,))

    def _step_obs(self, row):
        return row.astype(np.int64)         # the reference builds the step observation from ints only (:234-240)

    def _agent_info(self, info, obs):
        return {"cleaned_squares": int(info[0])}


class HarvestFeatures(_FeatureEnv):
    """environments/harvest_features.py HarvestFeatures ('Harvest')."""
    KIND, MAP = "harvest", HARVEST_MAP

    def _make_spaces(self):
        n, H, W = self.num_agents, len(self.map), len(self.map[0])
        na = "".join(self.map).count("A")
        self.observation_space = spaces.Box(low=np.array([0.0] * (10 + 2 * n)),
                                            high=np.array([H, W, 4, H, W, 4, H, W, na + 1, na + 1] + [1] * (2 * n)))
        self.action_space = spaces.Discrete(7)
        self.continuous_action_space = spaces.Box(low=-10.0, high=10.0, shape=(7,))

    def _step_obs(self, row):
        return row.copy()

    def _agent_info(self, info, obs):
        return {"eaten_apples": int(info[0]), "eaten_close_apples": int(info[1]), "feature_obs": obs.copy()}


def feature_metrics(kind, raw, n, ended, contract=False):
    """The `metrics` dict of a CleanupFeatures / HarvestFeatures env (kind 'cleanup' / 'harvest') from its
    ssd_feat_get_metrics row `raw` (float64 [40] or longer, numpy).  ended: the episode reached its horizon (equality /
    sustainability are added then, and transfer_* with a contract)."""
    raw_rew = float(raw[1]) if raw[1] else 0
    if kind == "cleanup":
        m = {"dirt_cleaned": int(raw[0]), "raw_env_rewards": raw_rew, "transfers": _num(raw[2])}
    else:
        m = {"total_apples_eaten": int(raw[3]), "low_density_apples_eaten": int(raw[4]), "raw_env_rewards": raw_rew,
             "transfers": _num(raw[2])}
    if ended:
        m["equality"] = equality(list(raw[8:8 + n]))
        m["sustainability"] = sustainability(list(raw[8:8 + n]), list(raw[16:16 + n]))
        if contract:
            m["transfer_sustainability"] = sustainability(list(raw[24:24 + n]), list(raw[32:32 + n]))
            m["transfer_equality"] = equality(list(raw[24:24 + n]))
    return m

"""`CleanupEnv` / `HarvestEnv` with the reference's constructor kwargs and dict API
(environments/cleanup_new.py:59-267, environments/harvest_new.py:48-239), stepping on the GPU.

Each object owns `num_envs` environments (default 1) in one `BatchedGridEnv`.  The RLlib-style
`reset()` / `step({aid: action})` dict API addresses env `0` of that batch and is meant for
compatibility (one host round trip per call); throughput users step `self.batch` with device tensors.

Differences from the reference that a caller can observe:
  * randomness is a counter-based Philox stream keyed (seed, env_id) instead of the process-global
    NumPy / stdlib generators (kwargs `seed`, `env_id`); given the same draws the results are
    bit-identical (tests/test_dropin_api.py replays the reference's golden vectors through this API);
  * `render(mode="human")` does not open a matplotlib window: every mode returns the RGB frame.

`use_collective_reward` / `inequity_averse_reward` (+ `alpha`, `beta`; map_env.py:289-301) run on the
device (fused into the reward write).  `return_agent_actions` is accepted and has, as in the reference,
no effect on what CleanupEnv / HarvestEnv return: their `step`/`reset` keep only `curr_obs` of the
MapEnv observation dict (cleanup_new.py:204,258; harvest_new.py:171,230), so `other_agent_actions`,
`visible_agents` and `prev_visible_agents` (map_env.py:271-282) never reach the caller.
"""
import numpy as np
import torch

from .. import _lib, spaces
from ..batched import BatchedGridEnv
from ..maps import CLEANUP_MAP, HARVEST_MAP

class _GridWorldEnv:
    KIND = None
    DEFAULT_MAP = None
    N_ACTIONS = (0, 0)      # (disable_firing, firing enabled)

    def __init__(self, ascii_map=None, num_agents=1, disable_firing=True, image_obs=True,
                 return_agent_actions=False, use_collective_reward=False, inequity_averse_reward=False,
                 alpha=0.0, beta=0.0, horizon=1000, one_hot_id=False,
                 num_envs=1, seed=73907, env_id=0, device=None, **kwargs):
        if inequity_averse_reward and int(num_agents) < 2:
            raise AssertionError("Cannot use inequity aversion with only one agent!")     # map_env.py:294
        self.return_agent_actions = return_agent_actions
        self.use_collective_reward, self.inequity_averse_reward = bool(use_collective_reward), bool(inequity_averse_reward)
        self.alpha, self.beta = alpha, beta
        self.ascii_map = list(self.DEFAULT_MAP if ascii_map is None else ascii_map)
        self.num_agents = int(num_agents)
        self.disable_firing, self.image_obs, self.one_hot_id = disable_firing, image_obs, one_hot_id
        self.horizon = int(horizon)
        self.num_envs, self.seed_value, self.env_id, self.device = int(num_envs), int(seed), int(env_id), device
        self.agent_ids = ["a%d" % i for i in range(self.num_agents)]
        self.base_map = np.array([[c.encode() for c in row] for row in self.ascii_map])
        self._make_spaces()
        self._contract = None           # (class name, low, high, null_prob) once a contract wrapper binds
        self._batch = None
        self.timesteps = 0
        self._last_infos = None

    # ---- spaces (cleanup_new.py:90-169, harvest_new.py:85-130) ---------------------------------------
    def _make_spaces(self):
        n = self.num_agents
        na = self.N_ACTIONS[0 if self.disable_firing else 1]
        H, W = len(self.ascii_map), len(self.ascii_map[0])
        self.action_space = spaces.Discrete(na)
        self.continuous_action_space = spaces.Box(low=-10.0, high=10.0, shape=(na,))
        self.global_action_space = spaces.MultiDiscrete([na] * n)
        self.global_observation_space = spaces.Dict({"image": spaces.Box(low=0, high=1, shape=(H, W, 3), dtype=np.uint8)})
        self.concatenated_observation_space = spaces.Dict(
            {"image": spaces.Box(low=0, high=1, shape=(15, 15, 3 * n), dtype=np.uint8)})
        if not self.image_obs:
            self.observation_space = self._feature_space(H, W)
        else:
            d = {"image": spaces.Box(low=0, high=1, shape=(15, 15, 3), dtype=np.uint8)}
            if self.one_hot_id:
                d["features"] = spaces.Box(low=0, high=1, shape=(n,))
            self.observation_space = spaces.Dict(d)

    # ---- device batch -------------------------------------------------------------------------------
    @property
    def batch(self):
        if self._batch is None:
            c = self._contract or (None, 0.0, 0.0, 0.0)
            self._batch = BatchedGridEnv(self.KIND, self.num_envs, self.num_agents, self.ascii_map, horizon=self.horizon,
                                         contract=c[0], theta_low=c[1], theta_high=c[2], null_prob=c[3],
                                         seed=self.seed_value, first_env_id=self.env_id, device=self.device,
                                         use_collective_reward=self.use_collective_reward,
                                         inequity_averse_reward=self.inequity_averse_reward,
                                         alpha=self.alpha, beta=self.beta)
            try:                     # render() shows the beams of the last step (MapEnv.beam_pos); cheap at dict-API batch sizes
                self._batch.record_beams(True)
            except _lib.SsdError:    # the single-kernel fallback (maps > 1 KB) does not record them
                pass
        return self._batch

    def seed(self, seed=None):
        """MapEnv.seed (map_env.py:344-345) reseeds NumPy's global generator; here the Philox key of this env's stream.
        Takes effect at the next reset (the device handle is rebuilt)."""
        if seed is not None:
            self.seed_value = int(seed)
            if self._batch is not None:
                self._batch.close()
                self._batch = None
        return [self.seed_value]

    @property
    def agent_pos(self):
        """[[row, col], ...] of the agents in agent order (map_env.py:347-352)."""
        return self.batch.get_state()["pos"][0].cpu().numpy().tolist()

    def _bind_contract(self, name, low, high, null_prob):
        """Called by the contract wrappers: rebuild the device handle with the contract fused in."""
        if self._batch is not None:
            self._batch.close()
            self._batch = None
        self._contract = (name, float(low), float(high), float(null_prob))

    # ---- helpers ------------------------------------------------------------------------------------------
    def one_hot(self, key):
        v = np.zeros(self.num_agents)
        v[int(key[1:])] = 1
        return v

    def _image_obs(self, obs_u8):
        out = {}
        for i, k in enumerate(self.agent_ids):
            o = {"image": obs_u8[i].astype(np.float64) / 255}       # `curr_obs / 255` (cleanup_new.py:204,258)
            if self.one_hot_id:
                o["features"] = self.one_hot(k)
            out[k] = o
        return out

    def _actions_tensor(self, acts):
        a = np.full((self.num_envs, self.num_agents), 4, dtype=np.uint8)     # absent agents stay put
        for k, v in acts.items():
            a[0, int(k[1:])] = int(v)
        return torch.from_numpy(a).to(self.batch.device)

    # ---- MultiAgentEnv API --------------------------------------------------------------------------------
    def reset(self):
        obs = self.batch.reset()[0].cpu().numpy()
        self.timesteps = 0
        if not self.image_obs:
            return self._reset_feature_obs()
        return self._image_obs(obs)

    def step(self, acts):
        b = self.batch
        b.step(self._actions_tensor(acts), want_features=True)
        self.timesteps += 1
        snap = b.host_snapshot(index=0, features=True)             # one packed device -> host copy (was seven)
        self._last = {k: np.array(v) for k, v in snap.items()}
        self._last["done"] = bool(snap["done"])
        L = self._last
        infos = {}
        for i, k in enumerate(self.agent_ids):
            infos[k] = self._agent_info(L["info"][i])
            infos[k]["feature_obs"] = L["feat"][i].copy()
        d = L["done"]
        dones = {"__all__": d, "a0": d, "a1": d}            # the reference hard-codes these keys (cleanup_new.py:242)
        rews = {k: (np.float64(L["base_rew"][i]) if self.inequity_averse_reward else int(L["base_rew"][i]))
                for i, k in enumerate(self.agent_ids)}
        if not self.image_obs:
            obs_d = {k: L["feat"][i].copy() for i, k in enumerate(self.agent_ids)}
        else:
            obs_d = self._image_obs(L["obs"])
        self._last_infos = infos
        return obs_d, rews, dones, infos

    # ---- metrics (cleanup_new.py:186-189,213-232,264-266; harvest_new.py:152-155; two_stage_train.py:92-99) ----
    @property
    def metrics(self):
        raw = self.batch.metrics_raw()[0].cpu().numpy()
        if raw[5] != 0:
            raise RuntimeError("device error flags %d" % int(raw[5]))
        return grid_metrics(self.KIND, raw, self.num_agents, self.timesteps == self.horizon,
                            contract=self._contract is not None and self._contract[0] is not None,
                            float_rewards=self.inequity_averse_reward)

    def compute_equality(self, reward_dict):
        return equality([sum(v) for v in reward_dict.values()])

    def compute_sustainability(self, reward_dict):
        return sustainability([sum(v) for v in reward_dict.values()],
                              [sum(t * r for t, r in enumerate(v)) for v in reward_dict.values()])

    # ---- rendering ---------------------------------------------------------------------------------------------
    def full_map_to_colors(self):
        """RGB image of the whole map with the agents and the beams of the last step (map_env.py:354-375,389-392),
        written by the device (`ssd_render`)."""
        return self.batch.render()[0].cpu().numpy().astype(int)

    def global_view(self):
        """world_map_color without its padding (map_env.py:394-395), written by the device (`ssd_global_view`).  Unlike
        `full_map_to_colors` it shows the agents only from the first step on (MapEnv.reset does not paint them)."""
        return self.batch.global_view()[0].cpu().numpy()

    def get_global_obs(self):
        return {"image": self.global_view() / 255}

    def render(self, filename=None, mode="rgb_array"):
        return self.full_map_to_colors()

    def close(self):
        if self._batch is not None:
            self._batch.close()
            self._batch = None


def grid_metrics(kind, raw, n, ended, contract=False, float_rewards=False):
    """The `metrics` dict of a cleanup_new / harvest_new env (cleanup_new.py:186-189,213-232,264-266; harvest_new.py:152-155;
    two_stage_train.py:92-99) from its ssd_get_metrics row `raw` (float64 [56], numpy).  ended: the episode reached its
    horizon (the reference adds equality / sustainability then, and transfer_* with a contract).  float_rewards: env
    rewards are float64 (inequity aversion, map_env.py:293-300), else Python ints."""
    rew = float if float_rewards else int
    if kind == "cleanup_new":
        m = {"total_apples_eaten": int(raw[0]), "raw_env_rewards": rew(raw[2]), "dirt_cleaned": int(raw[4])}
        for i in range(n):
            m["a%d-waste_cleaned" % i] = int(raw[8 + i])
    else:
        m = {"total_apples_eaten": int(raw[0]), "low_density_apples_eaten": int(raw[1]), "raw_env_rewards": rew(raw[2])}
        for i in range(n):
            m["a%d-apples_consumed" % i] = int(raw[8 + i])
            m["a%d-close_apples_consumed" % i] = int(raw[16 + i])
    m["transfers"] = _num(raw[3])
    if ended:
        m["equality"] = equality([rew(x) for x in raw[24:24 + n]])
        m["sustainability"] = sustainability([rew(x) for x in raw[24:24 + n]], [rew(x) for x in raw[32:32 + n]])
        if contract:
            m["transfer_sustainability"] = sustainability(list(raw[40:40 + n]), list(raw[48:48 + n]))
            m["transfer_equality"] = equality(list(raw[40:40 + n]))
    return m


def _num(x):
    return int(x) if float(x).is_integer() else float(x)


def equality(totals):
    """1 - sum_ij |R_i - R_j| / (2 n sum R)  (cleanup_new.py:422-434), same operation order."""
    eq, total = 0, 0
    n = len(totals)
    for i in totals:
        for j in totals:
            eq += abs(i - j)
        total += i
    if total == 0:
        total = 0.001
    return 1 - eq / (2 * n * total)


def sustainability(totals, tsums):
    """mean_k sum_t t r_t / max(sum_t r_t, 1)  (cleanup_new.py:436-445)."""
    return np.mean([ts / max(tot, 1) for tot, ts in zip(totals, tsums)])


def _closest(points, pos):
    """np.argmin of L1 distances over a row-major point list: first minimum wins (cleanup_new.py:396-403)."""
    if len(points) == 0:
        return [0, 0]
    d = np.sum(np.abs(np.asarray(points) - np.asarray(pos)), axis=1)
    return list(points[int(np.argmin(d))])


class CleanupEnv(_GridWorldEnv):
    """environments/cleanup_new.py CleanupEnv ('CleanupNew')."""
    KIND, DEFAULT_MAP, N_ACTIONS = "cleanup_new", CLEANUP_MAP, (8, 9)

    def _feature_space(self, H, W):
        n = self.num_agents
        flat = "".join(self.ascii_map)
        n_apple, area = flat.count("B"), flat.count("H") + flat.count("R")
        return spaces.Box(low=np.array([0.0] * (12 + n)),
                          high=np.array([H, W, 4, H, W, 4, H, W, H, W, n_apple + 1, area + 1] + [np.inf] * n))

    def _agent_info(self, row):
        return {"eaten_apples": int(row[0]), "cleaned_squares": int(row[1])}

    def _reset_feature_obs(self):
        """Feature observation at reset (cleanup_new.py:193-202), computed on the host from the device state."""
        st = self.batch.get_state()
        pos, ori = st["pos"][0].cpu().numpy(), st["ori"][0].cpu().numpy()
        # custom_reset fills these caches BEFORE the reset-time spawn (map_env.py:319-320): no apples yet,
        # waste = the map's initial 'H' cells
        apples = np.zeros((0, 2), dtype=int)
        wastes = np.argwhere(self.base_map == b"H")
        out = {}
        n = self.num_agents
        for i, k in enumerate(self.agent_ids):
            j = (1 if n > 1 else 0) if i == 0 else 0          # closest_pos quirk (cleanup_new.py:405-412)
            ca, cw = _closest(apples, pos[i]), _closest(wastes, pos[i])
            out[k] = np.array([float(pos[i][0]), float(pos[i][1]), float(ori[i]), float(pos[j][0]), float(pos[j][1]),
                               float(ori[j]), float(ca[0]), float(ca[1]), float(cw[0]), float(cw[1]),
                               len(apples), len(wastes)] + [0.0] * n)
        return out


class HarvestEnv(_GridWorldEnv):
    """environments/harvest_new.py HarvestEnv ('HarvestNew')."""
    KIND, DEFAULT_MAP, N_ACTIONS = "harvest_new", HARVEST_MAP, (7, 8)

    def _feature_space(self, H, W):
        n = self.num_agents
        n_apple = "".join(self.ascii_map).count("A")
        return spaces.Box(low=np.array([0.0] * (10 + 2 * n)),
                          high=np.array([H, W, 4, H, W, 4, H, W, n_apple + 1, n_apple + 1] + [1] * (2 * n)))

    def _agent_info(self, row):
        return {"eaten_apples": int(row[0]), "eaten_close_apples": int(row[1])}

    def _reset_feature_obs(self):
        """Feature observation at reset (harvest_new.py:160-168)."""
        st = self.batch.get_state()
        chars, pos, ori = st["map"][0].cpu().numpy(), st["pos"][0].cpu().numpy(), st["ori"][0].cpu().numpy()
        apples = np.argwhere(chars == ord("A"))
        n = self.num_agents
        H, W = chars.shape
        out = {}
        for i, k in enumerate(self.agent_ids):
            j = (1 if n > 1 else 0) if i == 0 else 0
            ca = _closest(apples, pos[i])
            close = 0                                    # count_apples_in_radius(5, pos) (harvest_new.py:326-336)
            for dr in range(-5, 6):
                for dc in range(-5, 6):
                    r, c = pos[i][0] + dr, pos[i][1] + dc
                    if dr * dr + dc * dc <= 5 and 0 <= r < H and 0 <= c < W and chars[r, c] == ord("A"):
                        close += 1
            out[k] = np.array([float(pos[i][0]), float(pos[i][1]), float(ori[i]), float(pos[j][0]), float(pos[j][1]),
                               float(ori[j]), float(ca[0]), float(ca[1]), float(close), float(len(apples))]
                              + [0.0] * (2 * n))
        return out

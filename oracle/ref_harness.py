"""Run the UNMODIFIED reference env code under counter-based RNG injection.

TEST INFRASTRUCTURE (oracle/), needs a checkout of the original project (SSD_REFERENCE_ROOT).  This is the
ground truth that pins both the C oracle (`oracle/ssd_oracle.c`) and the CUDA path: every
RNG call site of SURVEY.md §8a table R is monkey-patched (no reference source is edited or
copied) to read from the Philox stream defined in `oracle/philox.py`.  The golden vectors in
`tests/golden/` are produced from here by `oracle/make_golden.py`.

Patched names and the reference call sites they serve:
  np.random.shuffle  <- map_env.py:546 (R1), :685 (R2), :821 (R7); cleanup_new.py:339 (R4)
  np.random.randint  <- map_env.py:831 (R6); cleanup_features.py:109 / harvest_features.py:122 (R11)
  np.random.rand / np.random.uniform <- two_stage_train.py:163-164 (R8)
  environments.cleanup_new.rand / environments.harvest_new.rand <- cleanup_new.py:326, harvest_new.py:294 (R3/R5)
  random.sample / random.random <- two_stage_train.py:271,276 (R9); self_driving_car_accelerate.py:53,57 (R10);
                                   cleanup_features.py:115,122 / harvest_features.py:148 (R11)
  random.shuffle     <- cleanup_features.py:107 / harvest_features.py:118 (R11)
"""
import random as _pyrandom
import sys

import numpy as np

from . import philox as px
from . import ref_stubs

_CTX = None          # active DrawContext (None -> original RNG functions run)
_INSTALLED = False
_ORIG = {}


class DrawContext:
    """Identifies the Philox stream position of the env currently being driven."""

    def __init__(self, seed, env_id):
        self.seed = int(seed)
        self.env_id = int(env_id)
        self.episode = px.EPISODE_CONSTRUCT
        self.t = 0
        self.calls = {}

    def begin(self, episode, t):
        self.episode = int(episode)
        self.t = int(t)
        self.calls = {}

    def next_call(self, site):
        c = self.calls.get(site, 0)
        self.calls[site] = c + 1
        return c

    def u32(self, site, call, idx):
        return px.draws_u32(self.seed, self.env_id, self.episode, self.t, site, call, idx)

    def f64(self, site, call, idx):
        return px.draws_f64(self.seed, self.env_id, self.episode, self.t, site, call, idx)


class active:
    """`with active(ctx):` routes the patched RNG names to ctx."""

    def __init__(self, ctx):
        self.ctx = ctx

    def __enter__(self):
        global _CTX
        self.prev = _CTX
        _CTX = self.ctx
        return self.ctx

    def __exit__(self, *a):
        global _CTX
        _CTX = self.prev


def _caller_name(depth=2):
    return sys._getframe(depth).f_code.co_name


def _stateless_shuffle(x, site, canonical_sort):
    ctx = _CTX
    if canonical_sort:
        x.sort()
    call = ctx.next_call(site)
    keys = ctx.u32(site, call, np.arange(len(x)))
    order = np.argsort(keys, kind="stable")
    x[:] = [x[i] for i in order]


def _np_shuffle(x):
    if _CTX is None:
        return _ORIG["np.shuffle"](x)
    who = _caller_name()
    if who == "update_moves":
        _stateless_shuffle(x, px.SITE_MOVE_ORDER, False)
    elif who == "update_custom_moves":
        _stateless_shuffle(x, px.SITE_BEAM_ORDER, False)
    elif who == "spawn_apples_and_waste":
        _stateless_shuffle(x, px.SITE_WASTE_ORDER, True)
    elif who == "spawn_point":
        _stateless_shuffle(x, px.SITE_SPAWN_POINT, True)
    else:
        raise RuntimeError("np.random.shuffle from unexpected site %r" % who)


def _np_randint(*args, **kw):
    if _CTX is None:
        return _ORIG["np.randint"](*args, **kw)
    who = _caller_name()
    if who == "spawn_rotation":          # map_env.py:831  randint(4)
        site = px.SITE_SPAWN_ROT
    elif who in ("reset", "initialize_players"):   # feature envs: randint(0, 4)
        site = px.SITE_FEAT_ROT
    else:
        raise RuntimeError("np.random.randint from unexpected site %r" % who)
    call = _CTX.next_call(site)
    return int(_CTX.u32(site, call, 0)[0] >> np.uint32(30))


def _np_rand(*shape):
    if _CTX is None:
        return _ORIG["np.rand"](*shape)
    if shape:
        raise RuntimeError("np.random.rand(shape) from unexpected site %r" % _caller_name())
    return float(_CTX.f64(px.SITE_CONTRACT, 0, 0)[0])       # two_stage_train.py:163


def _np_uniform(low=0.0, high=1.0, size=None):
    if _CTX is None:
        return _ORIG["np.uniform"](low, high, size)
    if _caller_name() == "sample":                            # gym Box.sample <- negotiate (two_stage_train.py:725)
        u = _CTX.f64(px.SITE_SOLVER, 0, _CTX.next_call(px.SITE_SOLVER))[0]
    else:
        u = _CTX.f64(px.SITE_CONTRACT, 0, 1)[0]               # two_stage_train.py:164
    low64 = np.asarray(low, dtype=np.float64)
    high64 = np.asarray(high, dtype=np.float64)
    return low64 + (high64 - low64) * u


def _spawn_rand(k):
    """Replacement for the module-level `rand` of cleanup_new / harvest_new (R3/R5)."""
    if _CTX is None:
        return _ORIG["np.rand"](k)
    return _CTX.f64(px.SITE_SPAWN_DRAWS, 0, np.arange(k))


def _py_random():
    if _CTX is None:
        return _ORIG["py.random"]()
    who = _caller_name()
    if who == "step":                      # two_stage_train.py:276 (negotiate)
        return float(_CTX.f64(px.SITE_NEGOTIATE, 1, 0)[0])
    if who == "reset":                     # self_driving_car_accelerate.py:53,57: one draw per agent
        call = _CTX.next_call(px.SITE_SELFDRIVE_RESET)
        return float(_CTX.f64(px.SITE_SELFDRIVE_RESET, 0, call)[0])
    if who in ("spawn_apples_and_waste", "spawn_apples"):   # feature envs, sequential draws
        call = _CTX.next_call(px.SITE_FEAT_SPAWN)
        return float(_CTX.f64(px.SITE_FEAT_SPAWN, 0, call)[0])
    raise RuntimeError("random.random from unexpected site %r" % who)


def _py_sample(population, k):
    if _CTX is None:
        return _ORIG["py.sample"](population, k)
    pop = list(population)                 # two_stage_train.py:271  random.sample(range(1, n), 2)
    keys = _CTX.u32(px.SITE_NEGOTIATE, 0, np.arange(len(pop)))
    order = np.argsort(keys, kind="stable")
    return [pop[i] for i in order[:k]]


def _py_shuffle(x):
    if _CTX is None:
        return _ORIG["py.shuffle"](x)
    _stateless_shuffle(x, px.SITE_FEAT_ORDER, False)


def install():
    """Import the reference under stubs and patch its RNG call sites (idempotent)."""
    global _INSTALLED
    if _INSTALLED:
        return
    ref_stubs.install()
    import environments.cleanup_new as cn
    import environments.harvest_new as hn
    _ORIG.update({
        "np.shuffle": np.random.shuffle, "np.randint": np.random.randint,
        "np.rand": np.random.rand, "np.uniform": np.random.uniform,
        "py.random": _pyrandom.random, "py.sample": _pyrandom.sample,
        "py.shuffle": _pyrandom.shuffle,
    })
    np.random.shuffle = _np_shuffle
    np.random.randint = _np_randint
    np.random.rand = _np_rand
    np.random.uniform = _np_uniform
    cn.rand = _spawn_rand
    hn.rand = _spawn_rand
    _pyrandom.random = _py_random
    _pyrandom.sample = _py_sample
    _pyrandom.shuffle = _py_shuffle
    _INSTALLED = True


ORI_INT = {"UP": 0, "RIGHT": 1, "DOWN": 2, "LEFT": 3}


class RefGridEnv:
    """One reference CleanupEnv / HarvestEnv (+ optional SeparateContractSubgameStage) under injection.

    kind: 'cleanup' | 'harvest'.  contract: None (bare base env) or True (the contract the
    BASELINE configs pair with the env: CleanupContract / HarvestFeaturemodLocalContract).
    """

    def __init__(self, kind, num_agents, seed, env_id, contract=True, ascii_map=None,
                 null_prob=0.0, **env_kwargs):
        install()
        from utils.env_creator_functions import env_creator
        import contract.contract_list as cl
        self.kind = kind
        self.n = num_agents
        self.ctx = DrawContext(seed, env_id)
        self.episode = -1
        cfg = dict(num_agents=num_agents, env_params={}, image_obs=True)
        if ascii_map is not None:
            cfg["ascii_map"] = ascii_map
        cfg.update(env_kwargs)
        with active(self.ctx):
            self.ctx.begin(px.EPISODE_CONSTRUCT, 0)
            self.base = env_creator("CleanupNew" if kind == "cleanup" else "HarvestNew", cfg)
            if contract:
                c = cl.CleanupContract(num_agents) if kind == "cleanup" \
                    else cl.HarvestFeaturemodLocalContract(num_agents)
                self.env = env_creator("ContractWrapperSubgame", dict(
                    num_agents=num_agents, base_env=self.base, contract=c, convolutional=True,
                    null_prob=null_prob))
                orig = c.compute_transfer

                def capture(obs, acts, rews, params, infos=None):
                    self._base_rew = dict(rews)
                    tr = orig(obs, acts, rews, params, infos)
                    self._transfers = dict(tr)
                    return tr
                c.compute_transfer = capture
            else:
                self.env = self.base
        self.wrapped = bool(contract)
        self.keys = ["a%d" % i for i in range(num_agents)]

    # -- state snapshot ---------------------------------------------------------------------
    def _snapshot(self, obs):
        b = self.base
        out = {
            "map": np.frombuffer(b.world_map.tobytes(), dtype=np.uint8).reshape(b.world_map.shape).copy(),
            "pos": np.array([b.agents[k].pos for k in self.keys], dtype=np.int32),
            "ori": np.array([ORI_INT[b.agents[k].orientation] for k in self.keys], dtype=np.int32),
            "obs": np.stack([np.rint(obs[k]["image"] * 255.0).astype(np.uint8) for k in self.keys]),
            "t": int(b.timesteps),
        }
        if self.wrapped:
            out["theta"] = np.float64(self.env.params["a0"][0])
            out["contract_obs"] = np.stack([np.asarray(obs[k]["contract"], dtype=np.float64) for k in self.keys])
        return out

    def reset(self):
        self.episode += 1
        with active(self.ctx):
            self.ctx.begin(self.episode, 0)
            obs = self.env.reset()
        return self._snapshot(obs)

    def step(self, actions):
        acts = {k: int(a) for k, a in zip(self.keys, actions)}
        with active(self.ctx):
            self.ctx.begin(self.episode, self.base.timesteps + 1)
            obs, rew, done, info = self.env.step(acts)
        out = self._snapshot(obs)
        out["rew"] = np.array([rew[k] for k in self.keys], dtype=np.float64)
        out["done"] = bool(done["__all__"])
        out["eaten_apples"] = np.array([info[k]["eaten_apples"] for k in self.keys], dtype=np.int32)
        if self.kind == "cleanup":
            out["cleaned_squares"] = np.array([info[k]["cleaned_squares"] for k in self.keys], dtype=np.int32)
        else:
            out["eaten_close_apples"] = np.array([info[k]["eaten_close_apples"] for k in self.keys], dtype=np.int32)
        out["feature_obs"] = np.stack([np.asarray(info[k]["feature_obs"], dtype=np.float64) for k in self.keys])
        if self.wrapped:
            out["base_rew"] = np.array([self._base_rew[k] for k in self.keys], dtype=np.float64)
            out["transfers"] = np.array([self._transfers[k] for k in self.keys], dtype=np.float64)
        return out

    def metrics(self):
        return {k: float(np.asarray(v).reshape(-1)[0]) if np.ndim(v) else float(v)
                for k, v in self.base.metrics.items()}

    # -- state injection (for adversarial scenario tests) -------------------------------------
    def set_state(self, world_map=None, pos=None, ori=None):
        """Overwrite grid / agent state in place, keeping world_map_color consistent."""
        b = self.base
        inv = {v: k for k, v in ORI_INT.items()}
        # un-paint agents (map_env.py:238-240 does the same at step start)
        for a in b.agents.values():
            b.single_update_world_color_map(a.pos[0], a.pos[1], b.world_map[a.pos[0], a.pos[1]])
        if world_map is not None:
            wm = np.asarray(world_map, dtype=np.uint8)
            for r in range(wm.shape[0]):
                for c in range(wm.shape[1]):
                    b.single_update_map(r, c, bytes([wm[r, c]]))
        if pos is not None:
            for k, p in zip(self.keys, pos):
                b.agents[k].set_pos(np.array(p))
        if ori is not None:
            for k, o in zip(self.keys, ori):
                b.agents[k].set_orientation(inv[int(o)])
        # refresh the caches the next step's infos depend on (same calls custom_reset makes)
        b.compute_current_apples()
        if self.kind == "cleanup":
            b.compute_current_wastes()
        mwa = b.get_map_with_agents()
        for a in b.agents.values():
            a.full_map = mwa
            if b.world_map[a.pos[0], a.pos[1]] not in [b"F", b"C"]:
                b.single_update_world_color_map(a.pos[0], a.pos[1], a.get_char_id())


class ScriptedTrainer:
    """Stands in for the frozen RLlib PPOTrainer of SeparateContractNegotiateStage (two_stage_train.py:220-221,
    299-313): `compute_single_action` is called once per active agent per inner step, in agent order, and
    returns the next entry of a fixed action table [steps, n]."""

    def __init__(self, table):
        self.table = np.asarray(table)
        self.calls = 0

    def compute_single_action(self, obs, policy_id=None):
        t, i = divmod(self.calls, self.table.shape[1])
        self.calls += 1
        return int(self.table[t % self.table.shape[0], i])


class RefNegotiateEnv:
    """The reference's SeparateContractNegotiateStage (two_stage_train.py:190-358) under RNG injection, with the
    PPOTrainer construction (:220-221) bypassed: the object is allocated without running that __init__ and the
    fields it sets are assigned here (no reference source is edited)."""

    def __init__(self, kind, num_agents, seed, env_id, horizon, base_horizon, table, ascii_map=None):
        install()
        import gym
        from utils.env_creator_functions import env_creator
        import contract.contract_list as cl
        import environments.two_stage_train as tst
        self.kind, self.n = kind, num_agents
        self.ctx = DrawContext(seed, env_id)
        self.episode = -1
        cfg = dict(num_agents=num_agents, env_params={}, image_obs=True, horizon=base_horizon)
        if ascii_map is not None:
            cfg["ascii_map"] = ascii_map
        with active(self.ctx):
            self.ctx.begin(px.EPISODE_CONSTRUCT, 0)
            self.base = env_creator("CleanupNew" if kind == "cleanup" else "HarvestNew", cfg)
        c = cl.CleanupContract(num_agents) if kind == "cleanup" else cl.HarvestFeaturemodLocalContract(num_agents)
        env = object.__new__(tst.SeparateContractNegotiateStage)
        tst.SeparateContractEnv.__init__(env, self.base, c, num_agents, True)
        env.horizon = horizon
        env.convolutional = True
        env.shared = True
        env.frozen_trainer = ScriptedTrainer(table)
        env.action_space = gym.spaces.Box(low=np.concatenate((env.contract_low, np.array([0.0]))),
                                          high=np.concatenate((env.contract_high, np.array([1.0]))))
        env.metrics = {"contract": -1, "accepted": 0}
        self.env = env
        self.keys = ["a%d" % i for i in range(num_agents)]
        orig_step = self.base.step

        def stepped(acts):      # every inner base step gets its own draw coordinates (episode, t)
            self.ctx.begin(self.episode, self.base.timesteps + 1)
            return orig_step(acts)
        self.base.step = stepped

    def _pack(self, obs):
        return {"obs": np.stack([np.rint(obs[k]["image"] * 255.0).astype(np.uint8) for k in self.keys]),
                "contract_obs": np.stack([np.asarray(obs[k]["contract"], dtype=np.float64) for k in self.keys])}

    def reset(self):
        self.episode += 1
        self.env.frozen_trainer.calls = 0
        with active(self.ctx):
            self.ctx.begin(self.episode, 0)
            obs = self.env.reset()
        return self._pack(obs)

    def step(self, acts):
        """acts: float array [n, 2] = (proposal, accept probability) per agent."""
        d = {k: np.asarray(a, dtype=np.float64) for k, a in zip(self.keys, acts)}
        with active(self.ctx):
            self.ctx.begin(self.episode, 0)
            obs, rew, done, info = self.env.step(d)
        out = self._pack(obs)
        out["rew"] = np.array([rew[k] for k in self.keys], dtype=np.float64)
        out["done"] = bool(done["__all__"])
        out["accepted"] = int(self.env.metrics["accepted"])
        out["t"] = int(self.base.timesteps)
        return out

    def base_metrics(self):
        return {k: float(np.asarray(v).reshape(-1)[0]) if np.ndim(v) else float(v) for k, v in self.base.metrics.items()}


class ScriptedValueTrainer:
    """Stands in for the frozen PPOTrainer of NegotiationSolver.compute_vals (two_stage_train.py:693-703):
    `compute_single_action(obs)` then `get_policy(id).model.value_function().item()` once per agent, in agent
    order.  The value is oracle/scripted.py:scripted_value of the observation just passed in."""

    class _Val:
        def __init__(self, v):
            self.v = v

        def item(self):
            return self.v

    def __init__(self, num_agents, scale):
        self.n, self.scale, self.calls, self._obs = num_agents, scale, 0, None

    def compute_single_action(self, obs, policy_id=None):
        self._obs, self._agent = obs, self.calls % self.n
        self.calls += 1
        return 4

    def get_policy(self, policy_id):
        return self

    @property
    def model(self):
        return self

    def value_function(self):
        from .scripted import scripted_value
        return self._Val(scripted_value(self._obs, self._agent, self.n, self.scale))


class RefSolverEnv:
    """The reference's NegotiationSolver (two_stage_train.py:619-776) under RNG injection; the PPOTrainer
    construction (:652-653) is bypassed like in RefNegotiateEnv (no reference source is edited).

    NumPy drift: `contract_param_space.sample()` is a float32 array.  Under the NumPy the reference pins (< 1.24 via
    ray 2.2 / tf 2.11, requirements.yml) a float32 SCALAR combined with a Python int promotes to float64
    (`-params[k][0] * cleaned_squares`, contract_list.py:26; `rews[i] -= transfers[i]`, two_stage_train.py:85), so the
    transfers are float64 arithmetic on a float32-valued theta.  NumPy >= 2 (NEP 50, this container) would keep
    float32.  The harness restores the pinned behaviour by widening the stored parameter arrays to float64 after
    reset() — the values are unchanged."""

    def __init__(self, kind, num_agents, seed, env_id, num_samples, decision_rule, horizon=1000):
        install()
        import gym
        from utils.env_creator_functions import env_creator
        import contract.contract_list as cl
        import environments.two_stage_train as tst
        self.kind, self.n = kind, num_agents
        self.ctx = DrawContext(seed, env_id)
        self.episode = -1
        with active(self.ctx):
            self.ctx.begin(px.EPISODE_CONSTRUCT, 0)
            self.base = env_creator("CleanupNew" if kind == "cleanup" else "HarvestNew",
                                    dict(num_agents=num_agents, env_params={}, image_obs=True, horizon=horizon))
        c = cl.CleanupContract(num_agents) if kind == "cleanup" else cl.HarvestFeaturemodLocalContract(num_agents)
        env = object.__new__(tst.NegotiationSolver)
        tst.SeparateContractEnv.__init__(env, self.base, c, num_agents, True)
        env.horizon, env.convolutional, env.shared = horizon, True, True
        self.trainer = env.frozen_trainer = ScriptedValueTrainer(num_agents, float(c.contract_space.high[0]))
        env.contract_param_space = gym.spaces.Box(low=c.contract_space.low, high=c.contract_space.high)
        env.contract_low = c.contract_space.low
        env.num_samples, env.decision_rule, env.config = num_samples, decision_rule, {}
        self.env = env
        self.keys = ["a%d" % i for i in range(num_agents)]
        self.all_vals = self.all_params = None
        orig = env.compute_best_param

        def capture(all_vals, all_params, dec_rule=None):
            if dec_rule is None:                      # the outer call: the full candidate list
                self.all_vals = np.array([[v[k] for k in self.keys] for v in all_vals], dtype=np.float64)
                self.all_params = np.array([np.asarray(p, dtype=np.float64)[0] for p in all_params])
            return orig(all_vals, all_params, dec_rule)
        env.compute_best_param = capture

    def reset(self):
        self.episode += 1
        self.trainer.calls = 0
        with active(self.ctx):
            self.ctx.begin(self.episode, 0)
            obs = self.env.reset()
        self.env.params = {k: np.asarray(v, dtype=np.float64) for k, v in self.env.params.items()}
        return {"obs": np.stack([np.rint(obs[k]["image"] * 255.0).astype(np.uint8) for k in self.keys]),
                "contract_obs": np.stack([np.asarray(obs[k]["contract"], dtype=np.float64) for k in self.keys]),
                "params": self.all_params.copy(), "vals": self.all_vals.copy(),
                "theta": np.float64(np.asarray(self.env.contract_param)[0])}

    def step(self, actions):
        acts = {k: int(a) for k, a in zip(self.keys, actions)}
        with active(self.ctx):
            self.ctx.begin(self.episode, self.base.timesteps + 1)
            obs, rew, done, info = self.env.step(acts)
        return {"obs": np.stack([np.rint(obs[k]["image"] * 255.0).astype(np.uint8) for k in self.keys]),
                "contract_obs": np.stack([np.asarray(obs[k]["contract"], dtype=np.float64) for k in self.keys]),
                "rew": np.array([rew[k] for k in self.keys], dtype=np.float64), "done": bool(done["__all__"])}


class RefJointEnv:
    """The reference's JointEnv (two_stage_train.py:476-617) over CleanupEnv / HarvestEnv under RNG injection."""

    def __init__(self, kind, num_agents, seed, env_id, mode, horizon=1000):
        install()
        from utils.env_creator_functions import env_creator
        self.kind, self.n, self.mode = kind, num_agents, mode
        self.ctx = DrawContext(seed, env_id)
        self.episode = -1
        with active(self.ctx):
            self.ctx.begin(px.EPISODE_CONSTRUCT, 0)
            self.base = env_creator("CleanupNew" if kind == "cleanup" else "HarvestNew",
                                    dict(num_agents=num_agents, env_params={}, image_obs=True, horizon=horizon,
                                         disable_firing=False))
            self.env = env_creator("JointEnv", dict(base_env=self.base, num_agents=num_agents,
                                                    global_obs=mode == "global", concatenated_obs=mode == "concatenated"))

    @staticmethod
    def _img(obs):
        o = obs["a0"]
        return np.rint(o["image"] * 255.0).astype(np.uint8)

    def reset(self):
        self.episode += 1
        with active(self.ctx):
            self.ctx.begin(self.episode, 0)
            obs = self.env.reset()
        assert list(obs.keys()) == ["a0"]
        return self._img(obs)

    def step(self, actions):
        with active(self.ctx):
            self.ctx.begin(self.episode, self.base.timesteps + 1)
            obs, rew, done, info = self.env.step({"a0": np.asarray(actions)})
        assert sorted(done.keys()) == ["__all__", "a0"] and list(rew.keys()) == ["a0"]
        i = info["a0"]
        return {"obs": self._img(obs), "rew": np.float64(rew["a0"]), "done": bool(done["__all__"]),
                "eaten_apples": int(i["eaten_apples"]),
                "info1": int(i["cleaned_squares" if self.kind == "cleanup" else "eaten_close_apples"]),
                "feature_obs": np.asarray(i["feature_obs"], dtype=np.float64)}


class RefCarEnv:
    """The reference's SelfAcceleratingCarEnv (+ SeparateContractSubgameStage / SelfdriveContractDistprop) under RNG
    injection.  Done agents stop acting (what RLlib does once a done flag was returned); actions are passed as
    Python floats so that the arithmetic stays float64 under NumPy >= 2 scalar promotion (SURVEY.md §7.2-8)."""

    def __init__(self, num_agents, seed, env_id, contract=True, null_prob=0.0, **env_kwargs):
        """env_kwargs: low_bound, high_bound, start_vel, start_vel_ambulance (self_driving_car_accelerate.py:19)"""
        install()
        from utils.env_creator_functions import env_creator
        import contract.contract_list as cl
        self.n = num_agents
        self.ctx = DrawContext(seed, env_id)
        self.episode = -1
        self.keys = ["a%d" % i for i in range(num_agents)]
        self.base = env_creator("SelfDrive", dict(num_agents=num_agents, **env_kwargs))
        self.wrapped = bool(contract)
        if contract:
            c = cl.SelfdriveContractDistprop(num_agents)
            self.env = env_creator("ContractWrapperSubgame", dict(num_agents=num_agents, base_env=self.base, contract=c,
                                                                  convolutional=False, null_prob=null_prob))
            orig = c.compute_transfer

            def capture(obs, acts, rews, params, infos=None):
                self._base_rew = dict(rews)
                tr = orig(obs, acts, rews, params, infos)
                self._transfers = dict(tr)
                return tr
            c.compute_transfer = capture
        else:
            self.env = self.base
        self.t = 0

    def _obs(self, obs):
        D = 2 * (self.n + 1) + 3
        out = np.full((self.n, D + (2 if self.wrapped else 0)), np.nan)
        for i, k in enumerate(self.keys):
            if k in obs:
                out[i] = np.asarray(obs[k], dtype=np.float64)
        return out

    def reset(self):
        self.episode += 1
        self.t = 0
        with active(self.ctx):
            self.ctx.begin(self.episode, 0)
            obs = self.env.reset()
        out = {"obs": self._obs(obs)}
        if self.wrapped:
            out["theta"] = np.float64(self.env.params["a0"][0])
        return out

    def step(self, actions):
        acting = [k for k in self.keys if not self.base.agent_dones[k]]
        acts = {k: [float(np.float32(actions[int(k[1:])]))] for k in acting}
        self.t += 1
        with active(self.ctx):
            self.ctx.begin(self.episode, self.t)
            obs, rew, done, info = self.env.step(acts)
        n = self.n
        out = {"obs": self._obs(obs), "active": np.array([k in acts for k in self.keys], dtype=np.uint8),
               "rew": np.array([rew.get(k, 0.0) for k in self.keys], dtype=np.float64),
               "done": np.array([done[k] for k in self.keys] + [done["__all__"]], dtype=np.uint8),
               "just_passed": np.array([bool(info[k]["just_passed"]) if k in info else False for k in self.keys], dtype=np.uint8),
               "ambulance_rank": np.float64(info[acting[0]]["ambulance_rank"]),
               "ambulance_dist_to_front": np.float64(info[acting[0]]["ambulance_dist_to_front"]),
               "pos": np.array([self.base.agent_positions[k] for k in self.keys], dtype=np.float64),
               "vel": np.array([self.base.agent_vels[k] for k in self.keys], dtype=np.float64),
               "metric_transfers": np.float64(self.base.metrics["transfers"])}
        if self.wrapped:
            out["base_rew"] = np.array([self._base_rew.get(k, 0.0) for k in self.keys], dtype=np.float64)
            tr = np.zeros(n)
            for i, k in enumerate(self.keys):
                v = self._transfers.get(k, 0)
                tr[i] = v[0] if isinstance(v, tuple) else v
            out["transfers"] = tr
        return out


class RefFeatEnv:
    """The reference's CleanupFeatures / HarvestFeatures (+ SeparateContractSubgameStage) under RNG injection."""

    def __init__(self, kind, num_agents, seed, env_id, contract=True, horizon=1000, null_prob=0.0):
        install()
        from utils.env_creator_functions import env_creator
        import contract.contract_list as cl
        self.kind, self.n = kind, num_agents
        self.ctx = DrawContext(seed, env_id)
        self.episode = -1
        self.keys = ["a%d" % i for i in range(num_agents)]
        with active(self.ctx):
            self.ctx.begin(px.EPISODE_CONSTRUCT, 0)
            self.base = env_creator("Cleanup" if kind == "cleanup" else "Harvest", dict(num_agents=num_agents, horizon=horizon))
        self.wrapped = bool(contract)
        if contract:
            c = cl.CleanupContract(num_agents) if kind == "cleanup" else cl.HarvestFeaturemodLocalContract(num_agents)
            self.env = env_creator("ContractWrapperSubgame", dict(num_agents=num_agents, base_env=self.base, contract=c,
                                                                  convolutional=False, null_prob=null_prob))
            orig = c.compute_transfer

            def capture(obs, acts, rews, params, infos=None):
                self._base_rew = dict(rews)
                tr = orig(obs, acts, rews, params, infos)
                self._transfers = dict(tr)
                return tr
            c.compute_transfer = capture
        else:
            self.env = self.base

    def _cells(self):
        b = self.base
        cells = np.zeros((len(b.map), len(b.map[0])), dtype=np.uint8)
        for r, c in b.current_apple_points:
            cells[r, c] = 1
        for r, c in getattr(b, "current_waste_points", []):
            cells[r, c] = 2
        return cells

    def _snap(self, obs):
        b = self.base
        out = {"obs": np.stack([np.asarray(obs[k], dtype=np.float64) for k in self.keys]),
               "pos": np.array([b.agent_pos[k] for k in self.keys], dtype=np.int32),
               "ori": np.array([int(b.agent_orientation[k]) for k in self.keys], dtype=np.int32),
               "cells": self._cells()}
        return out

    def reset(self):
        self.episode += 1
        with active(self.ctx):
            self.ctx.begin(self.episode, 0)
            obs = self.env.reset()
        out = self._snap(obs)
        if self.wrapped:
            out["theta"] = np.float64(self.env.params["a0"][0])
        return out

    def step(self, actions):
        acts = {k: int(a) for k, a in zip(self.keys, actions)}
        with active(self.ctx):
            self.ctx.begin(self.episode, self.base.timesteps + 1)
            obs, rew, done, info = self.env.step(acts)
        out = self._snap(obs)
        out["rew"] = np.array([rew[k] for k in self.keys], dtype=np.float64)
        out["done"] = bool(done["__all__"])
        if self.kind == "cleanup":
            out["info0"] = np.array([info[k]["cleaned_squares"] for k in self.keys], dtype=np.int32)
            out["info1"] = np.zeros(self.n, dtype=np.int32)
        else:
            out["info0"] = np.array([info[k]["eaten_apples"] for k in self.keys], dtype=np.int32)
            out["info1"] = np.array([info[k]["eaten_close_apples"] for k in self.keys], dtype=np.int32)
        if self.wrapped:
            out["base_rew"] = np.array([self._base_rew[k] for k in self.keys], dtype=np.float64)
            out["transfers"] = np.array([self._transfers[k] for k in self.keys], dtype=np.float64)
        return out

    def metrics(self):
        return {k: float(np.asarray(v).reshape(-1)[0]) if np.ndim(v) else float(v) for k, v in self.base.metrics.items()}

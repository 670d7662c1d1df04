"""Generate the golden vectors in tests/golden/ by running the UNMODIFIED reference.

TEST INFRASTRUCTURE (oracle/): needs a checkout of the original project.  Run as
    SSD_REFERENCE_ROOT=<checkout> python -m oracle.make_golden
Each fixture is the reference's own output (oracle/ref_harness.py: reference code + RNG
injection) for a seeded action sequence: per-step grid, agent state, uint8 observations,
rewards before/after contract transfers, transfers, infos and feature_obs, plus episode
metrics.  Both the C oracle (CPU tests) and the CUDA path (GPU tests) must reproduce them
bit-exactly.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")

CRAMPED_CLEANUP = ["@@@@@@", "@PPPP@", "@PPPP@", "@HBBR@", "@PPPP@", "@@@@@@"]
CRAMPED_HARVEST = ["@@@@@@", "@PPPP@", "@PAAP@", "@PAAP@", "@PPPP@", "@@@@@@"]
OPEN_CLEANUP = [" PBH", "PRB ", "HPPB", "BPRP", "PPHP"]          # no walls: exercises map-edge bounds

# name -> (kind, n, seed, env_id, map (None = stock), horizon, episodes, steps/episode, action ids, action probs)
SCENARIOS = {
    "cleanup_n2": ("cleanup", 2, 73907, 0, None, 1000, 1, 300, 9, None),
    "cleanup_n8": ("cleanup", 8, 73907, 12345, None, 1000, 1, 250, 9, None),
    "cleanup_n5_short_horizon": ("cleanup", 5, 11, 3, None, 40, 3, 40, 8, None),
    "harvest_n4": ("harvest", 4, 73907, 77, None, 1000, 1, 250, 8, None),
    "harvest_n8_short_horizon": ("harvest", 8, 5, 4000000000, None, 30, 3, 30, 7, None),
    "cleanup_cramped_n8": ("cleanup", 8, 42, 9, CRAMPED_CLEANUP, 1000, 1, 400, 9,
                           [.2, .2, .2, .2, .04, .04, .04, .06, .02]),
    "harvest_cramped_n8": ("harvest", 8, 43, 10, CRAMPED_HARVEST, 1000, 1, 400, 8,
                           [.22, .22, .22, .22, .03, .03, .03, .03]),
    "cleanup_open_n6": ("cleanup", 6, 44, 11, OPEN_CLEANUP, 1000, 1, 300, 9, None),
    "cleanup_n8_nocontract": ("cleanup", 8, 3, 5, None, 1000, 1, 120, 9, None),
    # the deep spawning regime of the stock map: a cleaning-heavy policy takes #waste from 56 down to ~40 (below the
    # apple / waste spawn threshold of 47), so apples spawn at several different probabilities, get eaten, and waste
    # respawns through the shuffled first-success scan for hundreds of steps (cleanup_new.py:322-368)
    "cleanup_n8_deep": ("cleanup", 8, 71, 424242, None, 1000, 1, 700, 9,
                        [.14, .14, .14, .14, .02, .04, .04, .32, .02]),
    # use_collective_reward / inequity_averse_reward (map_env.py:289-301); short horizons so that the episode
    # metrics (equality / sustainability over the shaped rewards) are produced
    "cleanup_n4_collective": ("cleanup", 4, 51, 21, None, 60, 2, 60, 9, None),
    "harvest_n5_inequity": ("harvest", 5, 52, 22, None, 50, 2, 50, 8, None),
    "cleanup_cramped_n8_inequity": ("cleanup", 8, 53, 23, CRAMPED_CLEANUP, 80, 2, 80, 9,
                                    [.16, .16, .16, .16, .04, .04, .04, .12, .12]),
    "harvest_cramped_n6_collective_inequity": ("harvest", 6, 54, 24, CRAMPED_HARVEST, 40, 2, 40, 8, None),
}

# extra MapEnv kwargs of a scenario (cleanup_new.py:60-74)
SCENARIO_KWARGS = {
    "cleanup_n4_collective": dict(use_collective_reward=True),
    "harvest_n5_inequity": dict(inequity_averse_reward=True, alpha=5.0, beta=0.05),
    "cleanup_cramped_n8_inequity": dict(inequity_averse_reward=True, alpha=0.7, beta=-0.3),
    "harvest_cramped_n6_collective_inequity": dict(use_collective_reward=True, inequity_averse_reward=True,
                                                   alpha=1.5, beta=0.25),
}


def run_scenario(name):
    from .ref_harness import RefGridEnv
    kind, n, seed, env_id, amap, horizon, episodes, steps, act_hi, act_p = SCENARIOS[name]
    contract = not name.endswith("nocontract")
    kw = SCENARIO_KWARGS.get(name, {})
    ref = RefGridEnv(kind, n, seed, env_id, contract=contract, ascii_map=amap, horizon=horizon, **kw)
    b = ref.base
    ascii_map = amap if amap is not None else ["".join(ch.decode() for ch in row) for row in b.base_map]
    rng = np.random.RandomState(abs(hash(name)) % (2 ** 31) if False else sum(map(ord, name)))
    rec = {k: [] for k in ("actions", "map", "pos", "ori", "obs", "rew", "done", "eaten_apples", "info1",
                           "feature_obs", "base_rew", "transfers")}
    rst = {k: [] for k in ("map", "pos", "ori", "obs", "theta")}
    metrics = []
    for ep in range(episodes):
        s = ref.reset()
        for k in ("map", "pos", "ori", "obs"):
            rst[k].append(s[k])
        rst["theta"].append(s.get("theta", np.float64(0.0)))
        for k in rec:
            rec[k].append([])
        for t in range(steps):
            a = rng.choice(act_hi, size=n, p=act_p).astype(np.int32)
            o = ref.step(a)
            rec["actions"][-1].append(a)
            for k in ("map", "pos", "ori", "obs", "rew", "eaten_apples", "feature_obs"):
                rec[k][-1].append(o[k])
            rec["done"][-1].append(o["done"])
            rec["info1"][-1].append(o["cleaned_squares"] if kind == "cleanup" else o["eaten_close_apples"])
            rec["base_rew"][-1].append(o.get("base_rew", o["rew"]))
            rec["transfers"][-1].append(o.get("transfers", np.zeros(n)))
        m = ref.metrics()
        metrics.append(m)
    out = {"kind": kind, "n": n, "seed": seed, "env_id": env_id, "horizon": horizon, "contract": contract,
           "ascii_map": np.array(ascii_map), "metric_keys": np.array(sorted(metrics[0].keys())),
           "metrics": np.array([[m[k] for k in sorted(m.keys())] for m in metrics], dtype=np.float64),
           "reward_mode": (1 if kw.get("use_collective_reward") else 0) | (2 if kw.get("inequity_averse_reward") else 0),
           "alpha": np.float64(kw.get("alpha", 0.0)), "beta": np.float64(kw.get("beta", 0.0))}
    for k, v in rec.items():
        out[k] = np.array(v)
    for k, v in rst.items():
        out["reset_" + k] = np.array(v)
    return out


# name -> (kind, n, seed, env_id, negotiate horizon, base env horizon, episodes, action ids)
NEGOTIATE_SCENARIOS = {
    "negotiate_cleanup_n2": ("cleanup", 2, 21, 3, 30, 1000, 4, 9),
    "negotiate_cleanup_n5": ("cleanup", 5, 22, 40, 1000, 25, 4, 9),     # ends on the base env's own horizon
    "negotiate_harvest_n4": ("harvest", 4, 23, 7, 20, 1000, 4, 8),
    "negotiate_cleanup_n8": ("cleanup", 8, 27, 91, 60, 1000, 5, 9),      # BASELINE configs[2]: n = 8, 2 sampled acceptors
}


def run_negotiate(name):
    """SeparateContractNegotiateStage episodes: reset -> proposal step -> agreement step + scripted rollout."""
    from .ref_harness import RefNegotiateEnv
    kind, n, seed, env_id, horizon, base_horizon, episodes, act_hi = NEGOTIATE_SCENARIOS[name]
    rng = np.random.RandomState(sum(map(ord, name)))
    steps = min(horizon, base_horizon)
    table = rng.randint(0, act_hi, size=(steps, n))
    ref = RefNegotiateEnv(kind, n, seed, env_id, horizon, base_horizon, table)
    high = 0.2 if kind == "cleanup" else 10.0
    rec = {k: [] for k in ("reset_obs", "reset_contract_obs", "acts", "obs2", "contract_obs2", "rew2", "obs3",
                           "contract_obs3", "rew3", "accepted", "t_end", "base_metrics")}
    keys = None
    for ep in range(episodes):
        r0 = ref.reset()
        acts = np.stack([rng.uniform(0, high, size=n), rng.uniform(0.55, 1.0, size=n)], axis=1)
        if ep == 1:
            acts[1:, 1] = 0.0          # a certain rejection
        s2 = ref.step(acts)
        s3 = ref.step(acts)
        assert not s2["done"] and s3["done"]
        m = ref.base_metrics()
        keys = sorted(m.keys())
        for k, v in (("reset_obs", r0["obs"]), ("reset_contract_obs", r0["contract_obs"]), ("acts", acts),
                     ("obs2", s2["obs"]), ("contract_obs2", s2["contract_obs"]), ("rew2", s2["rew"]),
                     ("obs3", s3["obs"]), ("contract_obs3", s3["contract_obs"]), ("rew3", s3["rew"]),
                     ("accepted", s3["accepted"]), ("t_end", s3["t"]), ("base_metrics", [m[k] for k in keys])):
            rec[k].append(v)
    out = {"kind": kind, "n": n, "seed": seed, "env_id": env_id, "horizon": horizon, "base_horizon": base_horizon,
           "table": table, "metric_keys": np.array(keys)}
    out.update({k: np.array(v) for k, v in rec.items()})
    return out


# image_obs=False + non-convolutional wrapper: flat feature-vector observations (cleanup_new.py:193-202,243-254;
# two_stage_train.py:113-121,182-187).  name -> (kind, n, seed, env_id, horizon, episodes, steps, action ids)
FLATOBS_SCENARIOS = {
    "flatobs_cleanup_n3": ("cleanup", 3, 31, 2, 25, 2, 25, 9),
    "flatobs_harvest_n3": ("harvest", 3, 32, 6, 25, 2, 25, 8),
}


def run_flatobs(name):
    from . import ref_harness as rh
    from . import philox as px
    kind, n, seed, env_id, horizon, episodes, steps, act_hi = FLATOBS_SCENARIOS[name]
    rh.install()
    from utils.env_creator_functions import env_creator
    import contract.contract_list as cl
    ctx = rh.DrawContext(seed, env_id)
    with rh.active(ctx):
        ctx.begin(px.EPISODE_CONSTRUCT, 0)
        base = env_creator("CleanupNew" if kind == "cleanup" else "HarvestNew",
                           dict(num_agents=n, env_params={}, image_obs=False, horizon=horizon))
        c = cl.CleanupContract(n) if kind == "cleanup" else cl.HarvestFeaturemodLocalContract(n)
        env = env_creator("ContractWrapperSubgame", dict(num_agents=n, base_env=base, contract=c, convolutional=False))
    keys = ["a%d" % i for i in range(n)]
    rng = np.random.RandomState(sum(map(ord, name)))
    out = {"reset_obs": [], "actions": [], "obs": [], "rew": []}
    for ep in range(episodes):
        with rh.active(ctx):
            ctx.begin(ep, 0)
            o = env.reset()
        out["reset_obs"].append(np.stack([np.asarray(o[k], dtype=np.float64) for k in keys]))
        for k in ("actions", "obs", "rew"):
            out[k].append([])
        for t in range(steps):
            a = rng.randint(0, act_hi, size=n)
            with rh.active(ctx):
                ctx.begin(ep, base.timesteps + 1)
                o, r, d, info = env.step({k: int(x) for k, x in zip(keys, a)})
            out["actions"][-1].append(a)
            out["obs"][-1].append(np.stack([np.asarray(o[k], dtype=np.float64) for k in keys]))
            out["rew"][-1].append(np.array([r[k] for k in keys], dtype=np.float64))
    res = {"kind": kind, "n": n, "seed": seed, "env_id": env_id, "horizon": horizon}
    res.update({k: np.array(v) for k, v in out.items()})
    res["space_low"] = np.asarray(env.observation_space.low, dtype=np.float64)
    res["space_high"] = np.asarray(env.observation_space.high, dtype=np.float64)
    return res


# name -> (n, seed, env_id, contract, episodes, max steps/episode, action scale)
SELFDRIVE_SCENARIOS = {
    "selfdrive_n8": (8, 51, 0, True, 3, 400, 0.12),
    "selfdrive_n2": (2, 52, 9, True, 3, 400, 0.12),
    "selfdrive_n4_nocontract": (4, 53, 1000, False, 2, 400, 0.12),
    "selfdrive_n8_fast": (8, 54, 77, True, 3, 400, 0.3),          # accelerations mostly clipped: more overtaking attempts
    "selfdrive_n1": (1, 55, 2, False, 2, 100, 0.12),
}


def run_selfdrive(name):
    """Episodes run until every car is done (or max steps); actions are seeded float32 accelerations, biased
    forward so that episodes finish.  Steps after the end are padded with NaN / zeros and `length` says where."""
    from .ref_harness import RefCarEnv
    n, seed, env_id, contract, episodes, max_steps, scale = SELFDRIVE_SCENARIOS[name]
    ref = RefCarEnv(n, seed, env_id, contract=contract)
    rng = np.random.RandomState(sum(map(ord, name)))
    keys = ("obs", "active", "rew", "done", "just_passed", "ambulance_rank", "ambulance_dist_to_front", "pos", "vel",
            "metric_transfers", "base_rew", "transfers")
    rec = {k: [] for k in keys}
    out = {"reset_obs": [], "reset_theta": [], "actions": [], "length": []}
    for ep in range(episodes):
        r0 = ref.reset()
        out["reset_obs"].append(r0["obs"])
        out["reset_theta"].append(r0.get("theta", np.float64(0.0)))
        acts = (rng.uniform(-0.6, 1.0, size=(max_steps, n)) * scale).astype(np.float32)
        out["actions"].append(acts)
        ep_rec = {k: [] for k in keys}
        steps = 0
        for t in range(max_steps):
            o = ref.step(acts[t])
            steps += 1
            for k in keys:
                ep_rec[k].append(o.get(k, np.zeros(n)))
            if o["done"][-1]:
                break
        out["length"].append(steps)
        for k in keys:
            a = np.array(ep_rec[k], dtype=np.float64)
            pad = np.full((max_steps - steps,) + a.shape[1:], np.nan)
            rec[k].append(np.concatenate([a, pad], axis=0))
    res = {"n": n, "seed": seed, "env_id": env_id, "contract": contract}
    res.update({k: np.array(v) for k, v in out.items()})
    res.update({k: np.array(v) for k, v in rec.items()})
    return res


# name -> (kind, n, seed, env_id, contract, horizon, episodes, steps/episode, action ids, action probs)
FEATURES_SCENARIOS = {
    "features_cleanup_n8": ("cleanup", 8, 61, 5, True, 1000, 1, 400, 8, [.12, .12, .12, .12, .06, .06, .06, .34]),
    "features_cleanup_n2_short": ("cleanup", 2, 62, 6, True, 60, 3, 60, 9, [.1, .1, .1, .1, .05, .05, .05, .4, .05]),
    "features_harvest_n8": ("harvest", 8, 63, 7, True, 1000, 1, 400, 7, None),
    "features_harvest_n4_short": ("harvest", 4, 64, 8, True, 50, 3, 50, 8, None),
    "features_cleanup_n3_nocontract": ("cleanup", 3, 65, 9, False, 1000, 1, 200, 8, [.12, .12, .12, .12, .06, .06, .06, .34]),
}


def run_features(name):
    from .ref_harness import RefFeatEnv
    kind, n, seed, env_id, contract, horizon, episodes, steps, act_hi, act_p = FEATURES_SCENARIOS[name]
    ref = RefFeatEnv(kind, n, seed, env_id, contract=contract, horizon=horizon)
    rng = np.random.RandomState(sum(map(ord, name)))
    keys = ("actions", "obs", "pos", "ori", "cells", "rew", "done", "info0", "info1", "base_rew", "transfers")
    rec = {k: [] for k in keys}
    rst = {k: [] for k in ("obs", "pos", "ori", "cells", "theta")}
    metrics = []
    for ep in range(episodes):
        s0 = ref.reset()
        for k in ("obs", "pos", "ori", "cells"):
            rst[k].append(s0[k])
        rst["theta"].append(s0.get("theta", np.float64(0.0)))
        for k in keys:
            rec[k].append([])
        for t in range(steps):
            a = rng.choice(act_hi, size=n, p=act_p).astype(np.int32)
            o = ref.step(a)
            rec["actions"][-1].append(a)
            for k in keys[1:]:
                rec[k][-1].append(o.get(k, np.zeros(n)) if k not in ("base_rew",) else o.get(k, o["rew"]))
        metrics.append(ref.metrics())
    out = {"kind": kind, "n": n, "seed": seed, "env_id": env_id, "horizon": horizon, "contract": contract,
           "metric_keys": np.array(sorted(metrics[0].keys())),
           "metrics": np.array([[m[k] for k in sorted(m.keys())] for m in metrics], dtype=np.float64),
           "reward_mode": (1 if kw.get("use_collective_reward") else 0) | (2 if kw.get("inequity_averse_reward") else 0),
           "alpha": np.float64(kw.get("alpha", 0.0)), "beta": np.float64(kw.get("beta", 0.0))}
    out.update({k: np.array(v) for k, v in rec.items()})
    out.update({"reset_" + k: np.array(v) for k, v in rst.items()})
    return out


# NegotiationSolver (two_stage_train.py:619-776) with the scripted value function of oracle/scripted.py.
# name -> (kind, n, seed, env_id, contract_samples, decision_rule, episodes, steps per episode, action ids)
SOLVER_SCENARIOS = {
    "solver_cleanup_n4_majority": ("cleanup", 4, 61, 31, 12, "majority", 4, 12, 9),
    "solver_harvest_n3_max": ("harvest", 3, 62, 32, 9, "max", 3, 12, 8),
    "solver_cleanup_n2_majority": ("cleanup", 2, 63, 33, 20, "majority", 4, 6, 9),
    "solver_harvest_n8_majority": ("harvest", 8, 64, 34, 50, "majority", 3, 6, 8),
}


def run_solver(name):
    from .ref_harness import RefSolverEnv
    kind, n, seed, env_id, S, rule, episodes, steps, act_hi = SOLVER_SCENARIOS[name]
    ref = RefSolverEnv(kind, n, seed, env_id, S, rule)
    rng = np.random.RandomState(sum(map(ord, name)))
    rec = {k: [] for k in ("reset_obs", "reset_contract_obs", "params", "vals", "theta", "actions", "obs", "contract_obs", "rew")}
    for ep in range(episodes):
        r = ref.reset()
        for k, v in (("reset_obs", r["obs"]), ("reset_contract_obs", r["contract_obs"]), ("params", r["params"]),
                     ("vals", r["vals"]), ("theta", r["theta"])):
            rec[k].append(v)
        for k in ("actions", "obs", "contract_obs", "rew"):
            rec[k].append([])
        for t in range(steps):
            a = rng.randint(0, act_hi, size=n)
            o = ref.step(a)
            rec["actions"][-1].append(a)
            for k in ("obs", "contract_obs", "rew"):
                rec[k][-1].append(o[k])
    out = {"kind": kind, "n": n, "seed": seed, "env_id": env_id, "num_samples": S, "rule": rule}
    out.update({k: np.array(v) for k, v in rec.items()})
    return out


# JointEnv (two_stage_train.py:476-617).  name -> (kind, n, seed, env_id, mode, horizon, episodes, steps, action ids)
JOINT_SCENARIOS = {
    "joint_cleanup_n2_concatenated": ("cleanup", 2, 71, 41, "concatenated", 40, 2, 40, 9),   # cleanup-joint-2agents.json
    "joint_cleanup_n3_global": ("cleanup", 3, 72, 42, "global", 30, 2, 30, 9),
    "joint_harvest_n4_global": ("harvest", 4, 73, 43, "global", 30, 2, 30, 8),
    "joint_harvest_n5_concatenated": ("harvest", 5, 74, 44, "concatenated", 25, 2, 25, 8),
}


def run_joint(name):
    from .ref_harness import RefJointEnv
    kind, n, seed, env_id, mode, horizon, episodes, steps, act_hi = JOINT_SCENARIOS[name]
    ref = RefJointEnv(kind, n, seed, env_id, mode, horizon=horizon)
    rng = np.random.RandomState(sum(map(ord, name)))
    keys = ("obs", "rew", "done", "eaten_apples", "info1", "feature_obs")
    rec = {k: [] for k in keys + ("actions", "reset_obs")}
    for ep in range(episodes):
        rec["reset_obs"].append(ref.reset())
        for k in keys + ("actions",):
            rec[k].append([])
        for t in range(steps):
            a = rng.randint(0, act_hi, size=n)
            o = ref.step(a)
            rec["actions"][-1].append(a)
            for k in keys:
                rec[k][-1].append(o[k])
    out = {"kind": kind, "n": n, "seed": seed, "env_id": env_id, "mode": mode, "horizon": horizon}
    out.update({k: np.array(v) for k, v in rec.items()})
    return out


# render(mode='rgb_array') = full_map_to_colors (map_env.py:389-392,460-475): agents + the beams of the last step.
# name -> (kind, n, seed, env_id, map, horizon, episodes, steps, action probabilities)
RENDER_SCENARIOS = {
    "render_cleanup_n6": ("cleanup", 6, 81, 51, None, 30, 2, 30, [.1, .1, .1, .1, .05, .1, .1, .2, .15]),
    "render_harvest_n5": ("harvest", 5, 82, 52, None, 1000, 1, 40, [.12, .12, .12, .12, .06, .1, .1, .26]),
    "render_cleanup_cramped_n8": ("cleanup", 8, 83, 53, CRAMPED_CLEANUP, 1000, 1, 40, [.1, .1, .1, .1, .05, .1, .1, .2, .15]),
    "render_cleanup_open_n6": ("cleanup", 6, 84, 54, OPEN_CLEANUP, 1000, 1, 40, [.1, .1, .1, .1, .05, .1, .1, .2, .15]),
}


def run_render(name):
    from .ref_harness import RefGridEnv
    kind, n, seed, env_id, amap, horizon, episodes, steps, act_p = RENDER_SCENARIOS[name]
    ref = RefGridEnv(kind, n, seed, env_id, contract=False, ascii_map=amap, horizon=horizon, disable_firing=False)
    ascii_map = amap if amap is not None else ["".join(ch.decode() for ch in row) for row in ref.base.base_map]
    rng = np.random.RandomState(sum(map(ord, name)))
    frames, resets, actions = [], [], []
    for ep in range(episodes):
        ref.reset()
        resets.append(np.asarray(ref.base.render(mode="rgb_array"), dtype=np.uint8))
        frames.append([])
        actions.append([])
        for t in range(steps):
            a = rng.choice(len(act_p), size=n, p=act_p).astype(np.int32)
            ref.step(a)
            actions[-1].append(a)
            frames[-1].append(np.asarray(ref.base.render(mode="rgb_array"), dtype=np.uint8))
    return {"kind": kind, "n": n, "seed": seed, "env_id": env_id, "horizon": horizon, "ascii_map": np.array(ascii_map),
            "actions": np.array(actions), "obs": np.array(frames), "reset_obs": np.array(resets)}


def main(names=None):
    os.makedirs(OUT, exist_ok=True)
    for name in (names or list(SCENARIOS) + list(NEGOTIATE_SCENARIOS) + list(FLATOBS_SCENARIOS) + list(SELFDRIVE_SCENARIOS)
                 + list(FEATURES_SCENARIOS) + list(SOLVER_SCENARIOS) + list(JOINT_SCENARIOS) + list(RENDER_SCENARIOS)):
        if name in SOLVER_SCENARIOS or name in JOINT_SCENARIOS or name in RENDER_SCENARIOS:
            data = run_solver(name) if name in SOLVER_SCENARIOS else (run_joint(name) if name in JOINT_SCENARIOS else run_render(name))
            path = os.path.join(OUT, name + ".npz")
            np.savez_compressed(path, **data)
            print("%-32s %7.1f KiB  obs=%s %s" % (name, os.path.getsize(path) / 1024, data["obs"].shape,
                                                  ("theta=%s" % data["theta"]) if "theta" in data else ""))
            continue
        if name in FEATURES_SCENARIOS:
            data = run_features(name)
            path = os.path.join(OUT, name + ".npz")
            np.savez_compressed(path, **data)
            print("%-32s %7.1f KiB  steps=%s rewards=%.0f transfers=%.3f" % (name, os.path.getsize(path) / 1024, data["actions"].shape,
                                                                             data["base_rew"].sum(), np.abs(data["transfers"]).sum()))
            continue
        if name in SELFDRIVE_SCENARIOS:
            data = run_selfdrive(name)
            path = os.path.join(OUT, name + ".npz")
            np.savez_compressed(path, **data)
            print("%-28s %7.1f KiB  lengths=%s transfers=%s" % (name, os.path.getsize(path) / 1024, data["length"],
                                                              np.nanmax(np.abs(data["transfers"]), axis=(1, 2))))
            continue
        if name in FLATOBS_SCENARIOS:
            data = run_flatobs(name)
            path = os.path.join(OUT, name + ".npz")
            np.savez_compressed(path, **data)
            print("%-28s %7.1f KiB  obs=%s" % (name, os.path.getsize(path) / 1024, data["obs"].shape))
            continue
        if name in NEGOTIATE_SCENARIOS:
            data = run_negotiate(name)
            path = os.path.join(OUT, name + ".npz")
            np.savez_compressed(path, **data)
            print("%-28s %7.1f KiB  accepted=%s t_end=%s" % (name, os.path.getsize(path) / 1024, data["accepted"], data["t_end"]))
            continue
        data = run_scenario(name)
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **data)
        print("%-28s %7.1f KiB  steps=%s" % (name, os.path.getsize(path) / 1024, data["actions"].shape))


if __name__ == "__main__":
    main(sys.argv[1:] or None)

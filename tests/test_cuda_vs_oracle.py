"""GPU: CUDA path vs the C oracle on seeded random rollouts (many envs, every output, bit-exact)."""
import os

import numpy as np
import pytest

import golden_util as gu

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("logic_variant")]

CRAMPED_CLEANUP = ["@@@@@@", "@PPPP@", "@PPPP@", "@HBBR@", "@PPPP@", "@@@@@@"]
CRAMPED_HARVEST = ["@@@@@@", "@PPPP@", "@PAAP@", "@PAAP@", "@PPPP@", "@@@@@@"]

CASES = [
    # kind, n, map, E, steps, horizon, n_actions, seed, first_env_id
    ("cleanup", 8, None, 192, 260, 100, 9, 73907, 0),
    ("cleanup", 2, None, 67, 150, 1000, 8, 1, 4294967000),
    ("cleanup", 3, None, 33, 120, 50, 9, 2, 17),
    ("harvest", 4, None, 160, 220, 90, 8, 73907, 5),
    ("harvest", 8, None, 64, 150, 1000, 8, 3, 0),
    ("cleanup", 8, CRAMPED_CLEANUP, 128, 300, 1000, 9, 4, 0),
    ("harvest", 8, CRAMPED_HARVEST, 128, 300, 1000, 5, 5, 0),
    ("harvest", 1, None, 8, 60, 1000, 8, 6, 0),
    # whole episodes at the benchmark's horizon: the late-episode regime (spawning active, apples depleted: > 128 spawn
    # draws per step in harvest) and the re-reset at t = 1000
    ("cleanup", 8, None, 40, 1100, 1000, 8, 11, 0),
    ("harvest", 8, None, 40, 1100, 1000, 7, 12, 0),
    # reward shaping (map_env.py:289-301): use_collective_reward / inequity_averse_reward
    ("cleanup", 8, None, 96, 160, 70, 9, 7, 0, dict(inequity_averse_reward=True, alpha=5.0, beta=0.05)),
    ("harvest", 4, None, 96, 160, 70, 8, 8, 0, dict(use_collective_reward=True)),
    ("cleanup", 8, CRAMPED_CLEANUP, 64, 200, 1000, 9, 9, 0, dict(use_collective_reward=True, inequity_averse_reward=True, alpha=0.3, beta=-1.1)),
    ("harvest", 8, CRAMPED_HARVEST, 64, 200, 90, 8, 10, 0, dict(inequity_averse_reward=True, alpha=-0.7, beta=0.9)),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s-n%d-%s-E%d%s" % (c[0], c[1], "stock" if c[2] is None else "cramped", c[3],
                                                                           "-shaped" if len(c) > 9 else ""))
def test_rollout_matches_oracle(oracle_lib, case):
    import torch
    from contracts_b200.batched import BatchedGridEnv
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    kind, n, amap, E, steps, horizon, nact, seed, first = case[:9]
    shaping = case[9] if len(case) > 9 else {}
    amap = amap or (CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP)
    contract = None if n < 2 else ("CleanupContract" if kind == "cleanup" else "HarvestFeaturemodLocalContract")
    orc = oracle_lib.GridOracle(kind, E, n, amap, horizon=horizon, contract=contract, seed=seed, first_env_id=first, **shaping)
    env = BatchedGridEnv(kind + "_new", E, n, amap, horizon=horizon, contract=contract, seed=seed, first_env_id=first,
                         **shaping)
    rng = np.random.RandomState(seed)

    def check_state(ctx):
        so, sc = orc.get_state(), env.get_state()
        for k in ("map", "pos", "ori", "t"):
            gu.assert_same(k, sc[k].cpu().numpy(), so[k], ctx)
        gu.assert_same("theta", sc["theta"].cpu().numpy(), so["theta"], ctx)

    gu.assert_same("reset obs", env.reset().cpu().numpy(), orc.reset(), "reset")
    check_state("reset")
    for t in range(steps):
        a = rng.randint(0, nact, size=(E, n))
        wf = t % 7 == 0
        o = orc.step(a, want_features=wf)
        obs, rew, done, info = env.step(torch.as_tensor(a.astype(np.uint8)).cuda(), want_features=wf)
        ctx = "step %d" % t
        if wf:
            gu.assert_same("feature_obs", env.feature_obs.cpu().numpy(), o["feature_obs"], ctx)
        gu.assert_same("obs", obs.cpu().numpy(), o["obs"], ctx)
        gu.assert_same("rew", rew.cpu().numpy(), o["rew"], ctx)
        gu.assert_same("base_rew", env.base_rew.cpu().numpy(), o["base_rew"], ctx)
        gu.assert_same("transfers", env.transfers.cpu().numpy(), o["transfers"], ctx)
        gu.assert_same("info", info.cpu().numpy()[..., :3], o["info"][..., :3], ctx)
        gu.assert_same("done", done.cpu().numpy(), o["done"], ctx)
        if t % 10 == 0 or o["done"].any():
            check_state(ctx)
        if o["done"].any():          # masked reset of the finished envs (all of them here: equal horizons)
            mask = o["done"].copy()
            mask[::3] = 0             # reset only a subset; the others keep running past the horizon
            gu.assert_same("masked reset obs", env.reset(torch.as_tensor(mask).cuda()).cpu().numpy()[mask.astype(bool)],
                           orc.reset(mask)[mask.astype(bool)], ctx)
            check_state(ctx + " after reset")
    gu.assert_same("metrics", env.metrics_raw().cpu().numpy(), orc.metrics_raw(), "end")


@pytest.mark.parametrize("kind,n,H,W", [("cleanup", 8, 44, 60), ("harvest", 6, 40, 63), ("cleanup", 3, 48, 64)])
def test_big_map_matches_oracle(oracle_lib, kind, n, H, W):
    import torch
    from contracts_b200.batched import BatchedGridEnv
    amap = gu.big_map(kind, H, W, H * W)
    contract = "CleanupContract" if kind == "cleanup" else "HarvestFeaturemodLocalContract"
    E, steps = 24, 150
    orc = oracle_lib.GridOracle(kind, E, n, amap, horizon=60, contract=contract, seed=21, first_env_id=3)
    env = BatchedGridEnv(kind + "_new", E, n, amap, horizon=60, contract=contract, seed=21, first_env_id=3)
    assert env.state_map_bytes > 1024
    rng = np.random.RandomState(1)
    gu.assert_same("reset obs", env.reset().cpu().numpy(), orc.reset(), "reset")
    for t in range(steps):
        a = rng.randint(0, 9 if kind == "cleanup" else 8, size=(E, n))
        o = orc.step(a, want_features=(t % 5 == 0))
        obs, rew, done, info = env.step(torch.as_tensor(a.astype(np.uint8)).cuda(), want_features=(t % 5 == 0))
        ctx = "step %d" % t
        gu.assert_same("obs", obs.cpu().numpy(), o["obs"], ctx)
        gu.assert_same("rew", rew.cpu().numpy(), o["rew"], ctx)
        gu.assert_same("info", info.cpu().numpy()[..., :3], o["info"][..., :3], ctx)
        if t % 5 == 0:
            gu.assert_same("feature_obs", env.feature_obs.cpu().numpy(), o["feature_obs"], ctx)
        if o["done"].any():
            gu.assert_same("reset obs", env.reset(torch.as_tensor(o["done"]).cuda()).cpu().numpy()[o["done"].astype(bool)],
                           orc.reset(o["done"])[o["done"].astype(bool)], ctx)
    so, sc = orc.get_state(), env.get_state()
    for k in ("map", "pos", "ori", "t"):
        gu.assert_same(k, sc[k].cpu().numpy(), so[k], "end")
    gu.assert_same("metrics", env.metrics_raw().cpu().numpy(), orc.metrics_raw(), "end")


@pytest.mark.parametrize("kind,amap_name,n,nact", [("cleanup", "stock", 8, 9), ("cleanup", "cramped", 8, 9), ("harvest", "stock", 8, 8),
                                                   ("harvest", "cramped", 8, 8)])
def test_soak_many_envs_matches_oracle(oracle_lib, kind, amap_name, n, nact):
    """Thousands of envs for a few dozen steps: rare paths (long contested chains, 4+ shooters per env, overlapping
    agents, multi-apple spawns) at a rate the small rollouts do not reach."""
    import torch
    from contracts_b200.batched import BatchedGridEnv
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    amap = {"stock": CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP,
            "cramped": CRAMPED_CLEANUP if kind == "cleanup" else CRAMPED_HARVEST}[amap_name]
    contract = "CleanupContract" if kind == "cleanup" else "HarvestFeaturemodLocalContract"
    E, steps = 6000, 50
    orc = oracle_lib.GridOracle(kind, E, n, amap, horizon=1000, contract=contract, seed=99, first_env_id=123456)
    env = BatchedGridEnv(kind + "_new", E, n, amap, horizon=1000, contract=contract, seed=99, first_env_id=123456)
    rng = np.random.RandomState(7)
    gu.assert_same("reset obs", env.reset().cpu().numpy(), orc.reset(), "reset")
    if kind == "cleanup" and amap_name == "stock":       # start inside the spawning regime: clean most of the waste
        st = orc.get_state()
        m = st["map"].copy()
        waste = m == ord("H")
        keep = rng.rand(*m.shape) < 0.6
        m[waste & ~keep] = ord("R")
        orc.set_state(map=m); env.set_state(map=m)
    for t in range(steps):
        a = rng.randint(0, nact, size=(E, n))
        o = orc.step(a, want_features=False)
        obs, rew, done, info = env.step(torch.as_tensor(a.astype(np.uint8)).cuda())
        ctx = "step %d" % t
        gu.assert_same("rew", rew.cpu().numpy(), o["rew"], ctx)
        gu.assert_same("info", info.cpu().numpy()[..., :3], o["info"][..., :3], ctx)
        if t % 7 == 0 or t == steps - 1:
            gu.assert_same("obs", obs.cpu().numpy(), o["obs"], ctx)
            so, sc = orc.get_state(), env.get_state()
            for k in ("map", "pos", "ori"):
                gu.assert_same(k, sc[k].cpu().numpy(), so[k], ctx)
    gu.assert_same("metrics", env.metrics_raw().cpu().numpy(), orc.metrics_raw(), "end")


@pytest.mark.parametrize("kind", ["cleanup", "harvest"])
def test_random_maps_match_oracle(oracle_lib, kind):
    """Maps nobody drew by hand (golden_util.random_map: 6..14 x 6..14, inner walls, 2..8 agents, at least one cell of every
    dynamic kind — the same generator pins the oracle to the live reference in test_deep_differential.py): odd row pitches,
    one-entry point lists, windows that are mostly outside the map, corridors."""
    import torch
    from contracts_b200.batched import BatchedGridEnv
    contract = "CleanupContract" if kind == "cleanup" else "HarvestFeaturemodLocalContract"
    rng = np.random.RandomState(40 + len(kind))
    nact = 9 if kind == "cleanup" else 8
    for m in range(int(os.environ.get("SSD_GPU_MAPS", "10"))):
        n = int(rng.randint(2, 9))
        amap = gu.random_map(rng, kind, n)
        E, seed, first = 48, 500 + m, 1000 * m
        orc = oracle_lib.GridOracle(kind, E, n, amap, horizon=40, contract=contract, seed=seed, first_env_id=first)
        env = BatchedGridEnv(kind + "_new", E, n, amap, horizon=40, contract=contract, seed=seed, first_env_id=first)
        gu.assert_same("reset obs", env.reset().cpu().numpy(), orc.reset(), "map %d %r reset" % (m, amap))
        for t in range(60):
            a = rng.randint(0, nact, size=(E, n))
            feat = t % 4 == 0
            o = orc.step(a, want_features=feat)
            obs, rew, done, info = env.step(torch.as_tensor(a.astype(np.uint8)).cuda(), want_features=feat)
            ctx = "map %d %r step %d" % (m, amap, t)
            gu.assert_same("obs", obs.cpu().numpy(), o["obs"], ctx)
            gu.assert_same("rew", rew.cpu().numpy(), o["rew"], ctx)
            gu.assert_same("info", info.cpu().numpy()[..., :3], o["info"][..., :3], ctx)
            gu.assert_same("done", done.cpu().numpy(), o["done"], ctx)
            if feat:
                gu.assert_same("feature_obs", env.feature_obs.cpu().numpy(), o["feature_obs"], ctx)
            if o["done"].any():
                mask = o["done"].astype(bool)
                gu.assert_same("reset obs", env.reset(torch.as_tensor(o["done"]).cuda()).cpu().numpy()[mask], orc.reset(o["done"])[mask], ctx)
        so, sc = orc.get_state(), env.get_state()
        for k in ("map", "pos", "ori", "t"):
            gu.assert_same(k, sc[k].cpu().numpy(), so[k], "map %d end" % m)
        gu.assert_same("metrics", env.metrics_raw().cpu().numpy(), orc.metrics_raw(), "map %d end" % m)
        env.close()

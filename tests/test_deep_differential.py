"""Needs a checkout of the original project (SSD_REFERENCE_ROOT): the LIVE unmodified reference
(oracle/ref_harness.RefGridEnv, reference code under RNG injection) against the C oracle (oracle/ssd_oracle.c) over whole 1000-step episodes + re-resets, deep inside
the spawning regime that the short committed fixtures only touch: every output of every step by bit pattern — map,
agent positions / orientations, uint8 observations, rewards before / after transfers, transfers, infos, feature_obs,
theta at reset, and the episode metrics.  This is what pins the oracle (and through it the CUDA path, which the GPU
suite compares with the oracle on long rollouts) to the REFERENCE at depth, not only to the fixtures.

Default: 2 episodes of 1000 steps + a third reset per config (~10 s each).  SSD_DEEP_EPISODES=10 gives the >= 10^4
steps per config of SURVEY.md §8(c)(i).

Without a checkout of the reference, the default-size runs check the oracle's side of every comparison against
tests/golden/reference_tapes.json (golden_util.Tape: an ordered digest of the compared values).  Those digests were
recorded from the C oracle, which the live comparison of these exact runs had found bit-equal to the reference (the
runs were last extended in 177a073, and nothing under oracle/ changed after it), i.e. they are the reference's values
on the compared quantities; no reference checkout was at hand when they were stored.  The solver differential is not
stored: its decision rule consumes the reference's own value estimates.  Re-record them with a checkout present:
`SSD_REFERENCE_ROOT=<checkout> SSD_RECORD_REFERENCE_TAPES=1 python -m pytest tests/test_deep_differential.py`.
"""
import json
import os

import numpy as np
import pytest

import golden_util as gu
from oracle import ref_stubs

LIVE = ref_stubs.live_reference() is not None
EPISODES = int(os.environ.get("SSD_DEEP_EPISODES", "2"))
TAPES_PATH = os.path.join(gu.GOLDEN_DIR, "reference_tapes.json")
RECORD = os.environ.get("SSD_RECORD_REFERENCE_TAPES") == "1"
DEFAULT_SIZE = "SSD_DEEP_EPISODES" not in os.environ and "SSD_DEEP_MAPS" not in os.environ
needs_live = pytest.mark.skipif(not LIVE, reason="SSD_REFERENCE_ROOT does not name a checkout of the original project")


@pytest.fixture(autouse=True)
def reference_side(request):
    """With the reference: the live comparison (and, with SSD_RECORD_REFERENCE_TAPES=1, its digests are stored).  Without
    it: the comparisons run against the stored digests of the reference's values (gu.STORED stands for its outputs)."""
    if LIVE and not RECORD:
        yield
        return
    if not DEFAULT_SIZE:
        pytest.skip("stored reference digests cover the default run sizes only")
    name = request.node.name
    stored = None
    if not RECORD:
        with open(TAPES_PATH) as f:
            stored = json.load(f)[name]
    gu.TAPE = tape = gu.Tape(name, stored)
    try:
        yield
    finally:
        gu.TAPE = None
    tape.finish()
    if RECORD:
        tapes = json.load(open(TAPES_PATH)) if os.path.exists(TAPES_PATH) else {}
        tapes[name] = tape.marks
        with open(TAPES_PATH, "w") as f:
            json.dump(dict(sorted(tapes.items())), f, indent=0)
            f.write("\n")

# (kind, n, action ids, action probabilities): the cleaning-heavy cleanup policies drive #waste far below the spawn
# threshold so that apples spawn, are eaten, and waste respawns for most of the episode
CASES = [("cleanup", 8, 9, [.14, .14, .14, .14, .02, .04, .04, .32, .02]),
         ("cleanup", 2, 9, [.12, .12, .12, .12, .02, .05, .05, .38, .02]),
         ("cleanup", 8, 8, None),                                   # the benchmark's iid uniform policy
         ("harvest", 4, 8, None),
         ("harvest", 8, 7, None)]


@pytest.mark.parametrize("kind,n,nact,probs", CASES, ids=["%s_n%d_a%d" % c[:3] for c in CASES])
def test_reference_vs_oracle_full_episodes(oracle_lib, kind, n, nact, probs):
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    from oracle.ref_harness import RefGridEnv
    seed, env_id = 900 + n, 31000 + 17 * n
    contract = "CleanupContract" if kind == "cleanup" else "HarvestFeaturemodLocalContract"
    amap = CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP
    ref = RefGridEnv(kind, n, seed, env_id, contract=True, horizon=1000) if LIVE else None
    orc = oracle_lib.GridOracle(kind, 1, n, amap, horizon=1000, contract=contract, seed=seed, first_env_id=env_id)
    rng = np.random.RandomState(7 * n + len(kind))
    min_waste, max_apples, eaten, paid = 10 ** 9, 0, 0, 0
    for ep in range(EPISODES + 1):
        ctx = "%s n=%d episode %d reset" % (kind, n, ep)
        r0 = ref.reset() if ref else gu.STORED
        gu.assert_same("reset obs", orc.reset()[0], r0["obs"], ctx)
        st = orc.get_state()
        gu.assert_same("reset map", st["map"][0], r0["map"], ctx)
        gu.assert_same("reset pos", st["pos"][0], r0["pos"], ctx)
        gu.assert_same("reset ori", st["ori"][0], r0["ori"], ctx)
        gu.assert_same("reset theta", st["theta"][0], r0["theta"], ctx)
        if ep == EPISODES:
            break
        for t in range(1000):
            a = rng.choice(nact, size=n, p=probs).astype(np.int32)
            want = ref.step(a) if ref else gu.STORED
            got = orc.step(a[None], want_features=True)
            ctx = "%s n=%d episode %d step %d" % (kind, n, ep, t + 1)
            gu.assert_same("obs", got["obs"][0], want["obs"], ctx)
            gu.assert_same("rew", got["rew"][0], want["rew"], ctx)
            gu.assert_same("base_rew", got["base_rew"][0], want["base_rew"], ctx)
            gu.assert_same("transfers", got["transfers"][0], want["transfers"], ctx)
            gu.assert_same("eaten_apples", got["info"][0][:, 0], want["eaten_apples"], ctx)
            gu.assert_same("info1", got["info"][0][:, 1],
                           want["cleaned_squares"] if kind == "cleanup" else want["eaten_close_apples"], ctx)
            gu.assert_same("feature_obs", got["feature_obs"][0], want["feature_obs"], ctx)
            gu.assert_same("done", int(got["done"][0]), want["done"], ctx)
            assert bool(got["done"][0]) == (t == 999), ctx
            if t % 25 == 0 or t == 999:                      # full state (the observations already cover it every step)
                st = orc.get_state()
                gu.assert_same("map", st["map"][0], want["map"], ctx)
                gu.assert_same("pos", st["pos"][0], want["pos"], ctx)
                gu.assert_same("ori", st["ori"][0], want["ori"], ctx)
                # (the counters read the oracle's side: it has just been found equal to the reference's)
                if kind == "cleanup":
                    min_waste = min(min_waste, int((st["map"][0] == ord("H")).sum()))
                max_apples = max(max_apples, int((st["map"][0] == ord("A")).sum()))
            eaten += int(got["info"][0][:, 0].sum())
            paid += int((got["transfers"][0] != 0).sum())
        want_m = ref.metrics() if ref else gu.STORED
        assert "equality" in want_m and "transfer_sustainability" in want_m          # the episode really ended
        gu.check_episode_metrics(kind, n, True, orc.metrics_raw()[0], want_m, "%s n=%d episode %d end" % (kind, n, ep))
    # the run really was deep: the regime the short fixtures do not reach
    if kind == "cleanup" and probs is not None:
        # (two agents cannot out-clean the waste respawn: they hover at the spawn threshold of 47 cells)
        assert min_waste <= (42 if n == 8 else 47) and max_apples >= 10 and eaten > 0 and paid > 0, (min_waste, max_apples, eaten, paid)
    if kind == "harvest":
        assert eaten > 0


# ---- feature envs and selfdrive: the same differential, live reference vs C oracle ----------------------------------
# (default: one episode + re-reset per case to keep the CPU suite short; SSD_DEEP_EPISODES scales it up)
FEAT_EPISODES = max(1, EPISODES // 2)
FEAT_CASES = [("cleanup", 8, 9, None), ("cleanup", 3, 8, [.12, .12, .12, .12, .06, .06, .06, .34]), ("harvest", 8, 8, None),
              ("harvest", 4, 7, None)]


@pytest.mark.parametrize("kind,n,nact,probs", FEAT_CASES, ids=["feat_%s_n%d_a%d" % c[:3] for c in FEAT_CASES])
def test_reference_vs_oracle_feature_envs_full_episodes(oracle_lib, kind, n, nact, probs):
    """CleanupFeatures / HarvestFeatures (cleanup_features.py:156-284, harvest_features.py:173-336) + subgame wrapper:
    whole 1000-step episodes + re-resets of the LIVE reference against features_oracle.c — observations, positions,
    orientations, the apple / waste cells, rewards before / after transfers, transfers, infos, theta, done, metrics."""
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    from oracle.ref_harness import RefFeatEnv
    seed, env_id = 700 + n, 41000 + 13 * n
    contract = "CleanupContract" if kind == "cleanup" else "HarvestFeaturemodLocalContract"
    amap = CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP
    ref = RefFeatEnv(kind, n, seed, env_id, contract=True, horizon=1000) if LIVE else None
    orc = oracle_lib.FeatOracle(kind, 1, n, amap, horizon=1000, contract=contract, seed=seed, first_env_id=env_id)
    rng = np.random.RandomState(11 * n + len(kind) + nact)
    paid, eaten = 0, 0
    for ep in range(FEAT_EPISODES + 1):
        ctx = "features %s n=%d episode %d reset" % (kind, n, ep)
        r0 = ref.reset() if ref else gu.STORED
        gu.assert_same("reset obs", orc.reset()[0], r0["obs"][:, :orc.F], ctx)
        st = orc.get_state()
        for k in ("pos", "ori", "cells"):
            gu.assert_same("reset " + k, st[k][0], r0[k], ctx)
        gu.assert_same("reset theta", st["theta"][0], r0["theta"], ctx)
        if ep == FEAT_EPISODES:
            break
        for t in range(1000):
            a = rng.choice(nact, size=n, p=probs).astype(np.int32)
            want = ref.step(a) if ref else gu.STORED
            got = orc.step(a[None])
            ctx = "features %s n=%d episode %d step %d" % (kind, n, ep, t + 1)
            gu.assert_same("obs", got["obs"][0], want["obs"][:, :orc.F], ctx)
            gu.assert_same("rew", got["rew"][0], want["rew"], ctx)
            gu.assert_same("base_rew", got["base_rew"][0], want["base_rew"], ctx)
            gu.assert_same("transfers", got["transfers"][0], want["transfers"], ctx)
            gu.assert_same("info0", got["info"][0][:, 0], want["info0"], ctx)
            gu.assert_same("info1", got["info"][0][:, 1], want["info1"], ctx)
            gu.assert_same("done", bool(got["done"][0]), want["done"], ctx)
            paid += int(np.count_nonzero(got["transfers"][0])); eaten += int(got["base_rew"][0].sum())
            if t % 25 == 0 or t == 999:
                st = orc.get_state()
                for k in ("pos", "ori", "cells"):
                    gu.assert_same(k, st[k][0], want[k], ctx)
        raw = orc.metrics_raw()[0]
        m = ref.metrics() if ref else gu.STORED
        gu.assert_same("metric raw_env_rewards", np.float64(raw[1]), gu._f64(m["raw_env_rewards"]), "episode %d" % ep)
        gu.assert_same("metric transfers", np.float64(raw[2]), gu._f64(m["transfers"]), "episode %d" % ep)
    assert paid > 0 and eaten > 0          # the contract paid and apples were eaten: the interesting paths ran


# (n, contract, non-default constructor kwargs of SelfAcceleratingCarEnv, self_driving_car_accelerate.py:19)
CAR_CASES = [(8, True, {}), (4, True, {}), (2, False, {}),
             (5, True, dict(low_bound=-4.5, high_bound=6.25, start_vel=0.35, start_vel_ambulance=0.55)),
             (3, True, dict(low_bound=-20.0, high_bound=3.0, start_vel=0.05, start_vel_ambulance=1.0))]


@pytest.mark.parametrize("n,contract,track", CAR_CASES,
                         ids=["car_n%d_%s%s" % (n, "contract" if c else "plain", "_track" if k else "") for n, c, k in CAR_CASES])
def test_reference_vs_oracle_selfdrive_many_episodes(oracle_lib, n, contract, track):
    """SelfAcceleratingCarEnv (+ SelfdriveContractDistprop; self_driving_car_accelerate.py:49-250, contract_list.py:66-102):
    many whole episodes of the LIVE reference against selfdrive_oracle.c, every output by bit pattern."""
    from oracle.ref_harness import RefCarEnv
    seed, env_id = 800 + n, 51000 + 7 * n
    ref = RefCarEnv(n, seed, env_id, contract=contract, **track) if LIVE else None
    orc = oracle_lib.CarOracle(1, n, contract=contract, seed=seed, first_env_id=env_id, **track)
    rng = np.random.RandomState(3 * n + 1)
    D = orc.D
    steps_total, paid, overtakes = 0, 0, 0
    for ep in range(10 * EPISODES):
        ctx = "selfdrive n=%d episode %d reset" % (n, ep)
        r0 = ref.reset() if ref else gu.STORED
        gu.assert_same("reset obs", orc.reset()[0], r0["obs"][:, :D], ctx)
        if contract:
            gu.assert_same("reset theta", orc.get_state()["theta"][0], r0["theta"], ctx)
        scale = [0.15, 0.05, 0.3][ep % 3]
        for t in range(2000):
            a = (rng.uniform(-0.7, 1.0, size=n) * scale).astype(np.float32)
            want = ref.step(a) if ref else gu.STORED
            got = orc.step(a[None])
            ctx = "selfdrive n=%d episode %d step %d" % (n, ep, t + 1)
            gu.assert_same("active", got["info"][0][:, 1], want["active"], ctx)
            act = got["info"][0][:, 1].astype(bool)
            gu.assert_same("obs", got["obs"][0][act], want["obs"][act][:, :D], ctx)
            gu.assert_same("rew", got["rew"][0], want["rew"], ctx)
            gu.assert_same("done", got["done"][0], want["done"], ctx)
            gu.assert_same("just_passed", got["info"][0][:, 0].astype(np.uint8), want["just_passed"], ctx)
            first = int(np.argmax(act))
            gu.assert_same("ambulance_rank", np.float64(got["info"][0][first, 2]), want["ambulance_rank"], ctx)
            gu.assert_same("ambulance_dist_to_front", np.float64(got["info"][0][first, 3]), want["ambulance_dist_to_front"], ctx)
            st = orc.get_state()
            gu.assert_same("pos", st["pos"][0], want["pos"], ctx)
            gu.assert_same("vel", st["vel"][0], want["vel"], ctx)
            gu.assert_same("metric transfers", np.float64(st["transfers"][0]), want["metric_transfers"], ctx)
            if contract:
                gu.assert_same("base_rew", got["base_rew"][0], want["base_rew"], ctx)
                gu.assert_same("transfers", got["transfers"][0], want["transfers"], ctx)
                paid += int(np.count_nonzero(got["transfers"][0]))
            steps_total += 1
            if got["done"][0][-1]:
                break
        else:
            raise AssertionError("episode did not end")
    assert steps_total > (500 if not track else 100)
    assert (paid > 0) == bool(contract)


# ---- random maps: the live reference against the C oracle away from the two stock layouts -----------------------------
@pytest.mark.parametrize("kind", ["cleanup", "harvest"])
def test_reference_vs_oracle_random_maps(oracle_lib, kind):
    """MapEnv on maps it never shipped with (map_env.py:61-170 parses any ascii map): per map the reset, 150 steps and the
    step-151 state of the LIVE reference against the oracle — map parsing, point-list order, spawn probabilities
    (cleanup_new.py:351-372 for any waste area), view windows at the border, contested moves in corridors."""
    from oracle.ref_harness import RefGridEnv
    contract = "CleanupContract" if kind == "cleanup" else "HarvestFeaturemodLocalContract"
    maps = int(os.environ.get("SSD_DEEP_MAPS", "6")) * max(1, EPISODES // 2)
    rng = np.random.RandomState(20 + len(kind))
    eaten = fired = 0
    for m in range(maps):
        n = int(rng.randint(2, 9))
        amap = gu.random_map(rng, kind, n)
        seed, env_id = 300 + m, 52000 + 7 * m
        ref = RefGridEnv(kind, n, seed, env_id, contract=True, ascii_map=amap, horizon=100) if LIVE else None
        orc = oracle_lib.GridOracle(kind, 1, n, amap, horizon=100, contract=contract, seed=seed, first_env_id=env_id)
        ctx = "%s map %d %r reset" % (kind, m, amap)
        r0 = ref.reset() if ref else gu.STORED
        gu.assert_same("reset obs", orc.reset()[0], r0["obs"], ctx)
        st = orc.get_state()
        for k in ("map", "pos", "ori", "theta"):
            gu.assert_same("reset " + k, st[k][0], r0[k], ctx)
        nact = 9 if kind == "cleanup" else 8
        for t in range(150):
            if t == 100:                                        # the episode ended at the horizon: second episode
                r0 = ref.reset() if ref else gu.STORED
                gu.assert_same("re-reset obs", orc.reset()[0], r0["obs"], ctx)
            a = rng.randint(0, nact, size=n).astype(np.int32)
            want = ref.step(a) if ref else gu.STORED
            got = orc.step(a[None], want_features=True)
            ctx = "%s map %d %r step %d" % (kind, m, amap, t + 1)
            for k in ("obs", "rew", "base_rew", "transfers", "feature_obs"):
                gu.assert_same(k, got[k][0], want[k], ctx)
            gu.assert_same("eaten_apples", got["info"][0][:, 0], want["eaten_apples"], ctx)
            gu.assert_same("info1", got["info"][0][:, 1],
                           want["cleaned_squares"] if kind == "cleanup" else want["eaten_close_apples"], ctx)
            gu.assert_same("done", int(got["done"][0]), want["done"], ctx)
            if t % 10 == 0 or t == 149:
                st = orc.get_state()
                for k in ("map", "pos", "ori"):
                    gu.assert_same(k, st[k][0], want[k], ctx)
            eaten += int(got["info"][0][:, 0].sum())
            fired += int((a >= 7).sum())
    assert fired > 0 and (kind == "cleanup" or eaten > 0)


# ---- negotiation stage: many live agreement draws ----------------------------------------------------------------------
@pytest.mark.parametrize("kind,n", [("cleanup", 2), ("cleanup", 3), ("cleanup", 4), ("cleanup", 8), ("harvest", 4), ("harvest", 5)])
def test_reference_vs_oracle_negotiation_many_episodes(oracle_lib, kind, n):
    """SeparateContractNegotiateStage (two_stage_train.py:257-358) of the LIVE reference against the oracle over many
    episodes with accept probabilities across [0, 1]: the agreement (all agents for n <= 3, two sampled ones of a1.. for
    n > 3, product of their accept values against one uniform, :266-281), the contract every agent then observes, the summed
    rewards of the short frozen-policy rollout and the final observation."""
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    from oracle.ref_harness import RefNegotiateEnv
    episodes = 12 * max(1, EPISODES // 2)
    horizon, base_horizon = 4, 1000
    rng = np.random.RandomState(5 * n + len(kind))
    table = rng.randint(0, 9 if kind == "cleanup" else 8, size=(horizon, n))
    seed, env_id = 60 + n, 7000 + n
    ref = RefNegotiateEnv(kind, n, seed, env_id, horizon, base_horizon, table) if LIVE else None
    contract = "CleanupContract" if kind == "cleanup" else "HarvestFeaturemodLocalContract"
    orc = oracle_lib.GridOracle(kind, 1, n, CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP, horizon=base_horizon,
                                contract=contract, seed=seed, first_env_id=env_id)
    high = 0.2 if kind == "cleanup" else 10.0
    outcomes = set()
    for ep in range(episodes):
        ctx = "%s n=%d episode %d" % (kind, n, ep)
        r0 = ref.reset() if ref else gu.STORED
        gu.assert_same("reset obs", orc.reset()[0], r0["obs"], ctx)
        acts = np.stack([rng.uniform(0, high, size=n), rng.uniform(0.3, 1.0, size=n) ** (1.0 / max(1, min(n - 1, 2)))], axis=1)
        if ref:
            s2 = ref.step(acts)
            s3 = ref.step(acts)
            assert not s2["done"] and s3["done"], ctx
        else:
            s3 = gu.STORED
        dec = orc.negotiate(acts[0, 0], acts[:, 1])
        gu.assert_same("accepted", dec[0], s3["accepted"], ctx)
        gu.assert_same("theta", orc.get_state()["theta"][0], s3["contract_obs"][0, 0], ctx)
        total = np.zeros(n)
        for t in range(horizon):
            r = orc.step(table[t][None], want_features=False)
            total = total + r["rew"][0]
        gu.assert_same("summed rewards", total, s3["rew"], ctx)
        gu.assert_same("final obs", r["obs"][0], s3["obs"], ctx)
        outcomes.add(int(dec[0]))
    assert outcomes == {0, 1}, "both outcomes must occur: %r" % (outcomes,)


# ---- NegotiationSolver: many live candidate draws and decisions -----------------------------------------------------
@needs_live          # the decision rule consumes the reference's own value estimates (r0["vals"]): not stored
@pytest.mark.parametrize("kind,n,S,rule", [("cleanup", 2, 5, "max"), ("cleanup", 4, 20, "majority"), ("cleanup", 8, 50, "majority"),
                                           ("harvest", 4, 20, "max"), ("harvest", 8, 7, "majority")])
def test_reference_vs_oracle_solver_many_episodes(oracle_lib, kind, n, S, rule):
    """NegotiationSolver.negotiate / compute_best_param (two_stage_train.py:705-776) of the LIVE reference (scripted value
    function, oracle/scripted.py) against the oracle's restatement: the 1 + S candidate contracts of every episode, the
    chosen contract under the configured rule, and three contract-wrapped steps."""
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    from oracle.ref_harness import RefSolverEnv
    episodes = 10 * max(1, EPISODES // 2)
    seed, env_id = 80 + n + S, 9000 + 3 * n
    ref = RefSolverEnv(kind, n, seed, env_id, S, rule, horizon=50)
    contract = "CleanupContract" if kind == "cleanup" else "HarvestFeaturemodLocalContract"
    orc = oracle_lib.GridOracle(kind, 1, n, CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP, horizon=50, contract=contract,
                                seed=seed, first_env_id=env_id)
    high = float(np.float32(0.2)) if kind == "cleanup" else float(np.float32(10.0))
    rng = np.random.RandomState(n + S)
    chosen = set()
    for ep in range(episodes):
        ctx = "%s n=%d S=%d %s episode %d" % (kind, n, S, rule, ep)
        r0 = ref.reset()
        gu.assert_same("reset obs", orc.reset()[0], r0["obs"], ctx)
        params = oracle_lib.solver_candidates(seed, env_id, ep, 0.0, high, S)
        gu.assert_same("candidates", params, r0["params"], ctx)
        theta, idx = oracle_lib.solver_choose(params, r0["vals"], rule)
        gu.assert_same("theta", theta, r0["theta"], ctx)
        chosen.add(int(idx))
        orc.set_theta(theta)
        for t in range(3):
            a = rng.randint(0, 9 if kind == "cleanup" else 8, size=n).astype(np.int32)
            want = ref.step(a)
            got = orc.step(a[None], want_features=False)
            gu.assert_same("obs", got["obs"][0], want["obs"], ctx)
            gu.assert_same("rew", got["rew"][0], want["rew"], ctx)
            gu.assert_same("contract obs", np.array([theta, 0.0]), want["contract_obs"][0], ctx)
    assert len(chosen) > 1, "the decision never varied: %r" % (chosen,)


# ---- JointEnv layouts and rendered frames, live -------------------------------------------------------------------------
@pytest.mark.parametrize("kind,n,mode", [("cleanup", 2, "global"), ("cleanup", 8, "concatenated"), ("harvest", 4, "global"),
                                         ("harvest", 5, "concatenated")])
def test_reference_vs_oracle_joint_env_episodes(oracle_lib, kind, n, mode):
    """JointEnv (two_stage_train.py:476-617) of the LIVE reference against the oracle: the global map / the channel-
    concatenated windows, the summed reward, done, and the infos summed key by key, over whole short episodes + re-resets."""
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    from oracle.ref_harness import RefJointEnv
    horizon = 120
    seed, env_id = 40 + n, 3000 + n
    ref = RefJointEnv(kind, n, seed, env_id, mode, horizon=horizon) if LIVE else None
    orc = oracle_lib.GridOracle(kind, 1, n, CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP, horizon=horizon, contract=None,
                                seed=seed, first_env_id=env_id)
    rng = np.random.RandomState(3 * n + len(mode))
    view = (lambda obs: orc.global_view()[0]) if mode == "global" else (lambda obs: oracle_lib.concatenated_obs(obs)[0])
    for ep in range(max(2, EPISODES)):
        gu.assert_same("reset obs", view(orc.reset()), ref.reset() if ref else gu.STORED, "%s %s episode %d reset" % (kind, mode, ep))
        for t in range(horizon):
            ctx = "%s n=%d %s episode %d step %d" % (kind, n, mode, ep, t + 1)
            a = rng.randint(0, 9 if kind == "cleanup" else 8, size=n).astype(np.int32)
            want = ref.step(a) if ref else gu.STORED
            o = orc.step(a[None], want_features=True)
            gu.assert_same("obs", view(o["obs"]), want["obs"], ctx)
            rew = 0
            for r in o["rew"][0]:                                  # sum(env_rews.values()) in agent order (:592)
                rew = rew + r
            gu.assert_same("rew", np.float64(rew), want["rew"], ctx)
            gu.assert_same("done", int(o["done"][0]), want["done"], ctx)
            assert bool(o["done"][0]) == (t == horizon - 1), ctx
            gu.assert_same("eaten_apples", int(o["info"][0, :, 0].sum()), want["eaten_apples"], ctx)
            gu.assert_same("info1", int(o["info"][0, :, 1].sum()), want["info1"], ctx)
            feat = 0
            for i in range(n):
                feat = feat + o["feature_obs"][0, i]
            gu.assert_same("feature_obs", feat, want["feature_obs"], ctx)


@pytest.mark.parametrize("kind,n", [("cleanup", 8), ("harvest", 6)])
def test_reference_vs_oracle_rendered_frames(oracle_lib, kind, n):
    """render(mode='rgb_array') = full_map_to_colors with the beams of the last step (map_env.py:354-392,460-475), every
    frame of a firing-heavy rollout on the stock map."""
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    from oracle.ref_harness import RefGridEnv
    seed, env_id = 90 + n, 6100 + n
    probs = [.1, .1, .1, .1, .05, .1, .1, .2, .15] if kind == "cleanup" else [.12, .12, .12, .12, .06, .1, .1, .26]
    ref = RefGridEnv(kind, n, seed, env_id, contract=False, horizon=1000, disable_firing=False) if LIVE else None
    frame = (lambda: np.asarray(ref.base.render(mode="rgb_array"), dtype=np.uint8)) if ref else (lambda: gu.STORED)
    orc = oracle_lib.GridOracle(kind, 1, n, CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP, horizon=1000, seed=seed,
                                first_env_id=env_id)
    rng = np.random.RandomState(n)
    if ref:
        ref.reset()
    orc.reset()
    gu.assert_same("reset frame", orc.render()[0], frame(), "reset")
    beams = 0
    for t in range(150 * max(1, EPISODES // 2)):
        a = rng.choice(len(probs), size=n, p=probs).astype(np.int32)
        if ref:
            ref.step(a)
        orc.step(a[None], want_features=False)
        got = orc.render()[0]
        gu.assert_same("frame", got, frame(), "%s n=%d step %d" % (kind, n, t + 1))
        beams += int(((got == (255, 255, 0)).all(-1) | (got == (100, 255, 255)).all(-1)).sum())
    assert beams > 100


# ---- reward shaping over whole episodes ------------------------------------------------------------------------------
SHAPED = [("cleanup", 8, dict(use_collective_reward=True)),
          ("cleanup", 5, dict(inequity_averse_reward=True, alpha=5.0, beta=0.05)),
          ("harvest", 4, dict(use_collective_reward=True, inequity_averse_reward=True, alpha=-0.7, beta=0.9)),
          ("harvest", 8, dict(inequity_averse_reward=True, alpha=0.3, beta=-1.1))]


@pytest.mark.parametrize("kind,n,shaping", SHAPED, ids=["%s_n%d_%s" % (k, n, "+".join(sorted(s)[:2])) for k, n, s in SHAPED])
def test_reference_vs_oracle_shaped_rewards_full_episodes(oracle_lib, kind, n, shaping):
    """use_collective_reward / inequity_averse_reward (map_env.py:289-301) with the contract wrapper on top, whole 400-step
    episodes + re-reset: the float64 shaped rewards, the transfers computed from them, and the episode metrics."""
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    from oracle.ref_harness import RefGridEnv
    horizon = 400
    seed, env_id = 120 + n, 8800 + n
    contract = "CleanupContract" if kind == "cleanup" else "HarvestFeaturemodLocalContract"
    ref = RefGridEnv(kind, n, seed, env_id, contract=True, horizon=horizon, **shaping) if LIVE else None
    orc = oracle_lib.GridOracle(kind, 1, n, CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP, horizon=horizon, contract=contract,
                                seed=seed, first_env_id=env_id, **shaping)
    rng = np.random.RandomState(n)
    probs = [.12, .12, .12, .12, .02, .05, .05, .38, .02] if kind == "cleanup" else None
    nact = 9 if kind == "cleanup" else 8
    nonint = 0
    for ep in range(max(2, EPISODES)):
        gu.assert_same("reset obs", orc.reset()[0], ref.reset()["obs"] if ref else gu.STORED, "%s n=%d episode %d reset" % (kind, n, ep))
        for t in range(horizon):
            a = rng.choice(nact, size=n, p=probs).astype(np.int32)
            want = ref.step(a) if ref else gu.STORED
            got = orc.step(a[None], want_features=False)
            ctx = "%s n=%d %r episode %d step %d" % (kind, n, shaping, ep, t + 1)
            for k in ("obs", "rew", "base_rew", "transfers"):
                gu.assert_same(k, got[k][0], want[k], ctx)
            gu.assert_same("done", int(got["done"][0]), want["done"], ctx)
            nonint += int((got["base_rew"][0] != np.rint(got["base_rew"][0])).sum())
        gu.check_episode_metrics(kind, n, True, orc.metrics_raw()[0], ref.metrics() if ref else gu.STORED,
                                 "%s n=%d episode %d end" % (kind, n, ep))
    if shaping.get("inequity_averse_reward") and not shaping.get("use_collective_reward"):
        # (after the collective reward every agent holds the same sum, so the inequity terms vanish, map_env.py:289-301)
        assert nonint > 0, "the shaping never produced a fractional reward"


# ---- null contracts ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("family,kind,n", [("grid", "cleanup", 4), ("grid", "harvest", 3), ("feat", "cleanup", 5), ("feat", "harvest", 4),
                                           ("car", None, 6)])
def test_reference_vs_oracle_null_contract_probability(oracle_lib, family, kind, n):
    """SeparateContractSubgameStage.reset with null_prob > 0 (two_stage_train.py:159-166): `rand() > null_prob` decides
    between a uniform contract parameter and the null contract (contract_low); many resets, both branches, and a few
    steps under each drawn parameter."""
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    from oracle import ref_harness as rh
    null_prob, seed, env_id = 0.45, 140 + n, 7700 + n
    if family == "grid":
        contract = "CleanupContract" if kind == "cleanup" else "HarvestFeaturemodLocalContract"
        ref = rh.RefGridEnv(kind, n, seed, env_id, contract=True, null_prob=null_prob, horizon=1000) if LIVE else None
        orc = oracle_lib.GridOracle(kind, 1, n, CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP, horizon=1000, contract=contract,
                                    null_prob=null_prob, seed=seed, first_env_id=env_id)
        theta_of = lambda: orc.get_state()["theta"][0]                       # noqa: E731
        act = lambda rng: rng.randint(0, 9 if kind == "cleanup" else 8, size=n).astype(np.int32)   # noqa: E731
    elif family == "feat":
        contract = "CleanupContract" if kind == "cleanup" else "HarvestFeaturemodLocalContract"
        ref = rh.RefFeatEnv(kind, n, seed, env_id, contract=True, null_prob=null_prob, horizon=1000) if LIVE else None
        orc = oracle_lib.FeatOracle(kind, 1, n, CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP, horizon=1000, contract=contract,
                                    null_prob=null_prob, seed=seed, first_env_id=env_id)
        theta_of = lambda: orc.get_state()["theta"][0]                       # noqa: E731
        act = lambda rng: rng.randint(0, 8 if kind == "cleanup" else 7, size=n).astype(np.int32)   # noqa: E731
    else:
        ref = rh.RefCarEnv(n, seed, env_id, contract=True, null_prob=null_prob) if LIVE else None
        orc = oracle_lib.CarOracle(1, n, contract="SelfdriveContractDistprop", null_prob=null_prob, seed=seed, first_env_id=env_id)
        theta_of = lambda: orc.get_state()["theta"][0]                       # noqa: E731
        act = lambda rng: rng.uniform(-0.1, 0.1, size=n).astype(np.float32)  # noqa: E731
    rng = np.random.RandomState(n)
    nulls = drawn = 0
    for ep in range(30 * max(1, EPISODES // 2)):
        ctx = "%s %s n=%d episode %d" % (family, kind, n, ep)
        r0 = ref.reset() if ref else gu.STORED
        orc.reset()
        gu.assert_same("theta", theta_of(), r0["theta"], ctx)
        nulls += int(theta_of() == 0.0)
        drawn += int(theta_of() != 0.0)
        for t in range(4):
            a = act(rng)
            want = ref.step(a) if ref else gu.STORED
            got = orc.step(a[None]) if family != "grid" else orc.step(a[None], want_features=False)
            gu.assert_same("rew", got["rew"][0], want["rew"], ctx + " step %d" % t)
            gu.assert_same("transfers", got["transfers"][0], want["transfers"], ctx + " step %d" % t)
    assert nulls > 3 and drawn > 3, (nulls, drawn)

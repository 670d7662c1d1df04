"""GPU: the episode log (ssd_set_episode_log, contracts_b200/episodes.py) against the C oracles, bit for bit.

The expected record of an oracle env is its metrics row, t and theta read just before the oracle resets it, with its
episode counter.  Records are compared sorted by (env_id, episode)."""
import ctypes

import numpy as np
import pytest

import golden_util as gu

pytestmark = pytest.mark.gpu

CONTRACT = {"cleanup": "CleanupContract", "harvest": "HarvestFeaturemodLocalContract"}


def _maps(kind):
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    return CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP


class Expected:
    """records the oracle would have logged"""

    def __init__(self):
        self.rows = []

    def add(self, env_id, episode, t, ended, theta, metrics):
        m = np.zeros(56)
        m[:len(metrics)] = metrics
        self.rows.append((int(env_id), int(episode), int(t), bool(ended), np.float64(theta), m))

    def grid(self, orc, mask, first, horizon):
        """orc (GridOracle / FeatOracle of E envs) is about to reset the envs of mask (bool [E])"""
        rows, st = orc.metrics_raw(), orc.get_state()
        for i in np.nonzero(mask & (orc.episode >= 0))[0]:
            self.add(first + i, orc.episode[i], st["t"][i], st["t"][i] == horizon, st["theta"][i], rows[i])

    def check(self, got, ctx=""):
        rows = sorted(self.rows, key=lambda r: (r[0], r[1]))
        assert got["lost"] == 0, ctx
        assert len(got["env_id"]) == len(rows), "%s: %d records, want %d" % (ctx, len(got["env_id"]), len(rows))
        if not rows:
            return
        gu.assert_same("env_id", got["env_id"], [r[0] for r in rows], ctx)
        gu.assert_same("episode", got["episode"], [r[1] for r in rows], ctx)
        gu.assert_same("t", got["t"], [r[2] for r in rows], ctx)
        gu.assert_same("ended", got["ended"], [r[3] for r in rows], ctx)
        gu.assert_same("theta", got["theta"], [r[4] for r in rows], ctx)
        gu.assert_same("metrics", got["metrics"], np.stack([r[5] for r in rows]), ctx)


def _log(env, capacity=None):
    from contracts_b200.episodes import EpisodeLog
    log = EpisodeLog(env, capacity)
    env.set_episode_log(log)
    return log


def _check_stats(stats, m):
    """the ssd_set_episode_stats vector set on the same handle against sums over the records' metrics rows m [R, 56]"""
    s = stats.cpu().numpy()
    assert s[0] == m[:, 0].sum() and s[3] == m[:, 4].sum() and s[6] == len(m)          # integer-valued: exact
    assert s[7] == (m[:, 5].max() if len(m) else 0.0)
    for k, want in ((1, m[:, 2].sum()), (2, m[:, 3].sum()), (4, m[:, 40:48].sum()), (5, m[:, 24:32].sum())):
        assert np.isclose(s[k], want, rtol=1e-12, atol=1e-9), (k, s[k], want)      # atomics: summation order


# ---- 1. grid worlds ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("form", ["u8", "bf16"])
@pytest.mark.parametrize("kind", ["cleanup", "harvest"])
def test_grid_log_matches_oracle(oracle_lib, logic_variant, kind, form):
    import torch
    from contracts_b200.batched import BatchedGridEnv
    E, n, H, first, seed = 50, 5, 30, 1000, 17
    c = CONTRACT[kind]
    env = BatchedGridEnv(kind + "_new", E, n, _maps(kind), horizon=H, contract=c, seed=seed, first_env_id=first,
                         policy_dtype=torch.bfloat16 if form == "bf16" else None)
    orc = oracle_lib.GridOracle(kind, E, n, _maps(kind), horizon=H, contract=c, seed=seed, first_env_id=first)
    log = _log(env, 1000)
    stats = torch.zeros(8, dtype=torch.float64, device="cuda")
    env.set_episode_stats(stats)
    exp = Expected()
    rng = np.random.RandomState(5)
    nact = 9 if kind == "cleanup" else 8
    env.reset()
    orc.reset()
    dec = torch.zeros(E, dtype=torch.uint8, device="cuda")
    for t in range(4 * H):
        a = rng.randint(0, nact, size=(E, n))
        if t in (11, 47):                                   # masked resets mid-episode (and at t = 0 for some envs)
            m = rng.rand(E) < 0.3
            exp.grid(orc, m, first, H)
            env.reset(torch.as_tensor(m.astype(np.uint8)).cuda())
            orc.reset(m.astype(np.uint8))
        if t < 20:                                          # plain steps first: the envs end at different steps
            env.step(torch.as_tensor(a.astype(np.uint8)).cuda())
            orc.step(a, want_features=False)
            continue
        prop, acc = rng.uniform(0.0, 0.2, E), rng.uniform(0.3, 1.0, (E, n))
        env.step(torch.as_tensor(a.astype(np.uint8)).cuda(), auto_reset=True,
                 negotiation=(torch.as_tensor(prop).cuda(), torch.as_tensor(acc).cuda(), dec))
        o = orc.step(a, want_features=False)
        done = o["done"].astype(bool)
        if done.any():
            exp.grid(orc, done, first, H)
            orc.reset(o["done"])
            old = orc.get_state()["theta"]
            orc.negotiate(prop, acc)
            orc.set_state(theta=np.where(done, orc.get_state()["theta"], old))
    got = log.drain()
    assert got["ended"].sum() > E and (~got["ended"]).sum() > 5
    exp.check(got, "%s %s" % (kind, form))
    _check_stats(stats, got["metrics"])
    assert log.drain()["env_id"].size == 0                  # drained


# ---- 2. feature envs ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["device", "host_async"])
@pytest.mark.parametrize("kind", ["cleanup", "harvest"])
def test_feature_log_matches_oracle(oracle_lib, kind, path):
    """next-step auto-reset and masked resets, one single-env oracle per env (a finished one is reset instead of stepped)"""
    import torch
    from contracts_b200.features import BatchedFeatureEnv
    E, n, H, first = 41, 4, 23, 5
    c = CONTRACT[kind]
    env = BatchedFeatureEnv(kind, E, n, horizon=H, contract=c, seed=99, first_env_id=first)
    orcs = [oracle_lib.FeatOracle(kind, 1, n, _maps(kind), horizon=H, contract=c, seed=99, first_env_id=first + i) for i in range(E)]
    log = _log(env, 1000)
    exp = Expected()
    env.reset()
    for o in orcs:
        o.reset()
    rng = np.random.default_rng(3)
    nact = 9 if kind == "cleanup" else 8
    done_prev = np.zeros(E, bool)
    res = env.new_host_result() if path == "host_async" else None
    a_host = torch.zeros((E, n), dtype=torch.uint8).pin_memory()
    for t in range(100):
        a = rng.integers(0, nact, size=(E, n))
        if t in (7, 52):
            m = (np.arange(E) % 3 == t % 3) & ~done_prev
            for i in np.nonzero(m)[0]:
                exp.grid(orcs[i], np.ones(1, bool), first + i, H)
                orcs[i].reset()
            env.reset(torch.as_tensor(m.astype(np.uint8)).cuda())
        if path == "device":
            env.step(torch.as_tensor(a.astype(np.uint8)).cuda(), auto_reset=True)
            done = env.done.cpu().numpy().astype(bool)
        else:
            a_host.numpy()[:] = a
            env.step_host_wait(env.step_host_async(a_host, res, auto_reset=True))
            done = res.done.astype(bool).copy()
        for i in range(E):
            if done_prev[i]:
                exp.grid(orcs[i], np.ones(1, bool), first + i, H)
                orcs[i].reset()
            else:
                orcs[i].step(a[i][None])
        done_prev = done
    exp.check(log.drain(), "%s %s" % (kind, path))


# ---- 3. selfdrive ----------------------------------------------------------------------------------------------------------
def test_selfdrive_log_matches_oracle(oracle_lib):
    import torch
    from contracts_b200.selfdrive import BatchedCarEnv
    E, n, first = 24, 3, 70
    env = BatchedCarEnv(E, n, contract="SelfdriveContractDistprop", seed=11, first_env_id=first)
    orcs = [oracle_lib.CarOracle(1, n, contract=True, seed=11, first_env_id=first + i) for i in range(E)]
    log = _log(env, 1000)
    exp = Expected()
    env.reset()
    for o in orcs:
        o.reset()
    rng = np.random.RandomState(2)
    done_prev = np.zeros(E, bool)

    def expect(i, ended):
        st = orcs[i].get_state()
        exp.add(first + i, orcs[i].episode[0], st["t"][0], ended, st["theta"][0], [st["transfers"][0]])

    for t in range(400):
        a = rng.uniform(-0.1, 0.1, (E, n)).astype(np.float32)
        if t in (30, 210):
            m = np.arange(E) % 4 == t % 4
            for i in np.nonzero(m)[0]:
                expect(i, done_prev[i])
                orcs[i].reset()
            env.reset(torch.as_tensor(m.astype(np.uint8)).cuda())
            done_prev[m] = False
        env.step(torch.as_tensor(a).cuda(), auto_reset=True)
        done = env.done[:, n].cpu().numpy().astype(bool)
        for i in range(E):
            if done_prev[i]:
                expect(i, True)
                orcs[i].reset()
            else:
                orcs[i].step(a[i][None])
        done_prev = done
    got = log.drain()
    assert got["ended"].sum() >= E and (~got["ended"]).sum() > 0
    exp.check(got, "selfdrive")


# ---- 4. the reference's episode metrics ------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["cleanup_n5_short_horizon", "harvest_n8_short_horizon"])
def test_golden_episode_metrics(name):
    import torch
    from contracts_b200.batched import BatchedGridEnv
    fx = gu.load(name)
    kind, n = str(fx["kind"]), int(fx["n"])
    env = BatchedGridEnv(kind + "_new", 1, n, [str(r) for r in fx["ascii_map"]], horizon=int(fx["horizon"]),
                         contract=gu.contract_name(fx), seed=int(fx["seed"]), first_env_id=int(fx["env_id"]), **gu.shaping_kwargs(fx))
    log = _log(env, 8)
    episodes, steps = fx["actions"].shape[:2]
    for ep in range(episodes):
        env.reset()
        for t in range(steps):
            env.step(torch.as_tensor(np.asarray(fx["actions"][ep, t]).astype(np.uint8)[None]).cuda())
    env.reset()                                             # the last episode is logged by one more reset
    got = log.drain()
    assert got["lost"] == 0 and list(got["episode"]) == list(range(episodes)) and (got["env_id"] == int(fx["env_id"])).all()
    keys = [str(k) for k in fx["metric_keys"]]
    dicts = log.metrics(got)
    for ep in range(episodes):
        want = dict(zip(keys, fx["metrics"][ep]))
        gu.check_episode_metrics(kind, n, bool(fx["contract"]), got["metrics"][ep], want, "%s ep %d" % (name, ep))
        assert sorted(dicts[ep]) == sorted(want), (ep, sorted(dicts[ep]), sorted(want))
        for k, v in want.items():
            gu.assert_same("metrics()[%s]" % k, np.float64(dicts[ep][k]), np.float64(v), "%s ep %d" % (name, ep))


# ---- 5. ring wrap ------------------------------------------------------------------------------------------------------------
def test_ring_wrap_counts_lost_records():
    import torch
    from contracts_b200.batched import BatchedGridEnv
    E, H = 20, 10
    envs = [BatchedGridEnv("cleanup_new", E, 3, horizon=H, seed=4, first_env_id=3) for _ in range(2)]
    small, big = _log(envs[0], 7), _log(envs[1], 1000)

    def run(steps):
        for s in range(steps):
            for env in envs:
                a = env.random_actions(s, 9)
                env.step(a, auto_reset=True)

    for env in envs:
        env.reset()
    run(25)                                                   # 40 records
    ref = big.drain()
    got = small.drain()
    assert got["lost"] == len(ref["env_id"]) - 7 and len(got["env_id"]) == 7
    sel = np.arange(E) < 7                                    # the newest 7: one masked reset of 7 envs
    run(5)                                                    # 20 more records: all overwritten by the 7
    ref = big.drain()
    for env in envs:
        env.reset(torch.as_tensor(sel.astype(np.uint8)).cuda())
    got, last = small.drain(), big.drain()
    assert len(ref["env_id"]) == E and got["lost"] == E and len(last["env_id"]) == 7
    for k in ("env_id", "episode", "t", "ended", "theta", "metrics"):
        gu.assert_same(k, got[k], last[k], "wrap")


# ---- 6. CUDA graph -----------------------------------------------------------------------------------------------------------
def test_graph_replay_matches_eager():
    import torch
    from contracts_b200.batched import BatchedGridEnv
    E, H = 64, 10
    eager, graphed = (BatchedGridEnv("cleanup_new", E, 4, horizon=H, contract="CleanupContract", seed=8, first_env_id=9)
                      for _ in range(2))
    logs = [_log(eager, 2000), _log(graphed, 2000)]
    acts = [torch.empty((E, 4), dtype=torch.uint8, device="cuda") for _ in range(2)]

    def substep(env, a):
        env.random_actions(None, 9, out=a)
        env.step(a, auto_reset=True)

    for env in (eager, graphed):
        env.reset()
    torch.cuda.synchronize()
    cap = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=cap):
        for _ in range(20):
            substep(graphed, acts[1])
    for r in range(5):
        g.replay()
        for _ in range(20):
            substep(eager, acts[0])
    torch.cuda.synchronize()
    want, got = logs[0].drain(), logs[1].drain()
    assert want["lost"] == got["lost"] == 0 and len(want["env_id"]) >= 5 * 20 * E // H - E
    for k in ("env_id", "episode", "t", "ended", "theta", "metrics"):
        gu.assert_same(k, got[k], want[k], "graph")


# ---- 7. resume -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["cleanup_new", "cleanup", "selfdrive"])
def test_resume_logs_the_same_episode(kind):
    import torch
    E, H = 8, 30

    def make():
        if kind == "cleanup_new":
            from contracts_b200.batched import BatchedGridEnv
            return BatchedGridEnv(kind, E, 3, horizon=H, contract="CleanupContract", seed=6, first_env_id=2)
        if kind == "cleanup":
            from contracts_b200.features import BatchedFeatureEnv
            return BatchedFeatureEnv(kind, E, 3, horizon=H, contract="CleanupContract", seed=6, first_env_id=2)
        from contracts_b200.selfdrive import BatchedCarEnv
        return BatchedCarEnv(E, 3, contract="SelfdriveContractDistprop", seed=6, first_env_id=2)

    def act(env, s):
        return env.random_actions(s, -0.1, 0.1) if kind == "selfdrive" else env.random_actions(s, 8)

    a, b = make(), make()
    la = _log(a)
    a.reset()
    b.reset()
    for s in range(12):
        a.step(act(a, s))
        b.step(act(b, s))
    ck = b.checkpoint()
    del b
    torch.cuda.synchronize()
    c = make()
    lc = _log(c)
    c.restore(ck)
    for s in range(12, 120 if kind == "selfdrive" else H):
        a.step(act(a, s))
        c.step(act(c, s))
    a.reset()
    c.reset()
    want, got = la.drain(), lc.drain()
    assert len(want["env_id"]) == E and len(got["env_id"]) == E      # only the episode the final reset ends
    for k in ("env_id", "episode", "t", "ended", "theta", "metrics"):
        gu.assert_same(k, got[k], want[k], "resume %s" % kind)


# ---- 8. full size, bench.py's steady state ----------------------------------------------------------------------------------------
def test_full_size_cleanup8_counts_and_sums():
    import torch
    import bench
    cfg = bench.CONFIGS["cleanup8"]
    E = cfg["envs"]
    run = bench.Runner("cleanup8", cfg, E, 0, torch.device("cuda", 0))
    log = _log(run.env)                                        # 2 E records: 1.2 horizons append 1.2 E
    run.burn_in()                                              # zeroes the stats vector at its end
    log.drain()
    steps = int(1.2 * bench.HORIZON)
    resets = 0
    for s in range(steps):
        if s % 50 == 0:
            run.policy()
        run.substep(bench.HORIZON + s)
        resets += int(run.env.done.sum().item())
    got = log.drain()
    assert got["lost"] == 0 and len(got["env_id"]) == resets and resets >= E
    assert got["ended"].all() and (got["t"] == bench.HORIZON).all()
    _check_stats(run.stats, got["metrics"])


@pytest.mark.parametrize("name", ["features1m", "selfdrive8"])
def test_full_size_next_step_reset_logs_the_done_envs(name):
    """the records appended by step k are the envs that were done after step k - 1"""
    import torch
    import bench
    cfg = bench.CONFIGS[name]
    E = cfg["envs"]
    run = bench.Runner(name, cfg, E, 0, torch.device("cuda", 0))
    log = _log(run.env, E)
    run.burn_in()
    run.substep(999)                                           # (the dones of a burn-in step belong to envs it reset itself)
    log.drain()
    first = run.env.first_env_id
    for s in range(6):
        done = run.done_mask().clone() if name == "selfdrive8" else run.env.done.clone()
        run.substep(1000 + s)
        got = log.drain()
        want = np.nonzero(done.cpu().numpy())[0] + first
        gu.assert_same("env_id step %d" % s, got["env_id"], want, name)
        assert got["ended"].all()


# ---- 9. error surface ---------------------------------------------------------------------------------------------------------
def test_error_surface_and_switch_off():
    import torch
    from contracts_b200 import _lib
    from contracts_b200.batched import BatchedGridEnv
    env = BatchedGridEnv("harvest_new", 4, 2, horizon=5)
    lib = env.lib
    rec = torch.zeros((8, 480), dtype=torch.uint8, device="cuda")
    cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
    size = ctypes.sizeof(_lib.ssd_episode_log)

    def rc(**kw):
        d = dict(struct_size=size, capacity=8, records_dev=rec.data_ptr(), count_dev=cnt.data_ptr())
        d.update(kw)
        return lib.ssd_set_episode_log(env._h, ctypes.byref(_lib.ssd_episode_log(**d)))

    assert lib.ssd_set_episode_log(None, None) == -1
    assert rc(struct_size=size - 1) == -1
    assert rc(capacity=0) == -1 and rc(capacity=-3) == -1
    assert rc(records_dev=None) == -1 and rc(records_dev=rec.data_ptr() + 8) == -1
    assert rc(count_dev=None) == -1 and rc(count_dev=cnt.data_ptr() + 4) == -1
    assert rc() == 0
    env.reset()
    env.reset()
    torch.cuda.synchronize()
    assert int(cnt[0].item()) == 4
    assert lib.ssd_set_episode_log(env._h, None) == 0          # off: nothing more is appended
    env.reset()
    for s in range(6):
        env.step(env.random_actions(s, 8), auto_reset=True)
    torch.cuda.synchronize()
    assert int(cnt[0].item()) == 4
    assert rc(capacity=0) == -1 and int(cnt[0].item()) == 4    # a rejected struct leaves the log off
    env.reset()
    torch.cuda.synchronize()
    assert int(cnt[0].item()) == 4


# ---- the vector adapters ------------------------------------------------------------------------------------------------------
def test_vector_env_episode_metrics():
    """episode_metrics(): one dict per finished episode, as the drop-in class's metrics at its last step, + env_id / episode"""
    from contracts_b200.vector_env import SSDVectorEnv
    E, H = 4, 5
    vec = SSDVectorEnv("harvest_new", E, 2, contract="HarvestFeaturemodLocalContract", horizon=H, first_env_id=10)
    assert vec.episode_metrics() == []
    for _ in range(H):
        vec.send_action_array(np.full((E, 2), 4, np.uint8))
        s = vec.poll_arrays()
    assert s["done"].all()
    for e in range(E):
        vec.try_reset(e)
    vec.poll_arrays()
    ms = vec.episode_metrics()
    assert [(m["env_id"], m["episode"]) for m in ms] == [(10 + e, 0) for e in range(E)]
    for m in ms:
        assert {"equality", "sustainability", "transfer_equality", "transfer_sustainability", "transfers"} <= set(m)
    assert vec.episode_metrics() == []
    vec.stop()

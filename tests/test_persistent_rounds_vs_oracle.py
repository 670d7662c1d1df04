"""GPU: the feature-env and selfdrive step kernels (feat_kernel, car_kernel) against the C oracle across the rounds of their
persistent grids, and the solver queue across its blocks of SQ_BLOCK envs.

A persistent CTA takes env group after env group (`grp += gridDim.x`): at the benchmark's 131072 envs every CTA serves
several rounds, and a round inherits the shared-memory state of the env its octet served in the previous one.  G, the
envs one round serves (grid x envs per CTA), is read from the line SSD_DEBUG prints at create, for the configuration
under test.  The oracle emulates the next-step auto-reset of a whole batch with its skip step
(golden_util.auto_reset_step), so every env of every round is compared bit for bit after every step: observations (and
the policy's flat rows in every dtype, converted from the oracle's float64 rows by torch), rewards, transfers, infos,
dones, state, metrics, episode-log records and the pipelined host path's result block.
(Named to sort after test_cuda_kernel_variants.py, whose profiler records must not see this file's kernels.)"""
import re

import numpy as np
import pytest
import torch

import golden_util as gu
from test_cuda_flat_policy_step import flat_rows
from test_cuda_solver_queue import S as SAMPLES, _old_route, _theta_t, value_fn

pytestmark = pytest.mark.gpu

SEED = 73907                                  # bench.py
FULL_E = 131072                               # bench.py's envs per GPU for features1m / harvestfeat1m / selfdrive8
CONTRACT = {"cleanup": "CleanupContract", "harvest": "HarvestFeaturemodLocalContract", "selfdrive": "SelfdriveContractDistprop"}
NACT = {"cleanup": 8, "harvest": 7}           # bench.py's random actions
BENCH = {"features1m": ("cleanup", 8), "harvestfeat1m": ("harvest", 8), "selfdrive8": ("selfdrive", 8)}
ALL_FORMS = (None, torch.float32, torch.float16, torch.bfloat16)
SHORT_TRACK = dict(low_bound=-1.0, high_bound=1.0)        # selfdrive episodes of ~5-40 steps


def _maps(kind):
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    return CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP


def _make(kind, E, n, horizon, dtype=None, first=0, **kw):
    if kind == "selfdrive":
        from contracts_b200.selfdrive import BatchedCarEnv
        return BatchedCarEnv(E, n, contract=CONTRACT[kind], seed=SEED, first_env_id=first, policy_dtype=dtype, **kw)
    from contracts_b200.features import BatchedFeatureEnv
    return BatchedFeatureEnv(kind, E, n, horizon=horizon, contract=CONTRACT[kind], seed=SEED, first_env_id=first,
                             policy_dtype=dtype)


def _oracle(oracle_lib, kind, E, n, horizon, first=0, **kw):
    if kind == "selfdrive":
        return oracle_lib.CarOracle(E, n, contract=True, seed=SEED, first_env_id=first, **kw)
    return oracle_lib.FeatOracle(kind, E, n, _maps(kind), horizon=horizon, contract=CONTRACT[kind], seed=SEED, first_env_id=first)


# ---- the persistent grid ----------------------------------------------------------------------------------------------
_G = {}
_GRID_LINE = re.compile(r"\[ssd\] (?:feature|selfdrive) kernel: (\d+) CTAs/SM, \d+ B smem/CTA, grid (\d+), (\d+) envs/round")


def envs_per_round(capfd, monkeypatch, kind, n, **kw):
    """G of the step kernel's persistent grid for (kind, n): SSD_DEBUG prints it when a handle is created"""
    key = (kind, n) + tuple(sorted(kw.items()))
    if key not in _G:
        monkeypatch.setenv("SSD_DEBUG", "1")
        capfd.readouterr()
        probe = _make(kind, FULL_E, n, 24, **kw)
        err = capfd.readouterr().err
        probe.close()
        monkeypatch.delenv("SSD_DEBUG")
        m = _GRID_LINE.search(err)
        assert m, "SSD_DEBUG printed no %s grid: %r" % (kind, err)
        G = int(m.group(3))
        assert G < FULL_E, "the probe batch does not fill the persistent grid"
        print("[persistent grid] %s n=%d: %s CTAs/SM, grid %s, G = %d envs/round" % (kind, n, m.group(1), m.group(2), G))
        _G[key] = G
    return _G[key]


# ---- bit-exact comparison on the device ---------------------------------------------------------------------------------
def _same(name, got, want, ctx, rows_per_env=1):
    """got (device tensor) against want (numpy or tensor): floating values by bit pattern, integers by value; names the
    first differing envs"""
    if isinstance(want, np.ndarray):
        want = torch.from_numpy(np.ascontiguousarray(want))
    want = want.to(got.device)
    assert tuple(got.shape) == tuple(want.shape), "%s shape %r != %r at %s" % (name, tuple(got.shape), tuple(want.shape), ctx)
    if got.dtype.is_floating_point or want.dtype.is_floating_point:
        assert got.dtype == want.dtype, "%s dtype %s != %s" % (name, got.dtype, want.dtype)
        g, w = got.contiguous().view(torch.uint8), want.contiguous().view(torch.uint8)
    else:
        g, w = got.to(torch.int64), want.to(torch.int64)
    rows = got.shape[0] // rows_per_env
    bad = (g != w).reshape(rows, -1).any(1).nonzero().flatten()
    assert bad.numel() == 0, "%s differs from the oracle at %s in %d envs, first %r" % (name, ctx, bad.numel(), bad[:10].tolist())


class Records:
    """the episode-log records the oracle's batch would append: one per env whose episode a reset replaces"""

    def __init__(self, first, horizon):
        self.first, self.horizon, self.parts = first, horizon, []

    def before_reset(self, orc, mask, ended_car=None):
        """orc is about to reset the envs of mask (bool [E]); ended_car: selfdrive's all-done flags (bool [E])"""
        sel = mask & (orc.episode >= 0)
        if not sel.any():
            return
        idx = np.nonzero(sel)[0]
        st = orc.get_state()
        m = np.zeros((idx.size, 56))
        if ended_car is not None:
            m[:, 0] = st["transfers"][idx]
            ended = ended_car[idx]
        else:
            m[:, :40] = orc.metrics_raw()[idx]
            ended = st["t"][idx] == self.horizon
        self.parts.append((self.first + idx, orc.episode[idx], st["t"][idx], ended, st["theta"][idx], m))

    def check(self, got, ctx):
        assert got["lost"] == 0, ctx
        cols = [np.concatenate([p[k] for p in self.parts]) for k in range(6)] if self.parts else [np.zeros(0)] * 5 + [np.zeros((0, 56))]
        order = np.lexsort((cols[1], cols[0]))
        assert len(got["env_id"]) == order.size, "%s: %d records, want %d" % (ctx, len(got["env_id"]), order.size)
        for name, k in (("env_id", 0), ("episode", 1), ("t", 2), ("ended", 3)):
            gu.assert_same("record " + name, got[name].astype(np.int64), cols[k][order].astype(np.int64), ctx)
        gu.assert_same("record theta", got["theta"], cols[4][order], ctx)
        gu.assert_same("record metrics", got["metrics"], cols[5][order], ctx)
        return order.size


class Rollout:
    """One oracle of all E envs and CUDA batches of the same configuration, one per observation form (float64 first, with
    an episode log), driven with the same calls and compared with the oracle after each.  step(auto_reset=True) is
    emulated on the oracle by reset(done_prev) + step(skip=done_prev)."""

    def __init__(self, oracle_lib, kind, n, E, horizon, forms=(None,), first=0, log_capacity=0, **kw):
        from contracts_b200.episodes import EpisodeLog
        self.kind, self.n, self.E, self.horizon, self.forms, self.first = kind, n, E, horizon, forms, first
        self.car = kind == "selfdrive"
        self.envs = [_make(kind, E, n, horizon, dtype=f, first=first, **kw) for f in forms]
        self.orc = _oracle(oracle_lib, kind, E, n, horizon, first=first, **kw)
        self.done_prev = np.zeros(E, bool)
        self.restarts = np.zeros(E, np.int64)
        self.log, self.records = None, Records(first, horizon)
        if log_capacity:
            self.log = EpisodeLog(self.envs[0], log_capacity)
            self.envs[0].set_episode_log(self.log)

    def actions(self, t):
        env = self.envs[0]
        a = env.random_actions(t, -0.1, 0.1) if self.car else env.random_actions(t, NACT[self.kind])
        return a, a.cpu().numpy()

    def check_obs(self, want, ctx):
        """want: the oracle's float64 observation [E, n, D] (numpy)"""
        want = torch.from_numpy(want).cuda()
        theta = torch.from_numpy(self.orc.get_state()["theta"]).cuda()
        for f, env in zip(self.forms, self.envs):
            if f is None:
                _same("obs", env.obs, want, ctx)
            else:
                assert env.obs is None
                _same("policy rows", env.policy_obs, flat_rows(want, theta, True, f), "%s %s" % (f, ctx), rows_per_env=self.n)

    def check_outputs(self, o, ctx):
        w = {k: torch.from_numpy(np.ascontiguousarray(o[k])).cuda() for k in ("rew", "base_rew", "transfers", "info", "done")}
        for f, env in zip(self.forms, self.envs):
            c = "%s %s" % (f, ctx)
            _same("rew", env.rew, w["rew"], c)
            _same("base_rew", env.base_rew, w["base_rew"], c)
            _same("transfers", env.transfers, w["transfers"], c)
            _same("info", env.info if self.car else env.info[..., :2], w["info"] if self.car else w["info"][..., :2], c)
            _same("done", env.done, w["done"], c)
        self.check_obs(o["obs"], ctx)

    def check_state(self, ctx):
        so = self.orc.get_state()
        keys = ("pos", "vel", "theta", "transfers", "t") if self.car else ("pos", "ori", "cells", "theta", "t")
        for f, env in zip(self.forms, self.envs):
            sc = env.get_state()
            for k in keys:
                _same(k, sc[k], so[k], "%s %s" % (f, ctx))

    def reset(self, mask=None, ctx="reset"):
        m = np.ones(self.E, bool) if mask is None else np.asarray(mask, bool)
        self.records.before_reset(self.orc, m, self.done_prev if self.car else None)
        r = self.orc.reset(None if mask is None else m.astype(np.uint8))
        md = None if mask is None else torch.as_tensor(m.astype(np.uint8)).cuda()
        for env in self.envs:
            env.reset(md)
        if mask is None:
            want = r
        else:                                        # the untouched envs keep the observation of the last step
            want = self.last_obs.copy()
            want[m] = r[m]
        self.done_prev[m] = False                    # a reset clears a pending restart
        self.last_obs = want
        self.check_obs(want, ctx)
        self.check_state(ctx)

    def step(self, t, ctx, auto_reset=True, state=True):
        a_dev, a = self.actions(t)
        for env in self.envs:
            env.step(a_dev, auto_reset=auto_reset)
        if auto_reset:
            self.records.before_reset(self.orc, self.done_prev, self.done_prev if self.car else None)
            o = gu.auto_reset_step(self.orc, a, self.done_prev)
            self.restarts += self.done_prev
        else:
            o = self.orc.step(a)
        self.last_obs = o["obs"]
        self.check_outputs(o, ctx)
        if state:
            self.check_state(ctx)
        self.done_prev = (o["done"][:, self.n] if self.car else o["done"]).astype(bool)
        return o

    def finish(self, ctx="end"):
        self.check_state(ctx)
        if not self.car:
            want = torch.from_numpy(self.orc.metrics_raw()).cuda()
            for f, env in zip(self.forms, self.envs):
                _same("metrics", env.metrics_raw(), want, "%s %s" % (f, ctx))
        if self.log is not None:
            return self.records.check(self.log.drain(), "episode log " + ctx)
        return 0

    def close(self):
        for env in self.envs:
            env.close()


# ---- 1. full size, steady state, every observation form, episode log ------------------------------------------------
FULL_H = 24


@pytest.mark.parametrize("name", list(BENCH))
def test_full_size_steady_state_matches_oracle(oracle_lib, capfd, monkeypatch, name):
    """bench.py's configuration (131072 envs, n = 8, its contract and random actions), a short horizon staggered with
    bench's phase resets (feature envs) or masked resets (selfdrive), then auto-reset steps until every env has restarted;
    float64 and float32 / float16 / bfloat16 policy rows; the float64 batch logs every episode"""
    kind, n = BENCH[name]
    G = envs_per_round(capfd, monkeypatch, kind, n)
    E = FULL_E
    assert E >= 2 * G, "the batch no longer spans two rounds of the persistent grid (G = %d)" % G
    r = Rollout(oracle_lib, kind, n, E, FULL_H, forms=ALL_FORMS, log_capacity=5 * E)
    r.reset()
    if kind == "selfdrive":
        steps = 0
        while not (r.restarts > 0).all():
            assert steps < 500, "%d envs never restarted" % int((r.restarts == 0).sum())
            r.step(steps, "%s step %d" % (name, steps), state=steps % 8 == 0)
            if steps < 32:                             # desynchronise a quarter of the episodes
                r.reset(np.arange(E) % 128 == steps, "%s masked reset %d" % (name, steps))
            steps += 1
    else:
        phase = np.arange(E) % FULL_H
        for s in range(FULL_H):                        # bench.py's burn-in: env i restarts at step i mod horizon
            r.step(s, "%s burn-in step %d" % (name, s), auto_reset=False, state=s % 6 == 0)
            r.reset(phase == s, "%s burn-in reset %d" % (name, s))
        steps = FULL_H + 2
        for s in range(steps):
            r.step(FULL_H + s, "%s auto-reset step %d" % (name, s), state=s % 4 == 0)
        assert (r.restarts > 0).all()
    records = r.finish(name)
    print("[%s] E = %d, G = %d: %d rounds, %d steps, %d restarts, %d log records" %
          (name, E, G, -(-E // G), steps, int(r.restarts.sum()), records))
    r.close()


# ---- 2. ragged sizes around the grid --------------------------------------------------------------------------------------
RAGGED = {"cleanup_n5": ("cleanup", 5, {}), "harvest_n8": ("harvest", 8, {}), "selfdrive_n3": ("selfdrive", 3, SHORT_TRACK)}
SIZES = {"G-1": lambda G: G - 1, "G": lambda G: G, "G+1": lambda G: G + 1, "2G+1": lambda G: 2 * G + 1, "3G+17": lambda G: 3 * G + 17}
RAGGED_H = 8


def _round_masks(E, G):
    """masked resets: only the last (partial) round, one env per round, no env at all"""
    rounds = -(-E // G)
    last = np.arange(E) >= (rounds - 1) * G
    one = np.zeros(E, bool)
    for k in range(rounds):
        one[k * G + (37 * k + 5) % min(G, E - k * G)] = True
    return [("last round", last), ("one env per round", one), ("no env", np.zeros(E, bool))]


@pytest.mark.parametrize("size", list(SIZES))
@pytest.mark.parametrize("config", list(RAGGED))
def test_ragged_sizes_match_oracle(oracle_lib, capfd, monkeypatch, config, size):
    """E at and around multiples of G: partly filled last env groups (and, at G - 1, a last warp with three envs); about
    20 auto-reset steps with staggered episodes and masked resets that hit the last round, one env per round, or none"""
    kind, n, kw = RAGGED[config]
    G = envs_per_round(capfd, monkeypatch, kind, n, **kw)
    E = SIZES[size](G)
    r = Rollout(oracle_lib, kind, n, E, RAGGED_H, forms=(None, torch.bfloat16), first=3, log_capacity=8 * E, **kw)
    r.reset()
    if kind != "selfdrive":                            # env e finishes in step e mod H of the auto-reset steps
        phase = np.arange(E) % RAGGED_H
        for s in range(RAGGED_H):
            r.step(s, "E %d burn-in step %d" % (E, s), auto_reset=False, state=False)
            r.reset(phase == s, "E %d burn-in reset %d" % (E, s))
    masks = dict(zip((5, 9, 13), _round_masks(E, G)))
    for s in range(20):
        r.step(100 + s, "E %d auto-reset step %d" % (E, s))
        if s in masks:
            what, m = masks[s]
            r.reset(m, "E %d masked reset (%s) after step %d" % (E, what, s))
    assert r.restarts.sum() > 0
    r.finish("E %d" % E)
    r.close()


# ---- 3. the pipelined host path at full size ------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["cleanup", "selfdrive"])
def test_full_size_host_path_matches_oracle(oracle_lib, capfd, monkeypatch, kind):
    """step_host_async / step_host_wait with auto-reset: the expanded rewards and the dones equal the oracle's.  For the
    feature env the copied record prefix (the recent maximum + 25 % + 1024) is too short at least once, so the wait
    fetches the rest."""
    n, H = 8, 12
    G = envs_per_round(capfd, monkeypatch, kind, n)
    E = FULL_E
    assert E >= 2 * G
    env = _make(kind, E, n, H)
    orc = _oracle(oracle_lib, kind, E, n, H)
    env.reset()
    orc.reset()
    car = kind == "selfdrive"
    if not car:                                        # staggered episodes (bench.py's burn-in)
        phase = np.arange(E) % H
        for s in range(H):
            a = env.random_actions(s, NACT[kind])
            env.step(a)
            orc.step(a.cpu().numpy())
            m = phase == s
            env.reset(torch.as_tensor(m.astype(np.uint8)).cuda())
            orc.reset(m.astype(np.uint8))
    cap = env.host_result_layout().record_capacity
    res = [env.new_host_result(), env.new_host_result()]
    recent, misses, records = [0, 0], 0, 0
    done_prev = np.zeros(E, bool)
    steps = 2 * H if not car else 150
    for s in range(steps):
        a = (env.random_actions(100 + s, -0.1, 0.1) if car else env.random_actions(100 + s, NACT[kind])).cpu().pin_memory()
        prefix = min(max(recent) + max(recent) // 4 + 1024, cap)
        tk = env.step_host_async(a, res[s & 1], auto_reset=True)
        env.step_host_wait(tk)
        r = res[s & 1]
        o = gu.auto_reset_step(orc, a.numpy(), done_prev)
        ctx = "%s host step %d" % (kind, s)
        gu.assert_same("host rewards", r.rewards(), o["rew"], ctx)
        gu.assert_same("host done", r.done, o["done"], ctx)
        misses += r.count > prefix
        records += r.count
        recent[tk & 1] = r.count
        done_prev = (o["done"][:, n] if car else o["done"]).astype(bool)
    print("[host path %s] E = %d, G = %d: %d rounds, %d steps, %d records, %d prefix misses" %
          (kind, E, G, -(-E // G), steps, records, misses))
    if not car:
        assert misses >= 1, "the copied record prefix was never too short: the fetch of the rest did not run"
    env.close()


# ---- 4. the solver queue across blocks of SQ_BLOCK envs ---------------------------------------------------------------------
SQ_BLOCK = 1024


def _check_window(q, out, pending, start, oracle_lib, env, ctx):
    """the window after `start` envs of nonzero(pending) were resolved: the next C of them in env order"""
    want = torch.nonzero(pending).flatten()[start:]
    cnt, total = [int(x) for x in q.count.tolist()]
    assert (cnt, total) == (min(want.numel(), q.C), want.numel()), "%s: counts %r, want %r" % (ctx, (cnt, total), (min(want.numel(), q.C), want.numel()))
    got = q.env[:cnt].long()
    bad = (got != want[:cnt]).nonzero().flatten()
    assert bad.numel() == 0, "%s: window slots %r hold envs %r, want %r" % (ctx, bad[:5].tolist(), got[bad[:5]].tolist(), want[bad[:5]].tolist())
    assert bool((q.env[cnt:] == -1).all()), ctx + ": slots past the window"
    assert not bool(out[0][cnt:].view(torch.uint8).any()), ctx + ": rows past the window"
    return cnt


def _check_entries(q, vals, theta, index, env, oracle_lib, cnt, ctx):
    """window entries against the oracle's solver_candidates / solver_choose: the first and last of the window and every
    entry from the last block"""
    if cnt == 0:
        return
    ids = q.env[:cnt].cpu().numpy()
    last_block = (env.E - 1) // SQ_BLOCK
    sample = sorted({0, cnt - 1} | set(np.nonzero(ids // SQ_BLOCK == last_block)[0].tolist()))
    ep = q.episode[:cnt].cpu().numpy().view(np.uint32)
    params, v, th, ix = q.params.cpu().numpy(), vals.cpu().numpy(), theta.cpu().numpy(), index.cpu().numpy()
    high = float(np.float32(0.2)) if env.kind == "cleanup" else float(np.float32(100.0))
    for c in sample:
        want = oracle_lib.solver_candidates(env.seed, env.first_env_id + int(ids[c]), int(ep[c]), 0.0, high, q.S)
        gu.assert_same("candidates", params[c], want, "%s entry %d (env %d)" % (ctx, c, ids[c]))
        wt, wi = oracle_lib.solver_choose(want, v[c], q.rule)
        gu.assert_same("chosen theta", th[c], wt, "%s entry %d (env %d)" % (ctx, c, ids[c]))
        assert int(ix[c]) == int(wi), "%s entry %d (env %d): index %d, want %d" % (ctx, c, ids[c], ix[c], wi)


def _drain(q, A, oracle_lib, ctx, entries=True):
    """rows / resolve window after window until no env is pending, each window checked; returns the envs resolved"""
    pending = _theta_t(A)[1] == 0
    start, windows = 0, 0
    while True:
        out = q.rows()
        cnt = _check_window(q, out, pending, start, oracle_lib, A, "%s window %d" % (ctx, windows))
        vals = value_fn(out[0])
        theta, index = q.resolve(vals)
        assert int(q.stale.item()) == 0, ctx
        if entries:
            _check_entries(q, vals, theta, index, A, oracle_lib, cnt, "%s window %d" % (ctx, windows))
        start += cnt
        windows += 1
        if cnt == 0 or int(q.count[1]) <= cnt:
            break
    assert start == int(pending.sum()) and q.pending() == 0, ctx
    return pending, windows


def test_solver_queue_across_blocks(oracle_lib):
    """cleanup features at 131072 envs in bench.py's staggered steady state (horizon 24: ~E / 24 envs restart per step),
    a window of C = 3001 envs (not a multiple of SQ_BLOCK): windows that end inside a block, later blocks that return
    early; every env's theta equals the all-env route's (a twin batch)"""
    from contracts_b200.solver import SolverQueue
    E, n, H, C = FULL_E, 8, FULL_H, 3001
    A, B = _make("cleanup", E, n, H), _make("cleanup", E, n, H)
    q = SolverQueue(A, num_samples=SAMPLES, capacity=C)
    A.reset()
    B.reset()
    pend, windows = _drain(q, A, oracle_lib, "full reset")
    assert windows == -(-E // C)
    _old_route(B, pend)
    _same("theta after the full reset", _theta_t(A)[0], _theta_t(B)[0], "full reset")
    phase = torch.arange(E, device="cuda") % H
    for s in range(H):                                 # bench.py's burn-in (no solver: both keep the reset's draw)
        a = A.random_actions(s, NACT["cleanup"])
        for env in (A, B):
            env.step(a)
            env.reset((phase == s).to(torch.uint8))
    for s in range(H // 2 + 1):
        a = A.random_actions(H + s, NACT["cleanup"])
        A.step(a, auto_reset=True)
        B.step(a, auto_reset=True)
        pend, windows = _drain(q, A, oracle_lib, "steady step %d" % s)
        if s == 0:                                     # the envs that reach the horizon here restart in the next step
            assert int(pend.sum()) == 0, "steady step 0: %d pending" % int(pend.sum())
        else:                                          # ~E / H restarts per step: more than one window
            assert int(pend.sum()) > C and windows >= 2, "steady step %d: %d pending" % (s, int(pend.sum()))
        _old_route(B, pend)
        _same("theta", _theta_t(A)[0], _theta_t(B)[0], "steady step %d" % s)
        _same("obs", A.obs, B.obs, "steady step %d" % s)
    A.close()
    B.close()


def test_solver_queue_above_a_million_envs():
    """selfdrive n = 3 at 2^20 + 37 envs (1025 blocks: block 0's sum over the block counts takes two strides), after a
    full reset, windows of C = 262147: the window order and the all-env route's theta"""
    from contracts_b200.solver import SolverQueue
    E, n, C = (1 << 20) + 37, 3, 262147
    A, B = _make("selfdrive", E, n, 0), _make("selfdrive", E, n, 0)
    q = SolverQueue(A, num_samples=SAMPLES, capacity=C)
    A.reset()
    B.reset()
    pend, windows = _drain(q, A, None, "full reset", entries=False)
    assert int(pend.sum()) == E and windows == -(-E // C)
    _old_route(B, pend)
    _same("theta", _theta_t(A)[0], _theta_t(B)[0], "full reset")
    A.close()
    B.close()

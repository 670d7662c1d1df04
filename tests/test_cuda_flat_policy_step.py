"""GPU: the feature-env and selfdrive steps writing the policy's flat input rows directly (BatchedFeatureEnv /
BatchedCarEnv(policy_dtype=T), ssd_set_flat_policy_output).

An env in policy mode must hold, after every call, exactly `torch.cat((obs, theta, 0), -1).to(float32).to(T)` of the
float64 rows of a twin env (same configuration and seed) that took the same calls (the features alone without a
contract), and every other output must equal the twin's."""
import ctypes

import numpy as np
import pytest

import golden_util as gu

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

DTYPES = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}
CONTRACT = {"cleanup": "CleanupContract", "harvest": "HarvestFeaturemodLocalContract", "selfdrive": "SelfdriveContractDistprop"}
KINDS = ("cleanup", "harvest", "selfdrive")


def _make(kind, E, n, dtype, contract=True, horizon=12, seed=11, first_env_id=5):
    c = CONTRACT[kind] if contract else None
    if kind == "selfdrive":
        from contracts_b200.selfdrive import BatchedCarEnv
        return BatchedCarEnv(E, n, contract=c, seed=seed, first_env_id=first_env_id, policy_dtype=dtype)
    from contracts_b200.features import BatchedFeatureEnv
    return BatchedFeatureEnv(kind, E, n, horizon=horizon, contract=c, seed=seed, first_env_id=first_env_id, policy_dtype=dtype)


def flat_rows(obs, theta, contract, dtype):
    """the policy's rows of float64 rows [E, n, F] and theta [E]: (features ++ [theta, 0]).to(float32).to(dtype)"""
    E, n, F = obs.shape
    x = obs.reshape(E * n, F)
    if contract:
        th = theta.to(x.device, torch.float64).repeat_interleave(n).unsqueeze(1)
        x = torch.cat((x, th, torch.zeros_like(th)), -1)
    return x.to(torch.float32).to(dtype)


class Twins:
    """a float64 env and a policy-mode env of the same configuration, driven with the same calls"""

    def __init__(self, kind, E, n, dtype, contract=True, **kw):
        from contracts_b200.episodes import EpisodeLog
        self.u, self.q = _make(kind, E, n, None, contract, **kw), _make(kind, E, n, dtype, contract, **kw)
        self.kind, self.E, self.n, self.dtype, self.contract = kind, E, n, dtype, contract
        self.car = kind == "selfdrive"
        self.rng = np.random.RandomState(7)
        self.logs = [EpisodeLog(e, capacity=64 * E if E <= 4096 else 2 * E) for e in (self.u, self.q)]
        for e, log in zip((self.u, self.q), self.logs):
            e.set_episode_log(log)

    def check(self, ctx):
        torch.cuda.synchronize()
        assert self.q.obs is None
        want = flat_rows(self.u.obs, self.u.get_state()["theta"], self.contract, self.dtype)
        assert self.q.policy_obs.shape == (self.E * self.n, self.q.policy_width)
        if not torch.equal(self.q.policy_obs, want):
            bad = (self.q.policy_obs != want).nonzero()[:5].tolist()
            raise AssertionError("policy rows differ after %s at %r" % (ctx, bad))

    def same(self, ctx):
        for name in ("rew", "base_rew", "transfers", "info", "done"):
            assert torch.equal(getattr(self.u, name), getattr(self.q, name)), "%s differs after %s" % (name, ctx)
        su, sq = self.u.get_state(), self.q.get_state()
        for k in su:
            assert torch.equal(su[k], sq[k]), "state %s differs after %s" % (k, ctx)
        if not self.car:
            assert torch.equal(self.u.metrics_raw(), self.q.metrics_raw()), ctx

    def same_log(self):
        ru, rq = (log.drain() for log in self.logs)
        assert len(ru["env_id"]) > 0 and ru["lost"] == 0
        for k in ru:
            assert np.array_equal(ru[k], rq[k]), "episode log %s differs" % k

    def actions(self):
        if self.car:
            return torch.as_tensor(self.rng.uniform(-0.02, 0.1, size=(self.E, self.n)).astype(np.float32)).cuda()
        nact = 9 if self.kind == "cleanup" else 8
        return torch.as_tensor(self.rng.randint(0, nact, size=(self.E, self.n)).astype(np.uint8)).cuda()

    def host_actions(self):
        return self.actions().cpu().pin_memory()

    def both(self, fn):
        return fn(self.u), fn(self.q)


def _run_twins(tw):
    from contracts_b200.batched import negotiate, solver_choose, solver_sample
    E, n = tw.E, tw.n
    r_u, r_q = tw.both(lambda e: e.reset())
    assert r_q is tw.q.policy_obs
    tw.check("reset")
    for t in range(4):
        a = tw.actions()
        o_q = tw.both(lambda e: e.step(a))[1][0]
        assert o_q is tw.q.policy_obs
        tw.check("step %d" % t)
        tw.same("step %d" % t)
    finished = 0
    for t in range(90 if tw.car else 2 * tw.u.horizon + 2):   # every env finishes and restarts at least once
        a = tw.actions()
        tw.both(lambda e: e.step(a, auto_reset=True))
        finished += int((tw.u.done[:, -1] if tw.car else tw.u.done).sum())
        tw.check("auto-reset step %d" % t)
        tw.same("auto-reset step %d" % t)
    assert finished >= E
    mask = torch.as_tensor(tw.rng.randint(0, 2, E).astype(np.uint8)).cuda()
    tw.both(lambda e: e.reset(mask))
    tw.check("reset(mask)")
    theta = torch.as_tensor(tw.rng.uniform(0.0, 0.2, E)).cuda()
    tw.both(lambda e: e.set_contract_params(theta))
    tw.check("set_contract_params")
    prop = torch.as_tensor(tw.rng.uniform(0.0, 0.2, E)).cuda()
    acc = torch.as_tensor(tw.rng.uniform(0.0, 1.0, (E, n))).cuda()
    mask = torch.as_tensor(tw.rng.randint(0, 2, E).astype(np.uint8)).cuda()
    d_u, d_q = tw.both(lambda e: negotiate(e, prop, acc, mask))
    assert torch.equal(d_u, d_q)
    tw.check("negotiate(mask)")
    if tw.contract:
        params = solver_sample(tw.u, 3)
        assert torch.equal(params, solver_sample(tw.q, 3))
        vals = torch.as_tensor(tw.rng.uniform(size=(E, 4, n))).cuda()
        tw.both(lambda e: solver_choose(e, params, vals))
        tw.check("solver_choose")
    a = tw.actions()
    tw.both(lambda e: e.step(a))
    tw.check("step after the theta calls")
    tw.same("step after the theta calls")
    # checkpoint / restore / copy_envs
    ck_u, ck_q = tw.both(lambda e: e.checkpoint())
    assert ck_q.obs.dtype == tw.dtype and tuple(ck_q.obs.shape) == (E, n, tw.q.policy_width)
    assert torch.equal(ck_q.rows, ck_u.rows)
    with pytest.raises(ValueError, match="observation"):
        tw.q.restore(ck_u)
    for t in range(3):
        a = tw.actions()
        tw.both(lambda e: e.step(a, auto_reset=True))
    tw.u.restore(ck_u)
    tw.q.restore(ck_q)
    tw.check("restore")
    tw.same("restore")
    ck_rows = tw.u.checkpoint(with_obs=False)           # rows alone: the checkpoint's theta, the observation rows kept
    theta = torch.as_tensor(tw.rng.uniform(0.0, 0.2, E)).cuda()
    tw.both(lambda e: e.set_contract_params(theta))
    tw.both(lambda e: e.restore(ck_rows))
    tw.check("restore(with_obs=False)")
    a = tw.actions()
    tw.both(lambda e: e.step(a))
    tw.check("step after restore")
    tw.same("step after restore")
    src = torch.as_tensor(tw.rng.randint(0, E, E // 2)).cuda()
    dst = torch.as_tensor(tw.rng.permutation(E)[:E // 2]).cuda()
    tw.both(lambda e: e.copy_envs(src, dst))
    tw.check("copy_envs")
    a = tw.actions()
    tw.both(lambda e: e.step(a))
    tw.check("step after copy_envs")
    tw.same("step after copy_envs")
    # the pipelined host path with auto-reset
    res = [e.new_host_result() for e in (tw.u, tw.q)]
    for t in range(4):
        a_host = tw.host_actions()
        tk = [e.step_host_async(a_host, r, auto_reset=True) for e, r in zip((tw.u, tw.q), res)]
        for e, k in zip((tw.u, tw.q), tk):
            e.step_host_wait(k)
        tw.check("step_host_async %d" % t)
        assert np.array_equal(res[0].rewards(), res[1].rewards()) and np.array_equal(res[0].done, res[1].done)
    tw.same_log()


CASES = [(kind, n, contract) for kind in KINDS for n in range(1, 9) for contract in (True, False)
         if contract is False or kind == "selfdrive" or n >= 2]


@pytest.mark.parametrize("dt", sorted(DTYPES))
@pytest.mark.parametrize("kind,n,contract", CASES, ids=["%s-n%d-%s" % (k, n, "contract" if c else "plain") for k, n, c in CASES])
def test_policy_rows_twin(kind, n, contract, dt):
    """every row alignment: n = 1..8 at an odd batch size, with (W = F + 2) and without (W = F) a contract"""
    _run_twins(Twins(kind, 37, n, DTYPES[dt], contract))


@pytest.mark.parametrize("dt", ["f32", "bf16"])
@pytest.mark.parametrize("kind", KINDS)
def test_policy_rows_benchmark_size(kind, dt):
    """E = 131072, n = 8 (bench.py's features1m / harvestfeat1m / selfdrive8): auto-reset steps, the theta calls"""
    from contracts_b200.batched import negotiate
    E, n = 131072, 8
    tw = Twins(kind, E, n, DTYPES[dt], horizon=6, seed=73907, first_env_id=0)
    tw.both(lambda e: e.reset())
    tw.check("reset")
    for t in range(8):
        a = tw.actions()
        tw.both(lambda e: e.step(a, extras=False, auto_reset=True))
        tw.check("step %d" % t)
        for name in ("rew", "done"):
            assert torch.equal(getattr(tw.u, name), getattr(tw.q, name)), name
    theta = torch.as_tensor(tw.rng.uniform(0.0, 0.2, E)).cuda()
    tw.both(lambda e: e.set_contract_params(theta))
    tw.check("set_contract_params")
    mask = torch.as_tensor(tw.rng.randint(0, 2, E).astype(np.uint8)).cuda()
    tw.both(lambda e: negotiate(e, torch.full((E,), 0.1, dtype=torch.float64, device="cuda"),
                                torch.full((E, n), 0.8, dtype=torch.float64, device="cuda"), mask))
    tw.check("negotiate")
    tw.both(lambda e: e.reset(mask))
    tw.check("reset(mask)")


@pytest.mark.parametrize("dt", sorted(DTYPES))
@pytest.mark.parametrize("kind", KINDS)
def test_policy_rows_match_oracle(oracle_lib, kind, dt):
    """one rollout per kind against the C oracle: its float64 rows and theta, converted with torch"""
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    dtype = DTYPES[dt]
    if kind == "selfdrive":
        E, n, steps = 130, 3, 150
        orc = oracle_lib.CarOracle(E, n, contract=True, seed=7, first_env_id=123)
    else:
        E, n, steps = 67, 5, 120
        orc = oracle_lib.FeatOracle(kind, E, n, CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP, horizon=1000,
                                    contract=CONTRACT[kind], seed=4242, first_env_id=1000)
    env = _make(kind, E, n, dtype, horizon=1000, seed=7 if kind == "selfdrive" else 4242,
                first_env_id=123 if kind == "selfdrive" else 1000)

    def want(obs):
        return flat_rows(torch.from_numpy(np.ascontiguousarray(obs)), torch.from_numpy(orc.get_state()["theta"]), True, dtype)
    assert torch.equal(env.reset().cpu(), want(orc.reset())), "reset"
    rng = np.random.RandomState(n)
    for t in range(steps):
        if kind == "selfdrive":
            a = (rng.uniform(-0.7, 1.0, size=(E, n)) * 0.15).astype(np.float32)
        else:
            a = rng.randint(0, 9 if kind == "cleanup" else 8, size=(E, n)).astype(np.uint8)
        o = orc.step(a)
        obs, rew, done, _ = env.step(torch.from_numpy(a).cuda())
        ctx = "%s step %d" % (kind, t)
        assert torch.equal(obs.cpu(), want(o["obs"])), ctx
        gu.assert_same("rew", rew.cpu().numpy(), o["rew"], ctx)
        if t % 25 == 24:
            m = (rng.random_sample(E) < 0.33).astype(np.uint8)
            r_orc = orc.reset(m)
            sel = torch.from_numpy(np.repeat(m.astype(bool), n))
            got = env.reset(torch.from_numpy(m).cuda()).cpu()
            assert torch.equal(got[sel], want(r_orc)[sel]), ctx + " masked reset"


@pytest.mark.parametrize("kind", KINDS)
def test_policy_rows_graph_replay_matches_eager(kind):
    """a captured 50-step CUDA graph in policy mode (device-side action counter, auto-reset) replays to what the same
    steps make uncaptured"""
    E, n = 4096, 8
    eager, graphed = (_make(kind, E, n, torch.bfloat16, horizon=30) for _ in range(2))
    actions = {id(e): torch.empty((E, n), dtype=torch.float32 if kind == "selfdrive" else torch.uint8, device="cuda")
               for e in (eager, graphed)}

    def substep(env):
        if kind == "selfdrive":
            a = env.random_actions(None, -0.02, 0.1, out=actions[id(env)])
        else:
            a = env.random_actions(None, 9 if kind == "cleanup" else 8, out=actions[id(env)])
        env.step(a, extras=False, auto_reset=True)
    for env in (eager, graphed):
        env.reset()
    cap = torch.cuda.Stream()
    cap.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(cap):
        for _ in range(3):
            substep(graphed)
    torch.cuda.current_stream().wait_stream(cap)
    for _ in range(3):
        substep(eager)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=cap):
        for _ in range(50):
            substep(graphed)
    for r in range(2):
        g.replay()
        for _ in range(50):
            substep(eager)
        torch.cuda.synchronize()
        assert torch.equal(eager.policy_obs, graphed.policy_obs), "replay %d" % r
        assert torch.equal(eager.rew, graphed.rew) and torch.equal(eager.done, graphed.done), "replay %d" % r


def test_policy_kernel_instantiations_launch():
    """every policy-form instantiation (feat_kernel: 2 kinds x {step, reset} x 3 dtypes, car_kernel: {step, reset} x 3
    dtypes) runs, under the name torch.profiler shows"""
    from torch.profiler import ProfilerActivity, profile
    envs = [(_make(kind, 64, 4, dt), kind) for kind in KINDS for dt in DTYPES.values()]
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for env, kind in envs:
            env.reset()
            a = env.random_actions(0, -0.1, 0.1) if kind == "selfdrive" else env.random_actions(0, 8)
            env.step(a)
        torch.cuda.synchronize()
    names = {e.name for e in prof.events()}
    for form in (1, 2, 3):
        for reset in ("true", "false"):
            for cleanup in ("true", "false"):
                want = "feat_kernel<%s, %s, %d>" % (cleanup, reset, form)
                assert any(want in s for s in names), (want, sorted(s for s in names if "kernel<" in s))
            want = "car_kernel<%s, %d>" % (reset, form)
            assert any(want in s for s in names), (want, sorted(s for s in names if "kernel<" in s))


def test_flat_policy_output_error_surface():
    from contracts_b200 import _lib
    from contracts_b200.batched import negotiate
    E, n = 16, 4
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for kind in KINDS:
        q = _make(kind, E, n, torch.float16)
        u = _make(kind, E, n, None)
        lib = q.lib
        car = kind == "selfdrive"
        q.reset()
        rows0 = q.policy_obs.clone()
        stray = torch.zeros((E, n, q.F if not car else q.D), dtype=torch.float64, device="cuda")
        io = _lib.ssd_selfdrive_io() if car else _lib.ssd_feat_io()
        io.actions_dev = (torch.zeros((E, n), dtype=torch.float32, device="cuda") if car
                          else torch.ones((E, n), dtype=torch.uint8, device="cuda")).data_ptr()
        io.obs_dev, io.rew_dev, io.done_dev = stray.data_ptr(), q.rew.data_ptr(), q.done.data_ptr()
        step = lib.ssd_selfdrive_step if car else lib.ssd_feat_step
        reset = lib.ssd_selfdrive_reset if car else lib.ssd_feat_reset
        assert step(q._h, ctypes.byref(io), stream) == -1                      # one observation form per handle
        assert b"flat policy" in lib.ssd_last_error(q._h)
        assert reset(q._h, None, ctypes.c_void_p(stray.data_ptr()), stream) == -1
        res = q.new_host_result()
        a_host = torch.zeros((E, n), dtype=torch.float32 if car else torch.uint8).pin_memory()
        tk = ctypes.c_int64(-1)
        async_step = lib.ssd_selfdrive_step_host_async if car else lib.ssd_feat_step_host_async
        assert async_step(q._h, ctypes.byref(io), ctypes.c_void_p(a_host.data_ptr()), ctypes.c_void_p(res.block.data_ptr()),
                          ctypes.byref(tk), stream) == -1
        torch.cuda.synchronize()
        assert torch.equal(q.policy_obs, rows0) and not bool(stray.any())

        def out(**kw):
            d = dict(struct_size=ctypes.sizeof(_lib.ssd_flat_policy_out), dtype=1, obs_dev=q.policy_obs.data_ptr())
            d.update(kw)
            return _lib.ssd_flat_policy_out(**d)
        for bad in (out(dtype=3), out(dtype=-1), out(obs_dev=q.policy_obs.data_ptr() + 2), out(obs_dev=None),
                    out(struct_size=8)):
            assert lib.ssd_set_flat_policy_output(u._h, ctypes.byref(bad)) == -1
        u.reset()                                      # nothing was stored: the float64 handle still writes its rows
        assert bool(u.obs.any())
        # NULL switches the mode off: the handle writes float64 rows again (and takes obs_dev)
        assert lib.ssd_set_flat_policy_output(q._h, None) == 0
        assert reset(q._h, None, ctypes.c_void_p(stray.data_ptr()), stream) == 0
        assert reset(u._h, None, ctypes.c_void_p(u.obs.data_ptr()), stream) == 0
        torch.cuda.synchronize()
        assert torch.equal(stray, u.obs) and torch.equal(q.policy_obs, rows0)
        # ... and the calls that change theta leave the old rows as they were
        q.set_contract_params(0.25)
        negotiate(q, torch.full((E,), 0.5, dtype=torch.float64, device="cuda"), torch.ones((E, n), dtype=torch.float64, device="cuda"))
        torch.cuda.synchronize()
        assert torch.equal(q.policy_obs, rows0)
        with pytest.raises(ValueError):
            _make(kind, E, n, torch.int8)
    from contracts_b200.batched import BatchedGridEnv
    grid = BatchedGridEnv("cleanup_new", 4, 2)
    buf = torch.zeros((8, 64), dtype=torch.float32, device="cuda")
    good = _lib.ssd_flat_policy_out(struct_size=ctypes.sizeof(_lib.ssd_flat_policy_out), dtype=0, obs_dev=buf.data_ptr())
    assert grid.lib.ssd_set_flat_policy_output(grid._h, ctypes.byref(good)) == -1
    assert b"gridworld" in grid.lib.ssd_last_error(grid._h)

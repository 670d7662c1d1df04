"""GPU: the grid-world step writing the policy's input tensors directly (BatchedGridEnv(policy_dtype=T),
ssd_set_policy_output).

An env in policy mode must hold, after every call, exactly what `policy_inputs(T)` makes of the uint8 windows of a twin
env (same configuration and seed) that took the same calls, and every other output must equal the twin's."""
import ctypes

import numpy as np
import pytest

import golden_util as gu

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

DTYPES = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}
CONTRACT = {"cleanup_new": "CleanupContract", "harvest_new": "HarvestFeaturemodLocalContract"}


def _make(kind, E, n, dtype, amap=None, horizon=14, seed=11, first_env_id=5):
    from contracts_b200.batched import BatchedGridEnv
    return BatchedGridEnv(kind, E, n, amap, horizon=horizon, contract=CONTRACT[kind], seed=seed, first_env_id=first_env_id,
                          policy_dtype=dtype)


class Twins:
    """a uint8 env and a policy-mode env of the same configuration, driven with the same calls"""

    def __init__(self, kind, E, n, dtype, amap=None, **kw):
        self.u, self.q, self.dtype, self.kind, self.E, self.n = _make(kind, E, n, None, amap, **kw), _make(kind, E, n, dtype, amap, **kw), \
            dtype, kind, E, n
        self.nact = 9 if kind == "cleanup_new" else 8
        self.rng = np.random.RandomState(7)

    def check(self, ctx):
        img, con = self.u.policy_inputs(self.dtype)
        torch.cuda.synchronize()
        assert self.q.obs is None
        assert torch.equal(self.q.policy_image, img), "image differs after %s" % ctx
        assert torch.equal(self.q.policy_contract, con), "contract rows differ after %s" % ctx

    def same(self, ctx, features=False):
        for name in ("rew", "base_rew", "transfers", "info", "done") + (("feature_obs",) if features else ()):
            assert torch.equal(getattr(self.u, name), getattr(self.q, name)), "%s differs after %s" % (name, ctx)
        assert torch.equal(self.u.get_state()["theta"], self.q.get_state()["theta"]), ctx

    def actions(self):
        return torch.as_tensor(self.rng.randint(0, self.nact, size=(self.E, self.n)).astype(np.uint8)).cuda()

    def negotiation(self):
        prop = torch.as_tensor(self.rng.uniform(0.0, 0.2, self.E)).cuda()
        acc = torch.as_tensor(self.rng.uniform(0.0, 1.0, (self.E, self.n))).cuda()
        return prop, acc

    def both(self, fn):
        return fn(self.u), fn(self.q)


def _run_twins(tw):
    E, n = tw.E, tw.n
    r_u, r_q = tw.both(lambda e: e.reset())
    assert r_q is tw.q.policy_image
    tw.check("reset")
    prop, acc = tw.negotiation()
    d_u, d_q = tw.both(lambda e: e.negotiate(prop, acc))
    assert torch.equal(d_u, d_q)
    tw.check("negotiate")
    for t in range(6):                               # moves, cleaning, firing; feature_obs on and off (both observe variants)
        a, feat = tw.actions(), t % 2 == 1
        o_q = tw.both(lambda e: e.step(a, want_features=feat))[1][0]
        assert o_q is tw.q.policy_image
        tw.check("step %d" % t)
        tw.same("step %d" % t, feat)
    mask = torch.as_tensor(tw.rng.randint(0, 2, E).astype(np.uint8)).cuda()
    tw.both(lambda e: e.reset(mask))
    tw.check("reset(mask)")
    dec_u, dec_q = (torch.zeros(E, dtype=torch.uint8, device="cuda") for _ in range(2))
    finished = 0
    for t in range(2 * tw.u.horizon):                # every env finishes (and negotiates) at least once
        a = tw.actions()
        prop, acc = tw.negotiation()
        tw.u.step(a, auto_reset=True, negotiation=(prop, acc, dec_u), want_features=t % 3 == 0)
        tw.q.step(a, auto_reset=True, negotiation=(prop, acc, dec_q), want_features=t % 3 == 0)
        finished += int(tw.u.done.sum())
        tw.check("auto-reset step %d" % t)
        tw.same("auto-reset step %d" % t, t % 3 == 0)
        assert torch.equal(dec_u, dec_q)
    assert finished >= E
    theta = torch.as_tensor(tw.rng.uniform(0.0, 0.2, E)).cuda()
    tw.both(lambda e: e.set_contract_params(theta))
    tw.check("set_contract_params")
    params = tw.u.solver_sample(3)
    vals = torch.as_tensor(tw.rng.uniform(size=(E, 4, n))).cuda()
    tw.both(lambda e: e.solver_choose(params, vals))
    tw.check("solver_choose")
    a_host = tw.actions().cpu().pin_memory()
    rews = [torch.zeros((E, n), dtype=torch.float64).pin_memory() for _ in range(2)]
    dones = [torch.zeros((E,), dtype=torch.uint8).pin_memory() for _ in range(2)]
    tw.u.step_host(a_host, rews[0], dones[0])
    o_q = tw.q.step_host(a_host, rews[1], dones[1])[0]
    assert o_q is tw.q.policy_image
    tw.check("step_host")
    assert torch.equal(rews[0], rews[1]) and torch.equal(dones[0], dones[1])
    res = [e.new_host_result() for e in (tw.u, tw.q)]
    for t in range(3):
        a_host = tw.actions().cpu().pin_memory()
        prop, acc = tw.negotiation()
        tk = [e.step_host_async(a_host, r, auto_reset=True, negotiation=(prop, acc, None)) for e, r in zip((tw.u, tw.q), res)]
        for e, k in zip((tw.u, tw.q), tk):
            e.step_host_wait(k)
        tw.check("step_host_async %d" % t)
        assert np.array_equal(res[0].rewards(), res[1].rewards()) and np.array_equal(res[0].done, res[1].done)
    ck_u, ck_q = tw.both(lambda e: e.checkpoint())
    assert ck_q.obs.dtype == tw.dtype and tuple(ck_q.obs.shape) == (E, n, 3, 15, 15)
    assert torch.equal(ck_q.rows, ck_u.rows)
    for t in range(3):
        a = tw.actions()
        tw.both(lambda e: e.step(a, auto_reset=True))
    tw.u.restore(ck_u)
    tw.q.restore(ck_q)
    tw.check("restore")
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


CASES = {
    "cleanup_n8": ("cleanup_new", 8, None),          # the stock maps: the layout-specialised observe kernels
    "harvest_n4": ("harvest_new", 4, None),
    "cleanup_n5": ("cleanup_new", 5, None),          # env blocks that start off 16-byte boundaries
    "harvest_n3": ("harvest_new", 3, None),
    "random_map": ("cleanup_new", 6, "random"),
}


@pytest.mark.parametrize("dt", sorted(DTYPES))
@pytest.mark.parametrize("case", sorted(CASES))
def test_policy_mode_twin_matches_policy_inputs(logic_variant, case, dt):
    kind, n, amap = CASES[case]
    if amap == "random":
        amap = gu.random_map(np.random.RandomState(3), "cleanup", n)
    _run_twins(Twins(kind, 37, n, DTYPES[dt], amap))


def _planar(obs_u8, dtype):
    """the reference's uint8 windows [.., 15, 15, 3] as the policy's image rows: / 255 in float64, float32, NCHW, T"""
    x = (np.asarray(obs_u8) / 255).astype(np.float32)
    return torch.from_numpy(x).reshape(-1, 15, 15, 3).permute(0, 3, 1, 2).to(dtype)


def _contract_rows(theta, n, dtype):
    t = torch.tensor([float(np.float32(theta)), 0.0], dtype=torch.float32).repeat(5)
    return t.to(dtype).expand(n, 10)


@pytest.mark.parametrize("dt", sorted(DTYPES))
@pytest.mark.parametrize("name", ["cleanup_n8", "harvest_n4"])
def test_policy_mode_replays_reference_fixture(logic_variant, name, dt):
    """the reference's observations (golden fixtures), converted on the host, against the policy-mode env alone"""
    from contracts_b200.batched import BatchedGridEnv
    fx, dtype, i = gu.load(name), DTYPES[dt], 1
    kind, n = ("cleanup_new" if str(fx["kind"]) == "cleanup" else "harvest_new"), int(fx["n"])
    env = BatchedGridEnv(kind, 3, n, [str(r) for r in fx["ascii_map"]], horizon=int(fx["horizon"]), contract=gu.contract_name(fx),
                         seed=int(fx["seed"]), first_env_id=(int(fx["env_id"]) - i) & 0xFFFFFFFF, policy_dtype=dtype,
                         **gu.shaping_kwargs(fx))
    rows = slice(i * n, (i + 1) * n)
    for ep in range(fx["actions"].shape[0]):
        img = env.reset()
        assert torch.equal(img[rows].cpu(), _planar(fx["reset_obs"][ep], dtype)), "reset ep %d" % ep
        if bool(fx["contract"]):
            assert torch.equal(env.policy_contract[rows].cpu(), _contract_rows(fx["reset_theta"][ep], n, dtype))
        for t in range(fx["actions"].shape[1]):
            a = torch.zeros((3, n), dtype=torch.uint8)
            a[:] = torch.as_tensor(fx["actions"][ep, t].astype(np.uint8))
            img, rew, done, _ = env.step(a.cuda())
            assert torch.equal(img[rows].cpu(), _planar(fx["obs"][ep, t], dtype)), "ep %d step %d" % (ep, t)
            gu.assert_same("rew", rew[i].cpu().numpy(), fx["rew"][ep, t], "ep %d step %d" % (ep, t))


@pytest.mark.parametrize("dt", sorted(DTYPES))
def test_policy_mode_replays_reference_negotiation(logic_variant, dt):
    from contracts_b200.batched import BatchedGridEnv
    fx, dtype, i = gu.load("negotiate_cleanup_n8"), DTYPES[dt], 1
    n = int(fx["n"])
    env = BatchedGridEnv("cleanup_new", 3, n, horizon=int(fx["base_horizon"]), contract="CleanupContract", seed=int(fx["seed"]),
                         first_env_id=(int(fx["env_id"]) - i) & 0xFFFFFFFF, policy_dtype=dtype)
    rows = slice(i * n, (i + 1) * n)
    steps = min(int(fx["horizon"]), int(fx["base_horizon"]))
    for ep in range(fx["acts"].shape[0]):
        img = env.reset()
        assert torch.equal(img[rows].cpu(), _planar(fx["reset_obs"][ep], dtype)), "reset ep %d" % ep
        acts = fx["acts"][ep]
        dec = env.negotiate(np.full(3, acts[0, 0]), np.tile(acts[:, 1], (3, 1)))
        assert int(dec[i]) == int(fx["accepted"][ep])
        assert torch.equal(env.policy_contract[rows].cpu(), _contract_rows(fx["contract_obs3"][ep][0, 0], n, dtype))
        total = np.zeros(n)
        for t in range(steps):
            img, rew, _, _ = env.step(torch.as_tensor(np.tile(fx["table"][t], (3, 1)).astype(np.uint8)).cuda())
            total = total + rew[i].cpu().numpy()
        gu.assert_same("summed rewards", total, fx["rew3"][ep], "ep %d" % ep)
        assert torch.equal(img[rows].cpu(), _planar(fx["obs3"][ep], dtype)), "final obs ep %d" % ep


def test_policy_mode_full_size_steady_state(oracle_lib):
    """E = 131072, cleanup n = 8, bf16: staggered episodes, auto-reset + negotiation in every step (the observe kernel's
    dynamic tail scheduler at the benchmark's size); the image and rewards of every env also against a full-size oracle
    driven through the same steps (step, reset(done), negotiate, theta of the finished envs from the negotiation)"""
    from contracts_b200.maps import CLEANUP_MAP
    E, n = 131072, 8
    tw = Twins("cleanup_new", E, n, torch.bfloat16, horizon=1000, seed=73907, first_env_id=0)
    orc = oracle_lib.GridOracle("cleanup", E, n, CLEANUP_MAP, horizon=1000, contract=CONTRACT["cleanup_new"], seed=73907)
    tw.both(lambda e: e.reset())
    orc.reset()
    phase = (torch.arange(E, dtype=torch.int32) % 1000).cuda()
    tw.both(lambda e: e.set_state(t=phase))          # staggered episodes: ~131 envs finish in every step
    orc.set_state(t=phase.cpu().numpy())
    dec_u, dec_q = (torch.zeros(E, dtype=torch.uint8, device="cuda") for _ in range(2))
    for t in range(20):
        a = tw.u.random_actions(1000 + t, 8)
        prop, acc = tw.negotiation()
        tw.u.step(a, extras=False, auto_reset=True, negotiation=(prop, acc, dec_u))
        tw.q.step(a, extras=False, auto_reset=True, negotiation=(prop, acc, dec_q))
        assert int(tw.u.done.sum()) > 0
        tw.check("full-size step %d" % t)
        for name in ("rew", "info", "done"):
            assert torch.equal(getattr(tw.u, name), getattr(tw.q, name)), name
        assert torch.equal(dec_u, dec_q)
        o = orc.step(a.cpu().numpy(), want_features=False)
        done = o["done"].astype(bool)
        want = o["obs"]
        want[done] = orc.reset(o["done"])[done]
        old = orc.get_state()["theta"]
        want_dec = orc.negotiate(prop.cpu().numpy(), acc.cpu().numpy())
        orc.set_state(theta=np.where(done, orc.get_state()["theta"], old))
        ctx = "full-size step %d" % t
        assert np.array_equal(tw.q.done.cpu().numpy(), o["done"]), ctx
        gu.assert_same("rew", tw.q.rew.cpu().numpy(), o["rew"], ctx)
        gu.assert_same("decisions", dec_q.cpu().numpy()[done], want_dec[done], ctx)
        img = tw.q.policy_image
        want_d = torch.from_numpy(want).cuda()
        for e0 in range(0, E, 16384):                 # the reference image, converted on the device 16384 envs at a time
            got = img[e0 * n:(e0 + 16384) * n]
            ref = gu.policy_image(want_d[e0:e0 + 16384], torch.bfloat16)
            if not torch.equal(got, ref):
                bad = (got != ref).reshape(-1, n * 675).any(1).nonzero().flatten()
                raise AssertionError("image differs from the oracle at %s in envs %r" % (ctx, (bad[:10] + e0).tolist()))


def test_policy_mode_graph_replay_matches_eager():
    """a captured CUDA graph of policy-mode steps (device-side action counter) replays to the tensors eager steps make"""
    E, n = 4096, 8
    eager, graphed = (_make("cleanup_new", E, n, torch.float16, horizon=30) for _ in range(2))
    prop = torch.full((E,), 0.1, dtype=torch.float64, device="cuda")
    acc = torch.full((E, n), 0.7, dtype=torch.float64, device="cuda")
    decs = [torch.zeros(E, dtype=torch.uint8, device="cuda") for _ in range(2)]

    actions = {id(e): torch.empty((E, n), dtype=torch.uint8, device="cuda") for e in (eager, graphed)}

    def substep(env, dec):
        env.step(env.random_actions(None, 9, out=actions[id(env)]), extras=False, auto_reset=True, negotiation=(prop, acc, dec))
    for env in (eager, graphed):
        env.reset()
    cap = torch.cuda.Stream()
    cap.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(cap):
        for _ in range(3):
            substep(graphed, decs[1])
    torch.cuda.current_stream().wait_stream(cap)
    for _ in range(3):
        substep(eager, decs[0])
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=cap):
        for _ in range(5):
            substep(graphed, decs[1])
    for r in range(4):
        g.replay()
        for _ in range(5):
            substep(eager, decs[0])
        torch.cuda.synchronize()
        assert torch.equal(eager.policy_image, graphed.policy_image), "replay %d" % r
        assert torch.equal(eager.policy_contract, graphed.policy_contract), "replay %d" % r
        assert torch.equal(eager.rew, graphed.rew) and torch.equal(decs[0], decs[1]), "replay %d" % r


def test_policy_output_error_surface():
    from contracts_b200 import _lib
    from contracts_b200.features import BatchedFeatureEnv
    from contracts_b200.selfdrive import BatchedCarEnv
    E, n = 16, 4
    q = _make("harvest_new", E, n, torch.float16)
    lib = q.lib
    q.reset()
    img0, rew0 = q.policy_image.clone(), q.rew.clone()
    stray = torch.zeros((E, n * 675), dtype=torch.uint8, device="cuda")
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    io = _lib.ssd_step_io()
    io.actions_dev = torch.ones((E, n), dtype=torch.uint8, device="cuda").data_ptr()
    io.obs_dev = stray.data_ptr()
    io.rew_dev = q.rew.data_ptr()
    io.done_dev = q.done.data_ptr()
    assert lib.ssd_step(q._h, ctypes.byref(io), stream) == -1                    # one observation form per handle
    assert b"policy output" in lib.ssd_last_error(q._h)
    assert lib.ssd_reset(q._h, None, ctypes.c_void_p(stray.data_ptr()), 0, stream) == -1
    torch.cuda.synchronize()
    assert torch.equal(q.policy_image, img0) and torch.equal(q.rew, rew0) and not bool(stray.any())

    def out(**kw):
        d = dict(struct_size=ctypes.sizeof(_lib.ssd_policy_out), dtype=1, image_dev=q.policy_image.data_ptr(), contract_dev=None)
        d.update(kw)
        return _lib.ssd_policy_out(**d)
    u = _make("harvest_new", E, n, None)
    for bad in (out(dtype=3), out(dtype=-1), out(image_dev=q.policy_image.data_ptr() + 2), out(image_dev=None),
                out(struct_size=8), out(contract_dev=q.policy_image.data_ptr() + 1)):
        assert lib.ssd_set_policy_output(u._h, ctypes.byref(bad)) == -1
    u.reset()                                          # nothing was stored: the uint8 handle still writes its windows
    assert bool(u.obs.any())
    feat = BatchedFeatureEnv("cleanup", 4, 2)
    car = BatchedCarEnv(4, 2)
    for e in (feat, car):
        assert lib.ssd_set_policy_output(e._h, ctypes.byref(out())) == -1
    # the uint8-only methods name the mode
    for call in (lambda: q.host_snapshot(), lambda: q.concatenated_obs(), lambda: q.policy_inputs(torch.float16)):
        with pytest.raises(ValueError, match="policy"):
            call()
    assert q.host_snapshot(obs=False)["rew"].shape == (E, n)
    # checkpoints: the rows restore across forms, observation rows only into their own form
    ck_u = u.checkpoint()
    with pytest.raises(ValueError, match="observation"):
        q.restore(ck_u)
    q.restore(u.checkpoint(with_obs=False))
    q.step(torch.zeros((E, n), dtype=torch.uint8, device="cuda"))
    u.step(torch.zeros((E, n), dtype=torch.uint8, device="cuda"))
    assert torch.equal(q.policy_image, u.policy_inputs(torch.float16)[0])
    with pytest.raises(ValueError):
        _make("harvest_new", E, n, torch.int8)
    # NULL switches the output off: the calls that change theta leave the old tensors as they were
    img1, con1 = q.policy_image.clone(), q.policy_contract.clone()
    assert lib.ssd_set_policy_output(q._h, None) == 0
    q.set_contract_params(0.25)
    q.negotiate(torch.full((E,), 0.5, dtype=torch.float64, device="cuda"), torch.ones((E, n), dtype=torch.float64, device="cuda"))
    torch.cuda.synchronize()
    assert torch.equal(q.policy_image, img1) and torch.equal(q.policy_contract, con1)

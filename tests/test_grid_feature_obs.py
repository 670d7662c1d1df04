"""GPU: the grid worlds' feature observation written by the device (BatchedGridEnv(image_obs=False), ssd_set_feature_output).

The feature form changes only the observation: the step's float64 rows must equal infos['feature_obs'] of the oracle and of
a uint8-window twin (same configuration and seed, same calls), whose every other output must stay equal; a reset row must
equal `reset_rows` below, a numpy restatement of GridWorldEnv._reset_feature_obs that itself reproduces the reference's
flatobs_* fixtures; the policy dtypes must hold `cat(f64 rows, theta, 0).to(float32).to(T)` of a float64 twin.

(The file sorts after the test_cuda_* files on purpose: test_cuda_kernel_variants reads each session's first kernel from
torch.profiler, and on a B200 that record was lost once enough GPU work had run earlier in the same process; run after
them, these tests leave the existing files' process history as it was.)"""
import ctypes
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import golden_util as gu

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "contracts_b200", "libssd_b200.so")
DTYPES = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}
CONTRACT = {"cleanup": "CleanupContract", "harvest": "HarvestFeaturemodLocalContract"}
KIND = {"cleanup": "cleanup_new", "harvest": "harvest_new"}

# The feature form's kernel instantiations: (env kind 0 cleanup / 1 harvest, mask words, output dtype 0..2 SSD_POLICY_* /
# 3 SSD_FEATURE_F64).  Mask words: 4 when both point lists fit 128 points (the stock maps), else 8 (big maps).
FEATURE_KERNELS = ["grid_feature_kernel<%d, %d, %d>" % (k, mw, o) for k in (0, 1) for mw in (4, 8) for o in range(4)] + \
                  ["grid_reset_features_kernel<%d, %d>" % (k, o) for k in (0, 1) for o in range(4)]
FAMILIES = ("grid_feature_kernel", "grid_reset_features_kernel")


def demangle(sym):
    """'_Z19grid_feature_kernelILi0ELi4ELi3EEv...' -> 'grid_feature_kernel<0, 4, 3>' (None for other symbols)"""
    m = re.match(r"_Z\d+(%s)I((?:Li\d+E)+)E" % "|".join(FAMILIES), sym)
    return None if not m else "%s<%s>" % (m.group(1), ", ".join(re.findall(r"Li(\d+)E", m.group(2))))


def test_feature_kernel_inventory():
    """CPU: every instantiation of the feature form's kernels in the built library has a row in FEATURE_KERNELS."""
    if not os.path.exists(LIB):
        pytest.skip("contracts_b200/libssd_b200.so is not built (__graft_entry__.build())")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    tool = os.path.join(os.path.dirname(nvcc), "cuobjdump")
    tool = tool if os.path.exists(tool) else shutil.which("cuobjdump")
    if tool is None:
        pytest.skip("cuobjdump not found beside nvcc")
    assert demangle("_Z26grid_reset_features_kernelILi1ELi3EEv10GridParamsPKhPvi") == "grid_reset_features_kernel<1, 3>"
    out = subprocess.run([tool, "-symbols", LIB], check=True, capture_output=True, text=True).stdout
    built = {k for k in (demangle(line.split()[-1]) for line in out.splitlines() if "STO_ENTRY" in line) if k}
    assert sorted(built - set(FEATURE_KERNELS)) == [], "feature-form instantiations without a FEATURE_KERNELS row"
    assert sorted(set(FEATURE_KERNELS) - built) == [], "FEATURE_KERNELS names kernels the library does not have"


# ---------------------------------------------------------------------------------------------------------------------
def _closest(points, pos):
    """np.argmin of L1 distances over a row-major point list, [0, 0] when empty (cleanup_new.py:396-403)"""
    if len(points) == 0:
        return [0, 0]
    return list(points[int(np.argmin(np.abs(points - np.asarray(pos)).sum(1)))])


def reset_rows(kind, ascii_map, st):
    """float64 [E, n, F]: the reset observation of every env from its state (get_state as numpy), restating
    GridWorldEnv._reset_feature_obs: cleanup's caches are from before the reset-time spawn (no apples; the waste list is
    the map's initial 'H' cells), harvest reads the map after it (count_apples_in_radius(5), j*j + k*k <= 5)."""
    base = np.array([list(r) for r in ascii_map])
    pos, ori = np.asarray(st["pos"]), np.asarray(st["ori"])
    E, n = ori.shape
    H, W = base.shape
    rows = []
    for e in range(E):
        apples = np.zeros((0, 2), int) if kind == "cleanup" else np.argwhere(np.asarray(st["map"][e]) == ord("A"))
        wastes = np.argwhere(base == "H")
        env = []
        for i in range(n):
            j = (1 if n > 1 else 0) if i == 0 else 0                  # closest_pos quirk (cleanup_new.py:405-412)
            head = [pos[e, i, 0], pos[e, i, 1], ori[e, i], pos[e, j, 0], pos[e, j, 1], ori[e, j]] + _closest(apples, pos[e, i])
            if kind == "cleanup":
                env.append(head + _closest(wastes, pos[e, i]) + [len(apples), len(wastes)] + [0] * n)
            else:
                close = sum(1 for r, c in apples if (r - pos[e, i, 0]) ** 2 + (c - pos[e, i, 1]) ** 2 <= 5)
                env.append(head + [close, len(apples)] + [0] * (2 * n))
        rows.append(env)
    return np.asarray(rows, dtype=np.float64).reshape(E, n, -1)


def _np_state(env):
    return {k: v.cpu().numpy() for k, v in env.get_state().items()}


def _make(kind, E, n, ascii_map=None, image_obs=False, policy_dtype=None, contract=True, **kw):
    from contracts_b200.batched import BatchedGridEnv
    return BatchedGridEnv(KIND[kind], E, n, ascii_map=ascii_map, contract=CONTRACT[kind] if contract else None,
                          image_obs=image_obs, policy_dtype=policy_dtype, **kw)


def _bits_equal(a, b):
    a, b = np.ascontiguousarray(a, np.float64), np.ascontiguousarray(b, np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def _actions(rng, kind, E, n):
    return torch.as_tensor(rng.randint(0, 9 if kind == "cleanup" else 8, size=(E, n)).astype(np.uint8)).cuda()


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", gu.fixture_names("flatobs_"))
def test_reset_restatement_and_fixture_replay(name):
    """The restatement reproduces the reference's reset observations, and whole fixture episodes replay through the device
    form: reset rows, step rows (features ++ [theta, 0] with the record's theta) and rewards bit for bit."""
    fx = gu.load(name)
    kind, n = str(fx["kind"]), int(fx["n"])
    env = _make(kind, 1, n, horizon=int(fx["horizon"]), seed=int(fx["seed"]), first_env_id=int(fx["env_id"]))
    ascii_map = env.ascii_map
    for ep in range(fx["actions"].shape[0]):
        obs = env.reset().cpu().numpy()
        st = _np_state(env)
        want = fx["reset_obs"][ep]
        F = obs.shape[-1]
        assert _bits_equal(reset_rows(kind, ascii_map, st)[0], want[:, :F]), "restatement, episode %d" % ep
        assert _bits_equal(obs[0], want[:, :F]), "device reset rows, episode %d" % ep
        assert _bits_equal(np.full(n, st["theta"][0]), want[:, F]) and not want[:, F + 1].any()
        for t in range(fx["actions"].shape[1]):
            obs, rew, done, info = env.step(torch.as_tensor(fx["actions"][ep, t].astype(np.uint8)).reshape(1, n).cuda())
            ctx = "episode %d step %d" % (ep, t)
            assert _bits_equal(obs.cpu().numpy()[0], fx["obs"][ep, t][:, :F]), ctx
            assert _bits_equal(rew.cpu().numpy()[0], fx["rew"][ep, t]), ctx
    env.close()


def _maps():
    from test_cuda_vs_oracle import CRAMPED_CLEANUP, CRAMPED_HARVEST
    rng = np.random.RandomState(5)
    return [("cleanup", 8, None), ("harvest", 4, None), ("cleanup", 8, CRAMPED_CLEANUP), ("harvest", 8, CRAMPED_HARVEST),
            ("cleanup", 6, gu.big_map("cleanup", 40, 50, 3)), ("harvest", 5, gu.big_map("harvest", 40, 50, 4)),
            ("cleanup", 3, gu.random_map(rng, "cleanup", 3)), ("harvest", 4, gu.random_map(rng, "harvest", 4))]


MAPS = _maps()


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(MAPS)), ids=["%s-n%d-%s" % (k, n, "stock" if m is None else "map%d" % i)
                                                        for i, (k, n, m) in enumerate(MAPS)])
def test_oracle_rollout(oracle_lib, logic_variant, case):
    """F64 rows equal the oracle's feature_obs bit for bit over a rollout with masked resets; reset rows equal the
    restatement."""
    kind, n, amap = MAPS[case]
    E, horizon, seed, first = 61, 1000, 19 + case, 3
    env = _make(kind, E, n, amap, horizon=horizon, seed=seed, first_env_id=first)
    orc = oracle_lib.GridOracle(kind, E, n, env.ascii_map, horizon=horizon, contract=CONTRACT[kind], seed=seed, first_env_id=first)
    orc.reset()
    obs = env.reset().cpu().numpy()
    assert _bits_equal(obs, reset_rows(kind, env.ascii_map, _np_state(env)))
    rng = np.random.RandomState(case)
    for t in range(40):
        if t % 9 == 8:
            mask = (rng.rand(E) < 0.3).astype(np.uint8)
            orc.reset(mask)
            obs = env.reset(torch.as_tensor(mask).cuda()).cpu().numpy()
            sel = mask.astype(bool)
            assert _bits_equal(obs[sel], reset_rows(kind, env.ascii_map, _np_state(env))[sel]), "masked reset at %d" % t
        a = _actions(rng, kind, E, n)
        o = orc.step(a.cpu().numpy(), want_features=True)
        obs, rew, done, info = env.step(a)
        assert _bits_equal(obs.cpu().numpy(), o["feature_obs"]), "feature rows at step %d" % t
        assert _bits_equal(rew.cpu().numpy(), o["rew"]), "rewards at step %d" % t
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", range(1, 9))
def test_agent_counts_odd_batch(oracle_lib, n):
    """n = 1..8 at an odd batch and a non-zero first_env_id, both kinds, against the oracle."""
    for kind in ("cleanup", "harvest"):
        E, seed, first = 37, 7 + n, 1001
        env = _make(kind, E, n, contract=n > 1, horizon=1000, seed=seed, first_env_id=first)
        orc = oracle_lib.GridOracle(kind, E, n, env.ascii_map, horizon=1000, contract=CONTRACT[kind] if n > 1 else None,
                                    seed=seed, first_env_id=first)
        orc.reset()
        assert _bits_equal(env.reset().cpu().numpy(), reset_rows(kind, env.ascii_map, _np_state(env)))
        rng = np.random.RandomState(n)
        for t in range(25):
            a = _actions(rng, kind, E, n)
            o = orc.step(a.cpu().numpy(), want_features=True)
            obs = env.step(a)[0]
            assert _bits_equal(obs.cpu().numpy(), o["feature_obs"]), "%s step %d" % (kind, t)
        env.close()


class Twin:
    """a uint8-window env (features asked for) and a feature-form env of the same configuration, driven alike"""

    def __init__(self, kind, E, n, amap=None, horizon=9, **kw):
        from contracts_b200.episodes import EpisodeLog
        self.kind, self.E, self.n = kind, E, n
        self.u = _make(kind, E, n, amap, image_obs=True, horizon=horizon, **kw)
        self.f = _make(kind, E, n, amap, image_obs=False, horizon=horizon, **kw)
        self.logs = [EpisodeLog(e, capacity=64 * E) for e in (self.u, self.f)]
        self.stats = [torch.zeros(8, dtype=torch.float64, device="cuda") for _ in range(2)]
        for e, log, s in zip((self.u, self.f), self.logs, self.stats):
            e.set_episode_log(log)
            e.set_episode_stats(s)

    def same(self, ctx):
        for name in ("rew", "base_rew", "transfers", "info", "done"):
            assert torch.equal(getattr(self.u, name), getattr(self.f, name)), "%s differs after %s" % (name, ctx)
        su, sf = self.u.get_state(), self.f.get_state()
        for k in su:
            assert torch.equal(su[k], sf[k]), "state %s differs after %s" % (k, ctx)
        assert torch.equal(self.u.metrics_raw(), self.f.metrics_raw()), ctx
        # episode statistics are atomicAdd sums over envs, in no fixed order: the integer-valued fields (apples, raw rewards,
        # dirt, raw sum, episodes, max err) are exact whatever the order, transfers and transferred rewards equal to rounding
        su, sf = self.stats
        exact = [0, 1, 3, 5, 6, 7]
        assert torch.equal(su[exact], sf[exact]), ctx
        assert torch.allclose(su[[2, 4]], sf[[2, 4]], rtol=1e-12, atol=1e-12), ctx


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ("cleanup", "harvest"))
def test_uint8_twin_auto_reset(logic_variant, kind):
    """Staggered auto-reset with negotiation: every output but the observation equals the uint8 twin's at every step (and
    the episode log); rows of continuing envs are the twin's feature_obs, rows of restarted envs their reset rows."""
    E, n = 45, 4
    tw = Twin(kind, E, n, seed=3, first_env_id=9)
    tw.u.reset(); tw.f.reset()
    stagger = torch.as_tensor((np.arange(E) % 3 == 0).astype(np.uint8)).cuda()
    rng = np.random.RandomState(1)
    for t in range(40):
        if t in (2, 5):                                       # staggered episodes
            tw.u.reset(stagger); tw.f.reset(stagger)
        a = _actions(rng, kind, E, n)
        prop = torch.as_tensor(rng.rand(E) * 0.2).cuda()
        acc = torch.as_tensor(rng.rand(E, n)).cuda()
        decs = [torch.zeros(E, dtype=torch.uint8, device="cuda") for _ in range(2)]
        tw.u.step(a, want_features=True, auto_reset=True, negotiation=(prop, acc, decs[0]))
        obs = tw.f.step(a, auto_reset=True, negotiation=(prop, acc, decs[1]))[0].cpu().numpy()
        torch.cuda.synchronize()
        tw.same("step %d" % t)
        assert torch.equal(decs[0], decs[1])
        done = tw.f.done.cpu().numpy().astype(bool)
        assert _bits_equal(obs[~done], tw.u.feature_obs.cpu().numpy()[~done]), "continuing envs at step %d" % t
        assert _bits_equal(obs[done], reset_rows(kind, tw.f.ascii_map, _np_state(tw.f))[done]), "restarted envs at step %d" % t
    ru, rf = (log.drain() for log in tw.logs)
    assert len(ru["env_id"]) > 0
    for k in ru:
        assert np.array_equal(ru[k], rf[k]), "episode log %s differs" % k


def flat_rows(obs, theta, contract, dtype):
    E, n, F = obs.shape
    x = obs.reshape(E * n, F)
    if contract:
        th = theta.to(x.device, torch.float64).repeat_interleave(n).unsqueeze(1)
        x = torch.cat((x, th, torch.zeros_like(th)), -1)
    return x.to(torch.float32).to(dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", sorted(DTYPES))
@pytest.mark.parametrize("kind,contract", [("cleanup", True), ("harvest", True), ("cleanup", False), ("harvest", False)])
def test_policy_dtype_twin(kind, contract, dt):
    """T rows equal cat(f64 rows, theta, 0).float().to(T) of a float64 twin through reset, step, auto-reset with
    negotiation, set_contract_params, negotiate, solver_choose and checkpoint save / load."""
    E, n, dtype = 33, 3, DTYPES[dt]
    u = _make(kind, E, n, contract=contract, horizon=6, seed=5, first_env_id=2)
    q = _make(kind, E, n, contract=contract, policy_dtype=dtype, horizon=6, seed=5, first_env_id=2)
    assert q.obs is None and q.policy_obs.shape == (E * n, q.policy_width) and q.policy_width == u.F + (2 if contract else 0)

    def check(ctx):
        torch.cuda.synchronize()
        want = flat_rows(u.obs, u.get_state()["theta"], contract, dtype)
        assert torch.equal(q.policy_obs, want), "policy rows differ after %s" % ctx
        for name in ("rew", "done", "info"):
            assert torch.equal(getattr(u, name), getattr(q, name)), "%s after %s" % (name, ctx)

    u.reset(); q.reset(); check("reset")
    rng = np.random.RandomState(2)
    for t in range(14):
        a = _actions(rng, kind, E, n)
        neg = None
        if contract:
            prop, acc = torch.as_tensor(rng.rand(E) * 0.2).cuda(), torch.as_tensor(rng.rand(E, n)).cuda()
            neg = (prop, acc, None)
        u.step(a, auto_reset=True, negotiation=neg); q.step(a, auto_reset=True, negotiation=neg)
        check("step %d" % t)
    if contract:
        th = torch.as_tensor(rng.rand(E) * 0.2).cuda()
        u.set_contract_params(th); q.set_contract_params(th); check("set_contract_params")
        prop, acc = torch.as_tensor(rng.rand(E) * 0.2).cuda(), torch.as_tensor(rng.rand(E, n)).cuda()
        mask = torch.as_tensor((np.arange(E) % 2).astype(np.uint8)).cuda()
        u.negotiate(prop, acc, mask=mask); q.negotiate(prop, acc, mask=mask); check("negotiate")
        params = u.solver_sample(4)
        vals = torch.as_tensor(rng.rand(E, 5, n)).cuda()
        u.solver_choose(params, vals); q.solver_choose(params, vals); check("solver_choose")
    cku, ckq = u.checkpoint(), q.checkpoint()
    for t in range(3):
        a = _actions(rng, kind, E, n)
        u.step(a); q.step(a)
    u.restore(cku); q.restore(ckq); check("checkpoint load")
    with pytest.raises(ValueError):
        q.restore(cku)                                       # float64 rows into a T-row env: another observation form
    u.close(); q.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ("cleanup", "harvest"))
def test_graph_replay_and_host_paths(kind):
    """A 50-step CUDA graph of the steady state (random actions, auto-reset with negotiation) equals eager steps; the
    host-buffer step and the pipelined host step write the same rows as ssd_step."""
    E, n = 300, 4
    g = _make(kind, E, n, horizon=20, seed=8)
    e = _make(kind, E, n, horizon=20, seed=8)
    prop = torch.full((E,), 0.1, dtype=torch.float64, device="cuda")
    acc = torch.full((E, n), 0.7, dtype=torch.float64, device="cuda")
    for env in (g, e):
        env.reset()
        env.reset(torch.as_tensor((np.arange(E) % 2).astype(np.uint8)).cuda())
    act_g = torch.empty((E, n), dtype=torch.uint8, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                                 # warm-up outside capture
        g.step(g.random_actions(None, 9 if kind == "cleanup" else 8, out=act_g), auto_reset=True, negotiation=(prop, acc, None))
    torch.cuda.current_stream().wait_stream(s)
    e.step(e.random_actions(None, 9 if kind == "cleanup" else 8), auto_reset=True, negotiation=(prop, acc, None))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(50):
            g.step(g.random_actions(None, 9 if kind == "cleanup" else 8, out=act_g), auto_reset=True, negotiation=(prop, acc, None))
    graph.replay()
    for _ in range(50):
        e.step(e.random_actions(None, 9 if kind == "cleanup" else 8), auto_reset=True, negotiation=(prop, acc, None))
    torch.cuda.synchronize()
    assert torch.equal(g.obs, e.obs) and torch.equal(g.rew, e.rew) and torch.equal(g.done, e.done)
    assert torch.equal(g.metrics_raw(), e.metrics_raw())
    # host paths: ssd_step_host and the pipelined ssd_step_host_async against ssd_step
    rng = np.random.RandomState(4)
    a = torch.as_tensor(rng.randint(0, 7, size=(E, n)).astype(np.uint8)).pin_memory()
    rew_h, done_h = torch.empty((E, n), dtype=torch.float64).pin_memory(), torch.empty(E, dtype=torch.uint8).pin_memory()
    g.step_host(a, rew_h, done_h)
    e.step(a.cuda())
    torch.cuda.synchronize()
    assert torch.equal(g.obs, e.obs) and torch.equal(rew_h, e.rew.cpu())
    res = g.new_host_result()
    a = torch.as_tensor(rng.randint(0, 7, size=(E, n)).astype(np.uint8)).pin_memory()
    g.step_host_wait(g.step_host_async(a, res))
    e.step(a.cuda())
    torch.cuda.synchronize()
    assert torch.equal(g.obs, e.obs) and np.array_equal(res.rewards(), e.rew.cpu().numpy())
    g.close(); e.close()


@pytest.mark.gpu
def test_full_size_cleanup_steady_state(oracle_lib):
    """The benchmark's size, cleanup n = 8 at 131072 envs: staggered episodes, masked resets, steps against a full-size
    oracle."""
    E, n = 131072, 8
    env = _make("cleanup", E, n, horizon=1000, seed=73907)
    orc = oracle_lib.GridOracle("cleanup", E, n, env.ascii_map, horizon=1000, contract="CleanupContract", seed=73907)
    orc.reset(); env.reset()
    rng = np.random.RandomState(0)
    for t in range(6):
        if t == 3:
            mask = (np.arange(E) % 5 == 0).astype(np.uint8)
            orc.reset(mask)
            obs = env.reset(torch.as_tensor(mask).cuda()).cpu().numpy()
            sel = mask.astype(bool)
            assert _bits_equal(obs[sel][:4096], reset_rows("cleanup", env.ascii_map, {k: v[sel][:4096] for k, v in _np_state(env).items()}))
        a = _actions(rng, "cleanup", E, n)
        o = orc.step(a.cpu().numpy(), want_features=True)
        obs, rew = env.step(a)[:2]
        assert _bits_equal(obs.cpu().numpy(), o["feature_obs"]), "step %d" % t
        assert _bits_equal(rew.cpu().numpy(), o["rew"]), "step %d" % t
    env.close()


@pytest.mark.gpu
def test_launched_kernels():
    """torch.profiler: the feature form launches grid_feature_kernel and (reset / auto-reset) grid_reset_features_kernel
    in every output form on the stock maps (cleanup: 4 mask words, harvest's 155 apple points: 8) — and never
    grid_obs_kernel."""
    forms = [(None, 3)] + [(DTYPES[d], o) for o, d in enumerate(("f32", "f16", "bf16"))]
    envs = [(_make(kind, 256, 4, horizon=3, policy_dtype=dt), kind) for kind in ("cleanup", "harvest") for dt, _ in forms]

    def run():
        for env, kind in envs:
            env.reset()
            a = env.random_actions(None, 8)
            for _ in range(4):
                env.step(env.random_actions(None, 8, out=a), auto_reset=True)
    names = gu.profiled_names(run)
    for k in (0, 1):
        for _, o in forms:
            for want in ("grid_feature_kernel<%d, %d, %d>" % (k, 4 if k == 0 else 8, o), "grid_reset_features_kernel<%d, %d>" % (k, o)):
                assert any(want in s for s in names), (want, sorted(s for s in names if "kernel<" in s))
    assert not any("grid_obs_kernel" in s for s in names), sorted(names)
    for env, _ in envs:
        env.close()


@pytest.mark.gpu
def test_error_surface():
    from contracts_b200 import _lib
    env = _make("cleanup", 8, 3)
    lib, h = env.lib, env._h
    buf = torch.zeros(8 * 3 * 32, dtype=torch.float64, device="cuda")
    size = ctypes.sizeof(_lib.ssd_feature_out)

    def setf(struct_size=size, dtype=_lib.FEATURE_F64, ptr=buf.data_ptr()):
        out = _lib.ssd_feature_out(struct_size=struct_size, dtype=dtype, obs_dev=ptr)
        return lib.ssd_set_feature_output(h, ctypes.byref(out))

    assert setf(struct_size=size - 1) == -1
    assert setf(dtype=4) == -1 and setf(dtype=-1) == -1
    assert setf(ptr=None) == -1 and setf(ptr=buf.data_ptr() + 8) == -1
    # the failed calls stored nothing: the env still writes its own rows
    env.reset()
    torch.cuda.synchronize()
    assert env.obs.abs().sum() > 0 and buf.abs().sum() == 0
    # obs_dev or feature_obs_dev while the form is set
    win = torch.zeros((8, 3 * 675), dtype=torch.uint8, device="cuda")
    stream = env._stream()
    assert lib.ssd_reset(h, None, ctypes.c_void_p(win.data_ptr()), 0, stream) == -1
    io = _lib.ssd_step_io()
    acts = torch.zeros((8, 3), dtype=torch.uint8, device="cuda")
    io.actions_dev, io.rew_dev, io.done_dev = acts.data_ptr(), env.rew.data_ptr(), env.done.data_ptr()
    io.obs_dev = win.data_ptr()
    assert lib.ssd_step(h, ctypes.byref(io), stream) == -1
    io.obs_dev, io.feature_obs_dev = None, buf.data_ptr()
    assert lib.ssd_step(h, ctypes.byref(io), stream) == -1
    io.feature_obs_dev = None
    assert lib.ssd_step(h, ctypes.byref(io), stream) == 0
    with pytest.raises(ValueError):
        env.step(acts, want_features=True)
    for call in (env.concatenated_obs, env.policy_inputs, env.host_snapshot):
        with pytest.raises(ValueError):
            call()
    # NULL switches back to windows: obs_dev is required again and gets the windows
    assert lib.ssd_set_feature_output(h, None) == 0
    assert lib.ssd_reset(h, None, ctypes.c_void_p(win.data_ptr()), 0, stream) == 0
    torch.cuda.synchronize()
    assert win.any()
    io.obs_dev = None
    assert lib.ssd_step(h, ctypes.byref(io), stream) == -1
    env.close()
    # non-grid handles
    from contracts_b200.features import BatchedFeatureEnv
    fe = BatchedFeatureEnv("cleanup", 8, 3)
    out = _lib.ssd_feature_out(struct_size=size, dtype=_lib.FEATURE_F64, obs_dev=buf.data_ptr())
    assert fe.lib.ssd_set_feature_output(fe._h, ctypes.byref(out)) == -1
    fe.close()
    from contracts_b200.selfdrive import BatchedCarEnv
    car = BatchedCarEnv(8, 2)
    assert car.lib.ssd_set_feature_output(car._h, ctypes.byref(out)) == -1
    car.close()

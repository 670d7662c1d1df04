"""GPU: JointEnv's global observation written by the device (BatchedGridEnv(global_obs=True), ssd_set_global_output).

The global form changes only the observation: its uint8 rows must equal GridOracle.global_view(), the reference's joint_*_global
fixtures and a uint8-window twin's global_view() (same configuration and seed, same calls), whose every other output must stay
equal; the policy dtypes must hold (u8.double() / 255).float().to(T).permute(0, 3, 1, 2) of a uint8 twin.  Every comparison
is by bit pattern.

(The file sorts after the test_cuda_* files on purpose: test_cuda_kernel_variants reads each session's first kernel from
torch.profiler, and on a B200 that record was lost once enough GPU work had run earlier in the same process.)"""
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
KIND = {"cleanup": "cleanup_new", "harvest": "harvest_new"}
NACT = {"cleanup": 9, "harvest": 8}

# The global form's kernel instantiations: (env kind 0 cleanup / 1 harvest, mask words, output dtype 0..2 SSD_POLICY_* /
# 4 SSD_GLOBAL_U8).  Mask words: 4 when both point lists fit 128 points, else 8 (big maps; harvest's stock map has 155 apple
# points).  Each row is launched by a test below: test_launched_kernels (stock maps) and test_other_mask_words_launch.
GLOBAL_KERNELS = ["grid_global_kernel<%d, %d, %d>" % (k, mw, o) for k in (0, 1) for mw in (4, 8) for o in (0, 1, 2, 4)] + \
                 ["grid_reset_global_kernel<%d, %d>" % (k, o) for k in (0, 1) for o in (0, 1, 2, 4)]
FAMILIES = ("grid_global_kernel", "grid_reset_global_kernel")


def demangle(sym):
    """'_Z18grid_global_kernelILi0ELi4ELi4EEv...' -> 'grid_global_kernel<0, 4, 4>' (None for other symbols)"""
    m = re.match(r"_Z\d+(%s)I((?:Li\d+E)+)E" % "|".join(FAMILIES), sym)
    return None if not m else "%s<%s>" % (m.group(1), ", ".join(re.findall(r"Li(\d+)E", m.group(2))))


def test_global_kernel_inventory():
    """CPU: every instantiation of the global form's kernels in the built library has a row in GLOBAL_KERNELS."""
    if not os.path.exists(LIB):
        pytest.skip("contracts_b200/libssd_b200.so is not built (__graft_entry__.build())")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    tool = os.path.join(os.path.dirname(nvcc), "cuobjdump")
    tool = tool if os.path.exists(tool) else shutil.which("cuobjdump")
    if tool is None:
        pytest.skip("cuobjdump not found beside nvcc")
    assert demangle("_Z24grid_reset_global_kernelILi1ELi4EEv10GridParamsPKhPvi") == "grid_reset_global_kernel<1, 4>"
    out = subprocess.run([tool, "-symbols", LIB], check=True, capture_output=True, text=True).stdout
    built = {k for k in (demangle(line.split()[-1]) for line in out.splitlines() if "STO_ENTRY" in line) if k}
    assert sorted(built - set(GLOBAL_KERNELS)) == [], "global-form instantiations without a GLOBAL_KERNELS row"
    assert sorted(set(GLOBAL_KERNELS) - built) == [], "GLOBAL_KERNELS names kernels the library does not have"


# ---------------------------------------------------------------------------------------------------------------------
def _make(kind, E, n, ascii_map=None, global_obs=True, policy_dtype=None, **kw):
    from contracts_b200.batched import BatchedGridEnv
    return BatchedGridEnv(KIND[kind], E, n, ascii_map=ascii_map, global_obs=global_obs, policy_dtype=policy_dtype, **kw)


def conv(u8, dtype):
    """get_global_obs() as VisionNetwork.forward feeds it: uint8 [E, H, W, 3] -> T [E, 3, H, W]"""
    return (u8.double() / 255).float().to(dtype).permute(0, 3, 1, 2)


def _actions(rng, kind, E, n):
    return torch.as_tensor(rng.randint(0, NACT[kind], size=(E, n)).astype(np.uint8)).cuda()


def _eq(got, want, ctx):
    got = got.cpu().numpy() if torch.is_tensor(got) else got
    assert got.shape == want.shape and np.array_equal(got, want), ctx


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", [f for f in gu.fixture_names("joint_") if f.endswith("_global")])
def test_fixture_replay(logic_variant, name):
    """Every reset and step observation of the uint8 form equals the reference's fixture; the policy dtypes equal its
    torch conversion."""
    fx = gu.load(name)
    kind, n = str(fx["kind"]), int(fx["n"])
    kw = dict(horizon=int(fx["horizon"]), seed=int(fx["seed"]), first_env_id=int(fx["env_id"]))
    envs = [_make(kind, 1, n, **kw)] + [_make(kind, 1, n, policy_dtype=DTYPES[d], **kw) for d in sorted(DTYPES)]

    def check(want, ctx):
        want_t = torch.as_tensor(want).cuda()[None]
        _eq(envs[0].obs, want[None], ctx)
        for e in envs[1:]:
            assert torch.equal(e.policy_obs, conv(want_t, e.policy_dtype)), "%s %s" % (e.policy_dtype, ctx)

    for ep in range(fx["actions"].shape[0]):
        for e in envs:
            e.reset()
        check(fx["reset_obs"][ep], "reset, episode %d" % ep)
        for t in range(fx["actions"].shape[1]):
            a = torch.as_tensor(fx["actions"][ep, t].astype(np.uint8)).reshape(1, n).cuda()
            for e in envs:
                e.step(a)
            check(fx["obs"][ep, t], "episode %d step %d" % (ep, t))
            assert float(envs[0].rew.sum()) == float(fx["rew"][ep, t])
    for e in envs:
        e.close()


def _maps():
    from test_cuda_vs_oracle import CRAMPED_CLEANUP, CRAMPED_HARVEST
    rng = np.random.RandomState(11)
    return [("cleanup", 8, None), ("harvest", 4, None), ("cleanup", 8, CRAMPED_CLEANUP), ("harvest", 8, CRAMPED_HARVEST),
            ("cleanup", 6, gu.big_map("cleanup", 48, 64, 3)), ("harvest", 5, gu.big_map("harvest", 47, 63, 4)),
            ("cleanup", 7, gu.big_map("cleanup", 45, 61, 8)), ("harvest", 3, gu.big_map("harvest", 48, 64, 9)),
            ("cleanup", 3, gu.random_map(rng, "cleanup", 3)), ("harvest", 4, gu.random_map(rng, "harvest", 4)),
            ("cleanup", 2, gu.random_map(rng, "cleanup", 2)), ("harvest", 1, gu.random_map(rng, "harvest", 1))]


MAPS = _maps()


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(MAPS)), ids=["%s-n%d-%s" % (k, n, "stock" if m is None else "map%d" % i)
                                                        for i, (k, n, m) in enumerate(MAPS)])
def test_oracle_rollout(oracle_lib, logic_variant, case):
    """uint8 rows equal GridOracle.global_view() over a rollout with masked resets mid-episode, at a batch that fills
    neither the last warp nor the last CTA."""
    kind, n, amap = MAPS[case]
    E, seed, first = 61, 19 + case, 3
    env = _make(kind, E, n, amap, horizon=1000, seed=seed, first_env_id=first)
    orc = oracle_lib.GridOracle(kind, E, n, env.ascii_map, horizon=1000, seed=seed, first_env_id=first)
    orc.reset()
    _eq(env.reset(), orc.global_view(), "reset")
    rng = np.random.RandomState(case)
    for t in range(40):
        if t % 9 == 8:
            mask = (rng.rand(E) < 0.3).astype(np.uint8)
            orc.reset(mask)
            _eq(env.reset(torch.as_tensor(mask).cuda()), orc.global_view(), "masked reset at %d" % t)
        a = _actions(rng, kind, E, n)
        o = orc.step(a.cpu().numpy(), want_features=False)
        obs, rew = env.step(a)[:2]
        _eq(obs, orc.global_view(), "view at step %d" % t)
        _eq(rew, o["rew"], "rewards at step %d" % t)
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", range(1, 9))
def test_agent_counts_odd_batch(oracle_lib, n):
    """n = 1..8 at an odd batch and a non-zero first_env_id, both kinds, against the oracle."""
    for kind in ("cleanup", "harvest"):
        E, seed, first = 37, 7 + n, 1001
        env = _make(kind, E, n, horizon=1000, seed=seed, first_env_id=first)
        orc = oracle_lib.GridOracle(kind, E, n, env.ascii_map, horizon=1000, seed=seed, first_env_id=first)
        orc.reset()
        _eq(env.reset(), orc.global_view(), "%s reset" % kind)
        rng = np.random.RandomState(n)
        for t in range(25):
            a = _actions(rng, kind, E, n)
            orc.step(a.cpu().numpy(), want_features=False)
            _eq(env.step(a)[0], orc.global_view(), "%s step %d" % (kind, t))
        env.close()


class Twin:
    """a uint8-window env and a global-form env of the same configuration, driven alike"""

    def __init__(self, kind, E, n, horizon=9, **kw):
        from contracts_b200.episodes import EpisodeLog
        self.shaped = kw.get("inequity_averse_reward", False)
        self.u = _make(kind, E, n, global_obs=False, horizon=horizon, **kw)
        self.g = _make(kind, E, n, horizon=horizon, **kw)
        self.logs = [EpisodeLog(e, capacity=64 * E) for e in (self.u, self.g)]
        self.stats = [torch.zeros(8, dtype=torch.float64, device="cuda") for _ in range(2)]
        for e, log, s in zip((self.u, self.g), self.logs, self.stats):
            e.set_episode_log(log)
            e.set_episode_stats(s)

    def same(self, ctx):
        torch.cuda.synchronize()
        for name in ("rew", "base_rew", "transfers", "info", "done"):
            assert torch.equal(getattr(self.u, name), getattr(self.g, name)), "%s differs after %s" % (name, ctx)
        su, sg = self.u.get_state(), self.g.get_state()
        for k in su:
            assert torch.equal(su[k], sg[k]), "state %s differs after %s" % (k, ctx)
        assert torch.equal(self.u.metrics_raw(), self.g.metrics_raw()), ctx
        # episode statistics are atomicAdd sums over envs in no fixed order: the integer-valued fields are exact, the others
        # (transfers; the raw rewards too under inequity aversion, whose shaped rewards are not integers) equal to rounding
        su, sg = self.stats
        exact = [0, 3, 6, 7] if self.shaped else [0, 1, 3, 5, 6, 7]
        close = [k for k in range(8) if k not in exact]
        assert torch.equal(su[exact], sg[exact]), ctx
        assert torch.allclose(su[close], sg[close], rtol=1e-12, atol=1e-12), ctx
        view = self.u.global_view()
        assert torch.equal(self.g.obs, view), "global rows differ from the twin's global_view() after %s" % ctx
        assert torch.equal(self.g.global_view(), view) and torch.equal(self.g.render(), self.u.render()), ctx


SHAPING = {"plain": {}, "collective": dict(use_collective_reward=True),
           "inequity": dict(inequity_averse_reward=True, alpha=0.5, beta=0.25)}


@pytest.mark.gpu
@pytest.mark.parametrize("shaping", sorted(SHAPING))
@pytest.mark.parametrize("kind", ("cleanup", "harvest"))
def test_uint8_twin_auto_reset(logic_variant, kind, shaping):
    """Staggered auto-reset (bench.py's steady state): every output but the observation equals the uint8 twin's after every
    call (and the episode log); the global rows are the twin's global_view(), restarted envs included."""
    E, n = 45, 4
    tw = Twin(kind, E, n, seed=3, first_env_id=9, **SHAPING[shaping])
    tw.u.record_beams(); tw.g.record_beams()
    tw.u.reset(); tw.g.reset()
    tw.same("reset")
    stagger = torch.as_tensor((np.arange(E) % 3 == 0).astype(np.uint8)).cuda()
    rng = np.random.RandomState(1)
    for t in range(40):
        if t in (2, 5):
            tw.u.reset(stagger); tw.g.reset(stagger)
            tw.same("staggered reset at %d" % t)
        a = _actions(rng, kind, E, n)
        tw.u.step(a, auto_reset=True)
        tw.g.step(a, auto_reset=True)
        tw.same("step %d" % t)
    ru, rg = (log.drain() for log in tw.logs)
    assert len(ru["env_id"]) > 0
    for k in ru:
        assert np.array_equal(ru[k], rg[k]), "episode log %s differs" % k


@pytest.mark.gpu
@pytest.mark.parametrize("dt", sorted(DTYPES))
@pytest.mark.parametrize("kind", ("cleanup", "harvest"))
def test_policy_dtype_twin(kind, dt):
    """T rows equal the torch conversion of a uint8 global twin through reset, masked reset, steps with auto-reset and a
    checkpoint round trip."""
    E, n, dtype = 33, 3, DTYPES[dt]
    u = _make(kind, E, n, horizon=6, seed=5, first_env_id=2)
    q = _make(kind, E, n, policy_dtype=dtype, horizon=6, seed=5, first_env_id=2)
    assert q.obs is None and q.policy_obs.shape == (E, 3, q.H, q.W) and q.observation is q.policy_obs

    def check(ctx):
        torch.cuda.synchronize()
        assert torch.equal(q.policy_obs, conv(u.obs, dtype)), "policy rows differ after %s" % ctx
        for name in ("rew", "done", "info"):
            assert torch.equal(getattr(u, name), getattr(q, name)), "%s after %s" % (name, ctx)

    u.reset(); q.reset(); check("reset")
    rng = np.random.RandomState(2)
    for t in range(14):
        if t == 4:
            mask = torch.as_tensor((np.arange(E) % 4 == 1).astype(np.uint8)).cuda()
            u.reset(mask); q.reset(mask); check("masked reset")
        a = _actions(rng, kind, E, n)
        u.step(a, auto_reset=True); q.step(a, auto_reset=True)
        check("step %d" % t)
    cku, ckq = u.checkpoint(), q.checkpoint()
    for t in range(3):
        a = _actions(rng, kind, E, n)
        u.step(a); q.step(a)
    u.restore(cku); q.restore(ckq); check("checkpoint load")
    with pytest.raises(ValueError):
        q.restore(cku)                                       # uint8 rows into a T-row env: another observation form
    u.close(); q.close()


@pytest.mark.gpu
@pytest.mark.parametrize("dt", ("u8", "bf16"))
@pytest.mark.parametrize("kind", ("cleanup", "harvest"))
def test_graph_replay_and_host_paths(kind, dt):
    """A 50-step CUDA graph of the steady state (random actions, auto-reset) equals eager steps; the host-buffer step and
    the pipelined host step (with auto-reset) write the same rows as ssd_step."""
    E, n = 300, 4
    dtype = None if dt == "u8" else DTYPES[dt]
    g = _make(kind, E, n, horizon=20, seed=8, policy_dtype=dtype)
    e = _make(kind, E, n, horizon=20, seed=8, policy_dtype=dtype)
    for env in (g, e):
        env.reset()
        env.reset(torch.as_tensor((np.arange(E) % 2).astype(np.uint8)).cuda())
    act_g = torch.empty((E, n), dtype=torch.uint8, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                                 # warm-up outside capture
        g.step(g.random_actions(None, NACT[kind], out=act_g), auto_reset=True)
    torch.cuda.current_stream().wait_stream(s)
    e.step(e.random_actions(None, NACT[kind]), auto_reset=True)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(50):
            g.step(g.random_actions(None, NACT[kind], out=act_g), auto_reset=True)
    graph.replay()
    for _ in range(50):
        e.step(e.random_actions(None, NACT[kind]), auto_reset=True)
    torch.cuda.synchronize()
    assert torch.equal(g.observation, e.observation) and torch.equal(g.rew, e.rew) and torch.equal(g.done, e.done)
    assert torch.equal(g.metrics_raw(), e.metrics_raw())
    rng = np.random.RandomState(4)
    a = torch.as_tensor(rng.randint(0, 7, size=(E, n)).astype(np.uint8)).pin_memory()
    rew_h, done_h = torch.empty((E, n), dtype=torch.float64).pin_memory(), torch.empty(E, dtype=torch.uint8).pin_memory()
    g.step_host(a, rew_h, done_h)
    e.step(a.cuda())
    torch.cuda.synchronize()
    assert torch.equal(g.observation, e.observation) and torch.equal(rew_h, e.rew.cpu())
    res = g.new_host_result()
    for _ in range(25):                                        # across the horizon: the auto-reset restarts every env once
        a = torch.as_tensor(rng.randint(0, 7, size=(E, n)).astype(np.uint8)).pin_memory()
        g.step_host_wait(g.step_host_async(a, res, auto_reset=True))
        e.step(a.cuda(), auto_reset=True)
        torch.cuda.synchronize()
        assert torch.equal(g.observation, e.observation) and np.array_equal(res.rewards(), e.rew.cpu().numpy())
    g.close(); e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", (8, 2))
def test_full_size_cleanup_steady_state(oracle_lib, n):
    """The benchmark's size, cleanup at 131072 envs: staggered episodes, masked resets, steps against a full-size oracle."""
    E = 131072
    env = _make("cleanup", E, n, horizon=1000, seed=73907)
    orc = oracle_lib.GridOracle("cleanup", E, n, env.ascii_map, horizon=1000, seed=73907)
    orc.reset(); env.reset()
    rng = np.random.RandomState(n)
    for t in range(6):
        if t == 3:
            mask = (np.arange(E) % 5 == 0).astype(np.uint8)
            orc.reset(mask)
            _eq(env.reset(torch.as_tensor(mask).cuda()), orc.global_view(), "masked reset")
        a = _actions(rng, "cleanup", E, n)
        o = orc.step(a.cpu().numpy(), want_features=False)
        obs, rew = env.step(a)[:2]
        _eq(obs, orc.global_view(), "step %d" % t)
        _eq(rew, o["rew"], "step %d" % t)
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("dt", ("u8", "f16"))
def test_checkpoint_copy_envs(dt):
    """checkpoint / restore / copy_envs carry the global rows; a restore of another form's rows is refused."""
    dtype = None if dt == "u8" else DTYPES[dt]
    E, n = 20, 3
    env = _make("cleanup", E, n, horizon=50, seed=2, policy_dtype=dtype)
    twin = _make("cleanup", E, n, horizon=50, seed=2, policy_dtype=dtype)
    win = _make("cleanup", E, n, global_obs=False, horizon=50, seed=2)
    rng = np.random.RandomState(0)
    for e in (env, twin, win):
        e.reset()
    for _ in range(5):
        a = _actions(rng, "cleanup", E, n)
        for e in (env, twin, win):
            e.step(a)
    ck = env.checkpoint()
    saved = env.observation.clone()
    for _ in range(4):
        a = _actions(rng, "cleanup", E, n)
        for e in (env, twin):
            e.step(a)
    env.restore(ck)
    torch.cuda.synchronize()
    assert torch.equal(env.observation, saved)
    a = _actions(rng, "cleanup", E, n)
    twin.restore(ck)
    env.step(a); twin.step(a)
    assert torch.equal(env.observation, twin.observation)
    env.copy_envs([0, 1, 2], [5, 6, 7])
    torch.cuda.synchronize()
    assert torch.equal(env.observation[5:8], env.observation[0:3])
    for k, v in env.get_state().items():
        assert torch.equal(v[5:8], v[0:3]), k
    with pytest.raises(ValueError):
        env.restore(win.checkpoint())                       # window rows into a global-form env
    with pytest.raises(ValueError):
        win.restore(ck)
    other = _make("cleanup", E, n, horizon=50, seed=2, policy_dtype=torch.float32 if dtype is None else None)
    with pytest.raises(ValueError):
        other.restore(ck)                                   # uint8 <-> T rows
    for e in (env, twin, win, other):
        e.close()


@pytest.mark.gpu
def test_launched_kernels():
    """torch.profiler: the global form launches grid_global_kernel and (reset / auto-reset) grid_reset_global_kernel in
    every output form on the stock maps (cleanup: 4 mask words; harvest's 155 apple points: 8) — and never grid_obs_kernel.
    (The other mask-word variants run in test_oracle_rollout's big maps.)"""
    forms = [(None, 4)] + [(DTYPES[d], o) for o, d in enumerate(("f32", "f16", "bf16"))]
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
            for want in ("grid_global_kernel<%d, %d, %d>" % (k, 4 if k == 0 else 8, o), "grid_reset_global_kernel<%d, %d>" % (k, o)):
                assert any(want in s for s in names), (want, sorted(s for s in names if "kernel<" in s))
    assert not any("grid_obs_kernel" in s for s in names), sorted(names)
    for env, _ in envs:
        env.close()


@pytest.mark.gpu
def test_other_mask_words_launch():
    """torch.profiler: a big cleanup map runs the 8-word cleanup variant and a small harvest map the 4-word one, in every
    output form; their views equal global_view()."""
    from test_cuda_vs_oracle import CRAMPED_HARVEST
    forms = [(None, 4)] + [(DTYPES[d], o) for o, d in enumerate(("f32", "f16", "bf16"))]
    maps = (("cleanup", gu.big_map("cleanup", 40, 50, 3), 8), ("harvest", CRAMPED_HARVEST, 4))
    envs = [(_make(kind, 64, 3, amap, policy_dtype=dt), kind, mw, o) for kind, amap, mw in maps for dt, o in forms]

    def run():
        for env, kind, _, _ in envs:
            env.reset()
            for _ in range(3):
                env.step(env.random_actions(None, NACT[kind]))
    names = gu.profiled_names(run)
    for env, kind, mw, o in envs:
        want = "grid_global_kernel<%d, %d, %d>" % (0 if kind == "cleanup" else 1, mw, o)
        assert any(want in s for s in names), (want, sorted(s for s in names if "kernel<" in s))
        view = env.global_view()
        got = env.obs if env.policy_dtype is None else env.policy_obs
        assert torch.equal(got, view if env.policy_dtype is None else conv(view, env.policy_dtype)), want
    for env, _, _, _ in envs:
        env.close()


@pytest.mark.gpu
def test_error_surface():
    from contracts_b200 import _lib
    E, n = 8, 3
    env = _make("cleanup", E, n)
    lib, h = env.lib, env._h
    buf = torch.zeros(E * 25 * 18 * 3 + 64, dtype=torch.uint8, device="cuda")
    size = ctypes.sizeof(_lib.ssd_global_out)

    def setg(struct_size=size, dtype=_lib.GLOBAL_U8, ptr=buf.data_ptr(), handle=h, L=lib):
        out = _lib.ssd_global_out(struct_size=struct_size, dtype=dtype, obs_dev=ptr)
        return L.ssd_set_global_output(handle, ctypes.byref(out))

    assert setg(struct_size=size - 1) == -1
    assert setg(dtype=_lib.FEATURE_F64) == -1 and setg(dtype=5) == -1 and setg(dtype=-1) == -1
    assert setg(ptr=None) == -1 and setg(ptr=buf.data_ptr() + 8) == -1
    # the failed calls stored nothing: the env still writes its own rows
    env.reset()
    torch.cuda.synchronize()
    assert env.obs.any() and not buf.any()
    # obs_dev or feature_obs_dev while the form is set, in every step and reset call
    win = torch.zeros((E, n * 675), dtype=torch.uint8, device="cuda")
    feat = torch.zeros((E, n, env.F), dtype=torch.float64, device="cuda")
    stream = env._stream()
    assert lib.ssd_reset(h, None, ctypes.c_void_p(win.data_ptr()), 0, stream) == -1
    acts = torch.zeros((E, n), dtype=torch.uint8, device="cuda")
    acts_h = torch.zeros((E, n), dtype=torch.uint8).pin_memory()
    rew_h = torch.zeros((E, n), dtype=torch.float64).pin_memory()
    res = env.new_host_result()
    io = _lib.ssd_step_io()
    io.actions_dev, io.rew_dev, io.done_dev = acts.data_ptr(), env.rew.data_ptr(), env.done.data_ptr()
    ticket = ctypes.c_int64(-1)
    calls = (lambda: lib.ssd_step(h, ctypes.byref(io), stream),
             lambda: lib.ssd_step_host(h, ctypes.byref(io), ctypes.c_void_p(acts_h.data_ptr()), ctypes.c_void_p(rew_h.data_ptr()), None, stream),
             lambda: lib.ssd_step_host_async(h, ctypes.byref(io), ctypes.c_void_p(acts_h.data_ptr()), ctypes.c_void_p(res.block.data_ptr()),
                                             ctypes.byref(ticket), stream))
    for call in calls:
        io.obs_dev, io.feature_obs_dev = win.data_ptr(), None
        assert call() == -1
        io.obs_dev, io.feature_obs_dev = None, feat.data_ptr()
        assert call() == -1
    io.obs_dev = io.feature_obs_dev = None
    assert lib.ssd_step(h, ctypes.byref(io), stream) == 0
    with pytest.raises(ValueError):
        env.step(acts, want_features=True)
    with pytest.raises(ValueError):
        env.step_host(acts_h, rew_h, want_features=True)
    for call in (env.concatenated_obs, env.policy_inputs, env.host_snapshot):
        with pytest.raises(ValueError):
            call()
    assert env.global_view().shape == (E, 25, 18, 3) and env.render().shape == (E, 25, 18, 3)
    # NULL switches back to windows: obs_dev is required again and gets the windows
    assert lib.ssd_set_global_output(h, None) == 0
    assert lib.ssd_reset(h, None, ctypes.c_void_p(win.data_ptr()), 0, stream) == 0
    torch.cuda.synchronize()
    assert win.any()
    assert lib.ssd_step(h, ctypes.byref(io), stream) == -1
    # each other setter replaces the form: after it no global row is written
    fbuf = torch.zeros((E, n, env.F), dtype=torch.float64, device="cuda")
    img = torch.zeros((E * n, 3, 15, 15), dtype=torch.float32, device="cuda")
    replace = (lambda: lib.ssd_set_feature_output(h, ctypes.byref(_lib.ssd_feature_out(
                   struct_size=ctypes.sizeof(_lib.ssd_feature_out), dtype=_lib.FEATURE_F64, obs_dev=fbuf.data_ptr()))),
               lambda: lib.ssd_set_policy_output(h, ctypes.byref(_lib.ssd_policy_out(
                   struct_size=ctypes.sizeof(_lib.ssd_policy_out), dtype=0, image_dev=img.data_ptr(), contract_dev=None))))
    for other, target in zip(replace, (fbuf, img)):
        assert setg() == 0
        buf.zero_(); target.zero_()
        assert other() == 0
        assert lib.ssd_reset(h, None, None, 0, stream) == 0
        assert lib.ssd_step(h, ctypes.byref(io), stream) == 0
        torch.cuda.synchronize()
        assert target.any() and not buf.any()
    # and the global setter replaces them: rows go to buf only
    assert setg() == 0
    fbuf.zero_(); img.zero_()
    assert lib.ssd_reset(h, None, None, 0, stream) == 0
    torch.cuda.synchronize()
    assert buf.any() and not fbuf.any() and not img.any()
    env.close()
    # a contract handle, feature-env and selfdrive handles
    from contracts_b200.batched import BatchedGridEnv
    ce = BatchedGridEnv("cleanup_new", E, n, contract="CleanupContract")
    assert setg(handle=ce._h, L=ce.lib) == -1
    ce.close()
    from contracts_b200.features import BatchedFeatureEnv
    fe = BatchedFeatureEnv("cleanup", E, n)
    assert setg(handle=fe._h, L=fe.lib) == -1
    fe.close()
    from contracts_b200.selfdrive import BatchedCarEnv
    car = BatchedCarEnv(E, 2)
    assert setg(handle=car._h, L=car.lib) == -1
    car.close()
    # the Python constructor's refusals
    with pytest.raises(ValueError):
        _make("cleanup", E, n, image_obs=False)
    with pytest.raises(ValueError):
        _make("cleanup", E, n, contract="CleanupContract")


@pytest.mark.gpu
@pytest.mark.parametrize("dt", ("f32", "bf16"))
def test_concatenated_identity(dt):
    """JointEnv's concatenated variant needs no kernel of its own: policy_image.view(E, 3 n, 15, 15) of a policy_dtype env
    without a contract equals the torch conversion of a uint8 twin's concatenated_obs(), after auto-reset too."""
    dtype = DTYPES[dt]
    for n in range(1, 9):
        for kind in ("cleanup", "harvest"):
            E = 29
            u = _make(kind, E, n, global_obs=False, horizon=7, seed=n)
            q = _make(kind, E, n, global_obs=False, policy_dtype=dtype, horizon=7, seed=n)
            rng = np.random.RandomState(n)

            def check(ctx):
                want = (u.concatenated_obs().double() / 255).float().to(dtype).permute(0, 3, 1, 2)
                assert torch.equal(q.policy_image.view(E, 3 * n, 15, 15), want), "%s n=%d %s" % (kind, n, ctx)

            u.reset(); q.reset(); check("reset")
            for t in range(10):
                a = _actions(rng, kind, E, n)
                u.step(a, auto_reset=True); q.step(a, auto_reset=True)
                check("step %d" % t)
            u.close(); q.close()

"""Checkpoint / restore / copy of env state (ssd_checkpoint_*, contracts_b200/checkpoint.py).

CPU: the ctypes mirror of ssd_checkpoint_layout, EnvCheckpoint's host logic (select / cat / state_dict through
torch.save + torch.load), branching of the oracles (tests/oracle_copy/).  GPU: a restored env continues bit for bit (same handle, fresh handle,
re-sharded handles, the other logic kernel, the pipelined host path), an env copied to another id continues exactly like
the oracle's copy, and corrupt rows or rows of another configuration are rejected without touching any env."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.fixture(scope="session")
def oracle_copy(oracle_lib, tmp_path_factory):
    """copy_envs for the three C oracles: tests/oracle_copy/*.c include the oracle sources unchanged (same struct layouts)
    and are built, like the oracle, with the system gcc into a helper library of their own."""
    import glob
    import subprocess
    so = str(tmp_path_factory.mktemp("oracle_copy") / "liboracle_copy.so")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    srcs = sorted(glob.glob(os.path.join(ROOT, "tests", "oracle_copy", "*.c")))
    subprocess.run([cc, "-O2", "-std=c11", "-ffp-contract=off", "-fPIC", "-shared", "-o", so] + srcs + ["-lm"], check=True)
    lib = ctypes.CDLL(so)
    fns = {}
    for cls, name in ((oracle_lib.GridOracle, "oracle_copy_envs"), (oracle_lib.FeatOracle, "feat_oracle_copy_envs"),
                      (oracle_lib.CarOracle, "car_oracle_copy_envs")):
        f = getattr(lib, name)
        f.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
        fns[cls] = f

    def copy_envs(orc, src, dst):
        """env dst[i] of the oracle batch `orc` takes env src[i]'s state (sets may overlap) and keeps its own stream"""
        s = np.ascontiguousarray(np.asarray(src, dtype=np.int32).reshape(-1))
        d = np.ascontiguousarray(np.asarray(dst, dtype=np.int32).reshape(-1))
        if s.shape != d.shape or (s.size and (min(s.min(), d.min()) < 0 or max(s.max(), d.max()) >= orc.E)):
            raise ValueError("copy_envs: src and dst must be index lists of equal length inside [0, %d)" % orc.E)
        if len(np.unique(d)) != d.size:
            raise ValueError("copy_envs: duplicate destinations")
        assert fns[type(orc)](orc._h, s.ctypes.data_as(ctypes.c_void_p), d.ctypes.data_as(ctypes.c_void_p), int(s.size)) == 0
        orc.episode[d] = orc.episode[s].copy()
    return copy_envs


def test_checkpoint_layout_struct_matches_header():
    from contracts_b200 import _lib
    text = open(os.path.join(ROOT, "include", "ssd_b200.h")).read()
    body = re.search(r"typedef struct ssd_checkpoint_layout \{(.*?)\} ssd_checkpoint_layout;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    decls = [d.split() for d in body.split(";") if d.strip()]
    assert [d[-1] for d in decls] == [f[0] for f in _lib.ssd_checkpoint_layout._fields_]
    ctype = {"int64_t": ctypes.c_int64, "uint64_t": ctypes.c_uint64}
    assert [ctype[d[0]] for d in decls] == [f[1] for f in _lib.ssd_checkpoint_layout._fields_]


def _synthetic(first=100, count=10, row_bytes=48, tag=(1 << 63) + 12345, seed=7, obs=True):
    import torch
    from contracts_b200.checkpoint import EnvCheckpoint
    g = torch.Generator().manual_seed(first)
    rows = torch.randint(0, 256, (count, row_bytes), dtype=torch.uint8, generator=g)
    o = torch.randn((count, 3, 5), dtype=torch.float64, generator=g) if obs else None
    return EnvCheckpoint("cleanup", tag, row_bytes, seed, torch.arange(first, first + count), rows, o)


def test_env_checkpoint_select_cat_state_dict(tmp_path):
    import torch
    from contracts_b200.checkpoint import EnvCheckpoint
    ck = _synthetic()
    part = ck.select(103, 4)
    assert part.env_ids.tolist() == [103, 104, 105, 106]
    assert torch.equal(part.rows, ck.rows[3:7]) and torch.equal(part.obs, ck.obs[3:7])
    # out of order / partial: select sorts by global id and keeps only the handle's range
    both = EnvCheckpoint.cat([ck.select(105, 100), ck.select(0, 105)])
    assert both.env_ids.tolist() == [105, 106, 107, 108, 109, 100, 101, 102, 103, 104]
    back = both.select(100, 10)
    assert torch.equal(back.env_ids, ck.env_ids) and torch.equal(back.rows, ck.rows) and torch.equal(back.obs, ck.obs)
    assert len(ck.select(200, 5)) == 0
    path = str(tmp_path / "ck.pt")
    torch.save(ck.state_dict(), path)
    ld = EnvCheckpoint.from_state_dict(torch.load(path))          # default weights_only load
    assert (ld.kind, ld.config_tag, ld.row_bytes, ld.seed) == (ck.kind, ck.config_tag, ck.row_bytes, ck.seed)
    assert torch.equal(ld.env_ids, ck.env_ids) and torch.equal(ld.rows, ck.rows) and torch.equal(ld.obs, ck.obs)
    nob = _synthetic(obs=False)
    torch.save(nob.state_dict(), path)
    assert EnvCheckpoint.from_state_dict(torch.load(path)).obs is None


def test_env_checkpoint_value_errors():
    import torch
    from contracts_b200.checkpoint import EnvCheckpoint, _index_tensor
    ck = _synthetic()
    with pytest.raises(ValueError, match="duplicate global env ids"):
        EnvCheckpoint.cat([ck, ck.select(104, 1)])
    with pytest.raises(ValueError, match="configurations"):
        EnvCheckpoint.cat([ck, _synthetic(first=200, tag=5)])
    with pytest.raises(ValueError, match="configurations"):
        EnvCheckpoint.cat([ck, _synthetic(first=200, seed=8)])
    with pytest.raises(ValueError, match="observations"):
        EnvCheckpoint.cat([ck, _synthetic(first=200, obs=False)])
    with pytest.raises(ValueError):
        EnvCheckpoint.cat([])
    with pytest.raises(ValueError, match="rows must be"):
        EnvCheckpoint("cleanup", 1, 32, 0, torch.arange(3), torch.zeros((3, 48), dtype=torch.uint8))
    with pytest.raises(ValueError, match="env_ids"):
        EnvCheckpoint("cleanup", 1, 48, 0, torch.arange(4), torch.zeros((3, 48), dtype=torch.uint8))
    with pytest.raises(ValueError, match="version"):
        EnvCheckpoint.from_state_dict(dict(ck.state_dict(), version=99))
    with pytest.raises(ValueError, match="inside|lie in"):
        _index_tensor([0, 5, 10], 10, "cpu", "restore")
    with pytest.raises(ValueError, match="lie in"):
        _index_tensor([-1], 10, "cpu", "checkpoint")
    assert _index_tensor(np.array([3, 1]), 10, "cpu", "checkpoint").tolist() == [3, 1]


def _oracle_pair(oracle_lib, fam, E=6, n=4):
    from contracts_b200.maps import CLEANUP_MAP
    if fam == "grid":
        return oracle_lib.GridOracle("cleanup", E, n, CLEANUP_MAP, horizon=50, contract="CleanupContract", seed=4)
    if fam == "feat":
        return oracle_lib.FeatOracle("cleanup", E, n, CLEANUP_MAP, horizon=50, contract="CleanupContract", seed=4)
    return oracle_lib.CarOracle(E, n, contract=True, low_bound=-3.0, high_bound=3.0, seed=4)


def _oracle_actions(fam, rng, E, n):
    if fam == "car":
        return rng.uniform(-0.05, 0.1, size=(E, n)).astype(np.float32)
    return rng.randint(0, 9, size=(E, n))


@pytest.mark.parametrize("fam", ["grid", "feat", "car"])
def test_oracle_copy_envs(oracle_lib, oracle_copy, fam):
    """oracle copy_envs: the destinations' state and metrics equal the sources' (a rotation: overlapping sets)."""
    E, n = 6, 4
    orc = _oracle_pair(oracle_lib, fam, E, n)
    orc.reset()
    rng = np.random.RandomState(1)
    for _ in range(9):
        orc.step(_oracle_actions(fam, rng, E, n))
    orc.reset(np.array([0, 0, 0, 0, 1, 0], np.uint8))      # different episode counters
    orc.step(_oracle_actions(fam, rng, E, n))
    src, dst = np.array([0, 1, 4, 5]), np.array([1, 4, 0, 2])
    st0, ep0 = orc.get_state(), orc.episode.copy()
    m0 = orc.metrics_raw() if fam != "car" else None
    oracle_copy(orc, src, dst)
    st1 = orc.get_state()
    for k in st0:
        assert np.array_equal(st1[k][dst], st0[k][src]), k
        assert np.array_equal(st1[k][3], st0[k][3]), k
    assert np.array_equal(orc.episode[dst], ep0[src])
    if m0 is not None:
        assert np.array_equal(orc.metrics_raw()[dst].view(np.uint64), m0[src].view(np.uint64))
    with pytest.raises(ValueError):
        oracle_copy(orc, [0, 1], [2, 2])
    with pytest.raises(ValueError):
        oracle_copy(orc, [0], [E])


# ---------------------------------------------------------------------------------------------------------------- GPU
CONFIGS = {
    "cleanup8": dict(fam="grid", kind="cleanup_new", n=8, contract="CleanupContract"),
    "harvest4": dict(fam="grid", kind="harvest_new", n=4, contract="HarvestFeaturemodLocalContract"),
    "cleanup5_shaped": dict(fam="grid", kind="cleanup_new", n=5, contract="CleanupContract",
                            shaping=dict(use_collective_reward=True, inequity_averse_reward=True, alpha=5.0, beta=0.05)),
    "cleanup4_null": dict(fam="grid", kind="cleanup_new", n=4, contract="CleanupContract", null_prob=0.5),
    "feat_cleanup8": dict(fam="feat", kind="cleanup", n=8, contract="CleanupContract"),
    "feat_harvest5": dict(fam="feat", kind="harvest", n=5, contract="HarvestFeaturemodLocalContract"),
    "car8": dict(fam="car", kind="selfdrive", n=8, contract="SelfdriveContractDistprop"),
}
HORIZON = 40
CAR_BOUNDS = dict(low_bound=-3.0, high_bound=3.0)


def _make_env(cfg, E, first_env_id=0, seed=11, ascii_map=None):
    if cfg["fam"] == "grid":
        from contracts_b200.batched import BatchedGridEnv
        return BatchedGridEnv(cfg["kind"], E, cfg["n"], ascii_map=ascii_map, horizon=HORIZON, contract=cfg["contract"],
                              null_prob=cfg.get("null_prob", 0.0), seed=seed, first_env_id=first_env_id, **cfg.get("shaping", {}))
    if cfg["fam"] == "feat":
        from contracts_b200.features import BatchedFeatureEnv
        return BatchedFeatureEnv(cfg["kind"], E, cfg["n"], horizon=HORIZON, contract=cfg["contract"],
                                 null_prob=cfg.get("null_prob", 0.0), seed=seed, first_env_id=first_env_id)
    from contracts_b200.selfdrive import BatchedCarEnv
    return BatchedCarEnv(E, cfg["n"], contract=cfg["contract"], null_prob=cfg.get("null_prob", 0.0), seed=seed,
                         first_env_id=first_env_id, **CAR_BOUNDS)


def _make_oracle(oracle_lib, cfg, E, first_env_id=0, seed=11):
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    if cfg["fam"] == "car":
        return oracle_lib.CarOracle(E, cfg["n"], contract=True, null_prob=cfg.get("null_prob", 0.0), seed=seed,
                                    first_env_id=first_env_id, **CAR_BOUNDS)
    base = cfg["kind"].replace("_new", "")
    amap = CLEANUP_MAP if base == "cleanup" else HARVEST_MAP
    if cfg["fam"] == "feat":
        return oracle_lib.FeatOracle(base, E, cfg["n"], amap, horizon=HORIZON, contract=cfg["contract"],
                                     null_prob=cfg.get("null_prob", 0.0), seed=seed, first_env_id=first_env_id)
    return oracle_lib.GridOracle(base, E, cfg["n"], amap, horizon=HORIZON, contract=cfg["contract"],
                                 null_prob=cfg.get("null_prob", 0.0), seed=seed, first_env_id=first_env_id, **cfg.get("shaping", {}))


def _actions(cfg, rng, E):
    if cfg["fam"] == "car":
        return rng.uniform(-0.05, 0.1, size=(E, cfg["n"])).astype(np.float32)
    return rng.randint(0, 8 if "harvest" in cfg["kind"] else 9, size=(E, cfg["n"])).astype(np.uint8)


def _negotiation(cfg, E, first_env_id=0):
    """the policy's negotiation outputs for every env (a function of the global id: shardable)"""
    import torch
    if cfg["fam"] != "grid":
        return None
    ids = np.arange(first_env_id, first_env_id + E)
    prop = torch.as_tensor((ids % 7) * 0.02, dtype=torch.float64).cuda()
    acc = torch.as_tensor(((ids[:, None] * 13 + np.arange(cfg["n"])[None]) % 11) / 10.0, dtype=torch.float64).cuda().contiguous()
    return prop, acc, torch.zeros(E, dtype=torch.uint8).cuda()


def _np(t):
    return np.ascontiguousarray(t.cpu().numpy())


def _run(env, cfg, a, neg=None, auto_reset=True):
    """one step; every output, the negotiation decisions and the episode accumulators as numpy copies"""
    import torch
    at = torch.as_tensor(a).cuda()
    if neg is not None:
        neg[2].zero_()                                   # decisions of this step only
    if cfg["fam"] == "grid":
        env.step(at, auto_reset=auto_reset, negotiation=neg if auto_reset else None)
    else:
        env.step(at, auto_reset=auto_reset)
    out = {k: _np(getattr(env, k)) for k in ("obs", "rew", "base_rew", "transfers", "info", "done")}
    if neg is not None and auto_reset:
        out["dec"] = _np(neg[2])
    if cfg["fam"] == "car":
        out.update({"state_" + k: _np(v) for k, v in env.get_state().items()})
    else:
        out["metrics"] = _np(env.metrics_raw())
    return out


def _same(name, got, want, ctx):
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert got.shape == want.shape, "%s %s: shape %s != %s" % (ctx, name, got.shape, want.shape)
    if not np.array_equal(got.view(np.uint8), want.view(np.uint8)):
        bad = np.argwhere(got != want) if got.dtype == want.dtype else "dtype %s vs %s" % (got.dtype, want.dtype)
        raise AssertionError("%s %s: bit patterns differ (first differences %s)" % (ctx, name, bad[:5] if not isinstance(bad, str) else bad))


def _same_outputs(got, want, ctx):
    assert sorted(got) == sorted(want)
    for k in want:
        _same(k, got[k], want[k], ctx)


def _resume(cfg, E=37, K=13, M=64, first=3):
    env = _make_env(cfg, E, first)
    env.reset()
    neg = _negotiation(cfg, E, first)
    rng = np.random.RandomState(5)
    acts = [_actions(cfg, rng, E) for _ in range(K + M)]
    for t in range(K):
        _run(env, cfg, acts[t], neg)
    ck = env.checkpoint()
    ref = [_run(env, cfg, acts[K + i], neg) for i in range(M)]
    ref_rows = _np(env.checkpoint(with_obs=False).rows)
    finished = sum(int(r["done"][:, -1].sum()) if cfg["fam"] == "car" else int(r["done"].sum()) for r in ref)
    assert finished > 0, "the recorded window must cross an episode boundary"
    for label, target in (("same handle", env), ("fresh handle", _make_env(cfg, E, first))):
        target.restore(ck)
        _same("restored obs", _np(target.obs), _np(ck.obs), label)
        for i in range(M):
            _same_outputs(_run(target, cfg, acts[K + i], neg), ref[i], "%s step %d" % (label, K + i))
        _same("final rows", _np(target.checkpoint(with_obs=False).rows), ref_rows, label)


@pytest.mark.gpu
def test_resume_cleanup8(logic_variant):
    _resume(CONFIGS["cleanup8"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["harvest4", "cleanup5_shaped", "cleanup4_null", "feat_cleanup8", "feat_harvest5", "car8"])
def test_resume(name):
    _resume(CONFIGS[name])


@pytest.mark.gpu
def test_reshard_and_logic_kernel_choice(monkeypatch, tmp_path):
    """ids 0..999 on one handle (thread-per-env logic kernel) against 0..399 + 400..999 on two handles (octet kernel),
    restored from a checkpoint cut in two, saved to a file, loaded, concatenated and selected per handle."""
    import torch
    from contracts_b200.checkpoint import EnvCheckpoint
    cfg = CONFIGS["cleanup8"]
    E, K, M = 1000, 11, 50
    monkeypatch.setenv("SSD_LOGIC8", "0")
    a = _make_env(cfg, E, 0)
    a.reset()
    neg_a = _negotiation(cfg, E, 0)
    rng = np.random.RandomState(8)
    acts = [_actions(cfg, rng, E) for _ in range(K + M)]
    for t in range(K):
        _run(a, cfg, acts[t], neg_a)
    ck = a.checkpoint()
    paths = []
    for i, part in enumerate((ck.select(0, 300), ck.select(300, 700))):
        paths.append(str(tmp_path / ("rank%d.pt" % i)))
        torch.save(part.state_dict(), paths[-1])
    full = EnvCheckpoint.cat([EnvCheckpoint.from_state_dict(torch.load(p)) for p in paths[::-1]])
    monkeypatch.setenv("SSD_LOGIC8", "1")
    b, c = _make_env(cfg, 400, 0), _make_env(cfg, 600, 400)
    b.restore(full.select(0, 400))
    c.restore(full.select(400, 600))
    neg_b, neg_c = _negotiation(cfg, 400, 0), _negotiation(cfg, 600, 400)
    for t in range(K, K + M):
        ra, rb, rc = _run(a, cfg, acts[t], neg_a), _run(b, cfg, acts[t][:400], neg_b), _run(c, cfg, acts[t][400:], neg_c)
        _same_outputs({k: np.concatenate([rb[k], rc[k]]) for k in ra}, ra, "re-sharded step %d" % t)


def _oracle_step(orc, cfg, a):
    return orc.step(a, want_features=False) if cfg["fam"] == "grid" else orc.step(a)


def _check_vs_oracle(env, orc, cfg, got, o, ctx):
    for k in ("obs", "rew", "base_rew", "transfers", "done"):
        _same(k, got[k], o[k].astype(got[k].dtype) if k == "done" else o[k], ctx)
    assert np.array_equal(got["info"].astype(np.float64), o["info"].astype(np.float64)), ctx + " info"
    if cfg["fam"] == "car":
        so = orc.get_state()
        for k in ("pos", "vel", "theta", "transfers", "t"):
            _same(k, got["state_" + k], so[k], ctx)
    else:
        _same("metrics", got["metrics"], orc.metrics_raw(), ctx)


def _lockstep(env, orc, cfg, rng, steps, ctx):
    """step both; envs whose episode ended are reset on both (masked reset)"""
    import torch
    E = env.E
    for t in range(steps):
        a = _actions(cfg, rng, E)
        got = _run(env, cfg, a, auto_reset=False)
        _check_vs_oracle(env, orc, cfg, got, _oracle_step(orc, cfg, a), "%s step %d" % (ctx, t))
        mask = (got["done"][:, -1] if cfg["fam"] == "car" else got["done"]).astype(np.uint8)
        if mask.any():
            want = orc.reset(mask)
            env.reset(torch.as_tensor(mask).cuda())
            sel = mask.astype(bool)
            _same("reset obs", _np(env.obs)[sel], want[sel], "%s step %d" % (ctx, t))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_copy_envs_matches_oracle(oracle_lib, oracle_copy, name):
    """copy_envs with overlapping sets (a rotation, and one env copied far away): the destinations continue on their own
    random streams exactly like the oracle's copies."""
    cfg = CONFIGS[name]
    E = 23
    env, orc = _make_env(cfg, E, 7, seed=21), _make_oracle(oracle_lib, cfg, E, 7, seed=21)
    _same("reset obs", _np(env.reset()), orc.reset(), name)
    rng = np.random.RandomState(3)
    _lockstep(env, orc, cfg, rng, 17, name + " before copy")
    src, dst = [0, 1, 2, 3, 4, 5, 6, 7, 20], [3, 4, 5, 6, 7, 0, 1, 2, 11]
    obs0 = _np(env.obs)
    env.copy_envs(src, dst)
    oracle_copy(orc, src, dst)
    _same("copied obs", _np(env.obs)[dst], obs0[src], name)
    _lockstep(env, orc, cfg, rng, 50, name + " after copy")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cleanup8", "harvest4", "feat_cleanup8", "car8"])
def test_restore_continues_pipelined_host_path(name):
    """Checkpoint after step_host_wait; the original and a restored handle continue with step_host_async alike."""
    import torch
    cfg = CONFIGS[name]
    E, K, M = 64, 6, 60
    env = _make_env(cfg, E, 0)
    env.reset()
    rng = np.random.RandomState(2)
    acts = [torch.as_tensor(_actions(cfg, rng, E)).pin_memory() for _ in range(K + M)]

    def run(h, steps):
        res, out = [h.new_host_result(), h.new_host_result()], []
        for t in steps:
            r = res[t & 1]
            h.step_host_wait(h.step_host_async(acts[t], r, auto_reset=True))
            out.append((r.rewards().copy(), r.done.copy()))
        return out

    run(env, range(K))
    ck = env.checkpoint()
    want = run(env, range(K, K + M))
    other = _make_env(cfg, E, 0)
    other.restore(ck)
    got = run(other, range(K, K + M))
    for i, ((rg, dg), (rw, dw)) in enumerate(zip(got, want)):
        _same("rewards", rg, rw, "%s step %d" % (name, K + i))
        _same("dones", dg, dw, "%s step %d" % (name, K + i))


@pytest.mark.gpu
def test_restore_rejects_other_configuration():
    """A tag mismatch raises before anything is launched: other n, other map, shaped vs unshaped, other kind."""
    import torch
    from contracts_b200 import _lib
    from contracts_b200.maps import CLEANUP_MAP
    base = CONFIGS["cleanup8"]
    src = _make_env(base, 16)
    src.reset()
    ck = src.checkpoint()
    other_map = list(CLEANUP_MAP)
    r = next(i for i, row in enumerate(other_map) if "B" in row)
    other_map[r] = other_map[r].replace("B", " ", 1)
    others = [_make_env(dict(base, n=4), 16), _make_env(base, 16, ascii_map=other_map),
              _make_env(dict(base, shaping=dict(use_collective_reward=True)), 16), _make_env(CONFIGS["feat_cleanup8"], 16),
              _make_env(CONFIGS["car8"], 16)]
    for dst in others:
        before = dst.kernel_launches
        with pytest.raises(_lib.SsdError, match="another configuration"):
            dst.restore(ck)
        rows = ck.rows.cuda()
        rc = dst.lib.ssd_checkpoint_load(dst._h, ctypes.c_uint64(ck.config_tag), None, len(ck), ctypes.c_void_p(rows.data_ptr()),
                                         None, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == -1 and b"config_tag" in dst.lib.ssd_last_error(dst._h)
        assert dst.kernel_launches == before
    # same configuration, other size / place / seed: same tag
    assert _make_env(base, 5, 100, seed=3).checkpoint_layout().config_tag == src.checkpoint_layout().config_tag


def _corrupt(cfg, env, rows):
    """corrupt rows 2, 5, 9 at the offsets include/ssd_b200.h documents"""
    n = cfg["n"]
    r = rows.clone()
    if cfg["fam"] == "grid":
        r[2, 0] = env.H                                  # agent 0 row off the map
        r[5, 4 + 1] = env.W + 3                          # agent 1 column off the map
        r[9, 8 + 2] = 5                                  # agent 2 orientation > 3
    elif cfg["fam"] == "feat":
        r[2, 32:36] = torch_u32(300)                     # apple list length above capacity
        r[5, 0] = env.H                                  # agent 0 off the map
        r[9, 36:40] = torch_u32(200)                     # waste list length above capacity
    else:
        meta, crossed = 16 * n + 28, 16 * n + 24
        r[2, meta] = 1
        r[2, crossed:crossed + 4] = torch_u32(n)         # crossing-order entry >= n
        r[5, meta] = n + 1                               # n_crossed > n
        r[9, meta] = 2
        r[9, crossed:crossed + 4] = torch_u32(0x0F1)     # second entry 15
    return r


def torch_u32(v):
    import torch
    return torch.as_tensor(np.array([v], dtype="<u4").view(np.uint8).copy())


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cleanup8", "feat_cleanup8", "car8"])
def test_restore_rejects_corrupt_rows(oracle_lib, name):
    """Rows of the handle's CURRENT state (in lockstep with the oracle), three of them corrupted: restore names exactly
    those rows, the handle's state is byte for byte what it was, and it is still in lockstep with the oracle."""
    from contracts_b200 import _lib
    from contracts_b200.checkpoint import EnvCheckpoint
    cfg = CONFIGS[name]
    E = 16
    env, orc = _make_env(cfg, E, 2), _make_oracle(oracle_lib, cfg, E, 2)
    _same("reset obs", _np(env.reset()), orc.reset(), name)
    rng = np.random.RandomState(4)
    _lockstep(env, orc, cfg, rng, 12, name)
    ck = env.checkpoint()
    bad = EnvCheckpoint(ck.kind, ck.config_tag, ck.row_bytes, ck.seed, ck.env_ids, _corrupt(cfg, env, ck.rows.cpu()).cuda(), ck.obs)
    with pytest.raises(_lib.SsdError, match=r"rows \[2, 5, 9\] failed validation"):
        env.restore(bad)
    _same("rows after the rejected restore", _np(env.checkpoint(with_obs=False).rows), _np(ck.rows), name)
    _lockstep(env, orc, cfg, rng, 30, name + " after rejected restore")


@pytest.mark.gpu
def test_full_size_restore():
    """E = 131072 cleanup n=8: checkpoint, restore into a second handle, 20 identical steps (compared on the device)."""
    import torch
    cfg = CONFIGS["cleanup8"]
    E = 131072
    a = _make_env(cfg, E)
    a.reset()
    for t in range(5):
        a.step(a.random_actions(t, 9), auto_reset=True)
    ck = a.checkpoint()
    b = _make_env(cfg, E)
    b.restore(ck)
    assert torch.equal(a.obs, b.obs)
    for t in range(5, 25):
        act = a.random_actions(t, 9)
        a.step(act, auto_reset=True)
        b.step(act, auto_reset=True)
        for k in ("obs", "rew", "base_rew", "transfers", "info", "done"):
            x, y = getattr(a, k), getattr(b, k)
            assert torch.equal(x.view(torch.uint8) if x.dtype != torch.uint8 else x,
                               y.view(torch.uint8) if y.dtype != torch.uint8 else y), "step %d %s" % (t, k)
    assert torch.equal(a.checkpoint(with_obs=False).rows, b.checkpoint(with_obs=False).rows)

"""GPU: size-independent properties at the full benchmark size (BASELINE configs: 131072 envs x 8 agents cleanup,
16384 envs x 4 agents harvest), and the whole batch against the CPU oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PALETTE = {(0, 0, 0), (180, 180, 180), (0, 255, 0), (99, 156, 194), (113, 75, 24), (0, 0, 255), (2, 81, 154),
           (204, 0, 204), (216, 30, 54), (254, 151, 0), (100, 255, 255), (99, 99, 255), (250, 204, 255)}
AGENT_RGB = [(0, 0, 255), (2, 81, 154), (204, 0, 204), (216, 30, 54), (254, 151, 0), (100, 255, 255), (99, 99, 255),
             (250, 204, 255)]


@pytest.mark.parametrize("kind,E,n,nact,contract", [("cleanup", 131072, 8, 9, "CleanupContract"),
                                                    ("harvest", 16384, 4, 8, "HarvestFeaturemodLocalContract")])
def test_full_size_rollout_properties(oracle_lib, kind, E, n, nact, contract):
    import torch
    from contracts_b200.batched import BatchedGridEnv
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    amap = CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP
    big = BatchedGridEnv(kind + "_new", E, n, horizon=40, contract=contract, seed=73907)
    k0, ks = E - 77, 64                                   # a slice near the end of the batch
    small = BatchedGridEnv(kind + "_new", ks, n, horizon=40, contract=contract, seed=73907, first_env_id=k0)
    orc = oracle_lib.GridOracle(kind, ks, n, amap, horizon=40, contract=contract, seed=73907, first_env_id=k0)
    orc_big = oracle_lib.GridOracle(kind, E, n, amap, horizon=40, contract=contract, seed=73907)      # every env of the batch
    ob, osm = big.reset(), small.reset()
    assert torch.equal(ob[k0:k0 + ks], osm)
    assert np.array_equal(osm.cpu().numpy(), orc.reset())
    assert torch.equal(ob, torch.from_numpy(orc_big.reset()).to(ob.device))
    cleaned_total = torch.zeros((), dtype=torch.float64, device=big.device)
    for t in range(90):                                    # crosses the horizon twice (masked re-resets)
        a = big.random_actions(t, nact)
        a_small = small.random_actions(t, nact)
        assert torch.equal(a[k0:k0 + ks], a_small)        # actions are keyed by the global env id too
        obs, rew, done, info = big.step(a)
        o2, r2, d2, i2 = small.step(a_small)
        # 1. sharding invariance: a slice of the big batch == a small handle with the same global ids == the oracle
        assert torch.equal(obs[k0:k0 + ks], o2) and torch.equal(rew[k0:k0 + ks], r2) and torch.equal(info[k0:k0 + ks], i2)
        o = orc.step(a_small.cpu().numpy(), want_features=False)
        assert np.array_equal(o2.cpu().numpy(), o["obs"]) and np.array_equal(r2.cpu().numpy().view(np.uint64), o["rew"].view(np.uint64))
        # 1b. the whole batch == the oracle (a skipped or doubled env anywhere in the observe kernel's schedule)
        ob_ = orc_big.step(a.cpu().numpy(), want_features=False)
        for name, got, want in (("obs", obs, ob_["obs"]), ("rew", rew.view(torch.int64), ob_["rew"].view(np.int64)),
                                ("base_rew", big.base_rew.view(torch.int64), ob_["base_rew"].view(np.int64)),
                                ("transfers", big.transfers.view(torch.int64), ob_["transfers"].view(np.int64)),
                                ("info", info[..., :3].to(torch.int32), ob_["info"][..., :3]), ("done", done, ob_["done"])):
            bad = (got != torch.from_numpy(np.ascontiguousarray(want)).to(got.device)).reshape(E, -1).any(1).nonzero().flatten()
            assert bad.numel() == 0, "%s differs from the oracle at step %d in %d envs, first %r" % (name, t, bad.numel(), bad[:10].tolist())
        # 2. transfers redistribute, they do not create reward
        assert float((rew.sum(1) - big.base_rew.sum(1)).abs().max()) < 1e-9
        if kind == "cleanup":
            cleaned_total += info[:, :, 1].sum()
        if t % 30 == 0:
            # 3. every pixel is a palette colour; the centre pixel of agent i is an agent colour >= its own index
            px = obs[::97].reshape(-1, 3).cpu().numpy()
            assert {tuple(p) for p in np.unique(px, axis=0)} <= PALETTE
            centre = obs[::97, :, 7, 7, :].cpu().numpy()
            for i in range(n):
                allowed = set(AGENT_RGB[i:n])
                assert {tuple(p) for p in np.unique(centre[:, i], axis=0)} <= allowed
        if bool(done.any()):
            assert bool(done.all())                        # equal horizons
            ob = big.reset(done)
            small.reset(d2)
            orc.reset(d2.cpu().numpy())
            assert torch.equal(ob, torch.from_numpy(orc_big.reset(done.cpu().numpy())).to(ob.device))   # all envs are done
            cleaned_total.zero_()
    m = big.metrics_raw()
    assert float(m[:, 5].max()) == 0.0                     # no device error flags
    assert np.array_equal(m.cpu().numpy().view(np.uint64), orc_big.metrics_raw().view(np.uint64))
    so, sc = orc_big.get_state(), big.get_state()
    for k in ("map", "pos", "ori", "t", "theta"):
        assert np.array_equal(np.asarray(sc[k].cpu().numpy(), dtype=so[k].dtype), so[k]), k
    if kind == "cleanup":
        assert float(m[:, 4].sum()) == float(cleaned_total)          # dirt_cleaned == sum of cleaned_squares infos
        st = big.get_state()
        assert int((st["map"] == ord("H")).sum()) > 0
    # 4. state round trip: get_state -> set_state on a fresh handle reproduces the next step
    st = small.get_state()
    clone = BatchedGridEnv(kind + "_new", ks, n, horizon=40, contract=contract, seed=73907, first_env_id=k0)
    clone.reset()
    for _ in range(10):                                    # bring the clone's episode counter / t in line
        pass
    clone.set_state(map=st["map"], pos=st["pos"], ori=st["ori"], t=st["t"], theta=st["theta"])
    st2 = clone.get_state()
    for k in ("map", "pos", "ori", "t", "theta"):
        assert torch.equal(st[k], st2[k]), k


def test_step_host_equals_step(logic_variant):
    """ssd_step_host (host buffers, overlapped D2H copy) produces exactly what ssd_step + explicit copies produce."""
    import torch
    from contracts_b200.batched import BatchedGridEnv
    for kind, contract, nact in (("cleanup_new", "CleanupContract", 8), ("harvest_new", "HarvestFeaturemodLocalContract", 8)):
        E, n = 300, 5
        a = BatchedGridEnv(kind, E, n, contract=contract, seed=12, first_env_id=40, horizon=25)
        b = BatchedGridEnv(kind, E, n, contract=contract, seed=12, first_env_id=40, horizon=25)
        a.reset(); b.reset()
        rng = np.random.RandomState(0)
        rew_h = torch.empty((E, n), dtype=torch.float64).pin_memory()
        done_h = torch.empty((E,), dtype=torch.uint8).pin_memory()
        for t in range(30):
            acts = torch.as_tensor(rng.randint(0, nact, size=(E, n)).astype(np.uint8)).pin_memory()
            obs_a, rew_a, done_a, _ = a.step(acts.cuda())
            obs_b, _, _ = b.step_host(acts, rew_h, done_h)
            assert torch.equal(obs_a.cpu(), obs_b.cpu()), (kind, t)
            assert np.array_equal(rew_a.cpu().numpy().view(np.uint64), rew_h.numpy().view(np.uint64)), (kind, t)
            assert torch.equal(done_a.cpu(), done_h), (kind, t)
            if done_h.any():
                a.reset(done_a); b.reset(done_h.cuda())


@pytest.mark.parametrize("kind,contract,E,n,theta", [("cleanup_new", "CleanupContract", 3000, 8, 0.15),
                                                     ("cleanup_new", "CleanupContract", 700, 5, 0.0),
                                                     ("harvest_new", "HarvestFeaturemodLocalContract", 2000, 4, 2.5),
                                                     ("cleanup_new", None, 500, 3, 0.0)])
def test_step_host_async_equals_step(logic_variant, kind, contract, E, n, theta):
    """ssd_step_host_async / _wait (double-buffered slots, compact int8 + sparse float64 result block, predicted copy
    size) delivers bit for bit what ssd_step produces: observations, dones, and — after ssd_host_result_expand — the
    float64 rewards.  Two steps are kept in flight, as the pipelined caller does."""
    import torch
    from contracts_b200.batched import BatchedGridEnv
    a = BatchedGridEnv(kind, E, n, contract=contract, seed=5, first_env_id=11, horizon=60)
    b = BatchedGridEnv(kind, E, n, contract=contract, seed=5, first_env_id=11, horizon=60)
    a.reset(); b.reset()
    if contract:
        a.set_contract_params(theta); b.set_contract_params(theta)
    rng = np.random.RandomState(1)
    nact = 9 if kind == "cleanup_new" else 8
    acts = [torch.as_tensor(rng.randint(0, nact, size=(E, n)).astype(np.uint8)).pin_memory() for _ in range(70)]
    res = [b.new_host_result(), b.new_host_result()]
    want = []
    for t in range(70):
        obs_a, rew_a, done_a, _ = a.step(acts[t].cuda())
        want.append((rew_a.cpu().numpy().copy(), done_a.cpu().numpy().copy(), obs_a.cpu().numpy().copy() if t % 23 == 0 else None))
        if done_a.any():
            a.reset(done_a)
            if contract:
                a.set_contract_params(theta)
    tickets, sparse_total = [], 0
    def check(t):
        nonlocal sparse_total
        b.step_host_wait(tickets[t])
        r = res[t & 1]
        assert np.array_equal(r.rewards().view(np.uint64), want[t][0].view(np.uint64)), (kind, t)
        assert np.array_equal(r.done, want[t][1]), (kind, t)
        # the compact form itself: int8 where it says so, records exactly for the other envs, each env once
        envs = r.rec_env[:r.count]
        assert len(np.unique(envs)) == r.count
        w = want[t][0]
        fits = (w == np.round(w)) & (np.abs(w) <= 127) & ~(np.signbit(w) & (w == 0))
        sparse_env = np.nonzero(~fits.all(1))[0]
        assert np.array_equal(np.sort(envs), sparse_env), (kind, t)
        sparse_total += r.count
    for t in range(70):
        tickets.append(b.step_host_async(acts[t], res[t & 1]))
        if want[t][2] is not None:                      # observations are on the device, stream-ordered after the step
            assert np.array_equal(b.obs.cpu().numpy(), want[t][2]), (kind, t)
        if want[t][1].any():                            # device-side masked reset, stream-ordered, no host round trip
            b.reset(b.done)
            if contract:
                b.set_contract_params(theta)
        if t >= 1:
            check(t - 1)
    check(69)
    if contract and theta:
        assert sparse_total > 0                         # transfers were paid: the record path was exercised
    else:
        assert sparse_total == 0
    # a slot that has not been waited for cannot be resubmitted
    from contracts_b200 import _lib
    t0 = b.step_host_async(acts[0], res[0]); t1 = b.step_host_async(acts[1], res[1])
    with pytest.raises(_lib.SsdError):
        b.step_host_async(acts[2], res[0])
    b.step_host_wait(t0); b.step_host_wait(t1)


def test_step_host_async_prefix_miss():
    """The copied record prefix is predicted from the previous steps; when a step suddenly has far more records than
    predicted (contract switched on for every env), ssd_step_host_wait fetches the remainder."""
    import torch
    from contracts_b200.batched import BatchedGridEnv
    E, n = 40000, 8
    b = BatchedGridEnv("cleanup_new", E, n, contract="CleanupContract", seed=2, horizon=1000)
    a = BatchedGridEnv("cleanup_new", E, n, contract="CleanupContract", seed=2, horizon=1000)
    a.reset(); b.reset()
    a.set_contract_params(0.0); b.set_contract_params(0.0)
    res = [b.new_host_result(), b.new_host_result()]
    rng = np.random.RandomState(3)
    for t in range(6):
        if t == 3:
            a.set_contract_params(0.1); b.set_contract_params(0.1)
        acts = torch.full((E, n), 7, dtype=torch.uint8).pin_memory() if t >= 2 else \
            torch.as_tensor(rng.randint(0, 7, size=(E, n)).astype(np.uint8)).pin_memory()
        _, rew_a, _, _ = a.step(acts.cuda())
        tk = b.step_host_async(acts, res[t & 1])
        b.step_host_wait(tk)
        assert np.array_equal(res[t & 1].rewards().view(np.uint64), rew_a.cpu().numpy().view(np.uint64)), t
        if t == 3:
            assert res[t & 1].count > 1024 + 2 * 0        # more records than the predicted prefix (1024 after quiet steps)


def test_masked_negotiate_and_episode_stats(oracle_lib):
    """Steady-state sampler pieces: reset(mask) + negotiate(mask) touch only the masked envs, and the episode
    statistics accumulated at reset equal the per-env metrics summed on the host."""
    import torch
    from contracts_b200.batched import BatchedGridEnv
    E, n = 512, 8
    env = BatchedGridEnv("cleanup_new", E, n, contract="CleanupContract", seed=9, horizon=30)
    stats = torch.zeros(8, dtype=torch.float64, device=env.device)
    env.set_episode_stats(stats)
    env.reset()
    assert float(stats.abs().sum()) == 0.0                # first resets replace nothing
    theta0 = env.get_state()["theta"].clone()
    mask = (torch.arange(E, device=env.device) % 3 == 0).to(torch.uint8)
    prop = torch.full((E,), 0.125, dtype=torch.float64, device=env.device)
    acc = torch.ones((E, n), dtype=torch.float64, device=env.device)
    dec = env.negotiate(prop, acc, mask=mask)
    th = env.get_state()["theta"]
    assert torch.equal(th[mask == 0], theta0[mask == 0])
    assert bool((th[mask == 1] == 0.125).all()) and bool((dec[mask == 1] == 1).all()) and bool((dec[mask == 0] == 0).all())
    full = BatchedGridEnv("cleanup_new", E, n, contract="CleanupContract", seed=9, horizon=30)
    full.reset()
    dec_full = full.negotiate(prop, torch.full((E, n), 0.5, dtype=torch.float64, device=env.device))
    dec_m = env.negotiate(prop, torch.full((E, n), 0.5, dtype=torch.float64, device=env.device), mask=mask)
    assert torch.equal(dec_m[mask == 1], dec_full[mask == 1])        # the same draw, masked or not
    want = np.zeros(8)
    for t in range(30):
        env.step(env.random_actions(t, 9))
    m = env.metrics_raw().cpu().numpy()
    sel = mask.cpu().numpy() == 1
    want[:] = [m[sel, 0].sum(), m[sel, 2].sum(), m[sel, 3].sum(), m[sel, 4].sum(), m[sel, 40:48].sum(), m[sel, 24:32].sum(),
               sel.sum(), m[sel, 5].max()]
    obs_before = env.obs.clone()
    env.reset(mask)
    got = stats.cpu().numpy()
    assert np.allclose(got, want, rtol=1e-12, atol=1e-9) and got[6] == sel.sum() and got[0] == want[0] and got[3] == want[3]
    assert torch.equal(env.obs[mask == 0], obs_before[mask == 0])    # untouched envs keep their observation
    st = env.get_state()
    assert bool((st["t"][mask == 1] == 0).all()) and bool((st["t"][mask == 0] == 30).all())
    env.set_episode_stats(None)
    env.reset()
    assert np.array_equal(stats.cpu().numpy(), got)


def test_handle_on_non_current_device():
    """A handle bound to cuda:1 works while cuda:0 is current, and no entry point changes the caller's device."""
    import torch
    from contracts_b200.batched import BatchedGridEnv
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    torch.cuda.set_device(0)
    e1 = BatchedGridEnv("cleanup_new", 64, 4, contract="CleanupContract", seed=3, device="cuda:1")
    e0 = BatchedGridEnv("cleanup_new", 64, 4, contract="CleanupContract", seed=3, device="cuda")
    assert e0.device.index == 0 and torch.cuda.current_device() == 0
    o1, o0 = e1.reset(), e0.reset()
    for t in range(20):
        a0 = e0.random_actions(t, 9)
        r1 = e1.step(a0.to("cuda:1"))
        r0 = e0.step(a0)
        assert torch.cuda.current_device() == 0
        assert torch.equal(r1[0].cpu(), r0[0].cpu()) and torch.equal(r1[1].cpu(), r0[1].cpu())
    e1.close(); e0.close()
    assert torch.cuda.current_device() == 0


@pytest.mark.parametrize("kind,contract,n,negotiate", [("cleanup_new", "CleanupContract", 8, True), ("cleanup_new", "CleanupContract", 3, False),
                                                       ("harvest_new", "HarvestFeaturemodLocalContract", 4, True),
                                                       ("cleanup_new", None, 5, False)])
def test_auto_reset_equals_step_reset_negotiate(logic_variant, kind, contract, n, negotiate):
    """ssd_step_io.auto_reset (finished envs restart — and negotiate — inside the step) leaves exactly the state, outputs
    and episode statistics that step + reset(mask = done) + negotiate(mask = done) leave.  Horizons are staggered through
    set_state(t) so that a few envs finish in every step, as in a vectorised sampler's steady state."""
    import torch
    from contracts_b200.batched import BatchedGridEnv
    E, H = 900, 23
    a = BatchedGridEnv(kind, E, n, contract=contract, seed=31, first_env_id=5, horizon=H)
    b = BatchedGridEnv(kind, E, n, contract=contract, seed=31, first_env_id=5, horizon=H)
    sa, sb = (torch.zeros(8, dtype=torch.float64, device=a.device) for _ in range(2))
    a.set_episode_stats(sa); b.set_episode_stats(sb)
    a.reset(); b.reset()
    t0 = (torch.arange(E, device=a.device) % H).to(torch.int32)
    a.set_state(t=t0); b.set_state(t=t0)
    gen = torch.Generator(device=a.device); gen.manual_seed(1)
    nact = 9 if kind == "cleanup_new" else 8
    dec_a = torch.zeros(E, dtype=torch.uint8, device=a.device); dec_b = torch.zeros_like(dec_a)
    resets = 0
    for t in range(3 * H):
        prop = torch.rand(E, dtype=torch.float64, device=a.device, generator=gen) * 0.2
        acc = torch.rand((E, n), dtype=torch.float64, device=a.device, generator=gen) * 0.5 + 0.5
        act = a.random_actions(t, nact)
        oa, ra, da, ia = a.step(act)
        if bool(da.any()):
            oa = a.reset(da)
            if negotiate:
                a.negotiate(prop, acc, mask=da, out=dec_a)
        ob, rb, db, ib = b.step(act, auto_reset=True, negotiation=(prop, acc, dec_b) if negotiate else None)
        resets += int(da.sum())
        ctx = (kind, t)
        assert torch.equal(da, db) and int(da.sum()) > 0, ctx
        assert torch.equal(oa, ob), ctx
        assert torch.equal(ra.view(torch.int64), rb.view(torch.int64)) and torch.equal(ia, ib), ctx
        assert torch.equal(a.base_rew.view(torch.int64), b.base_rew.view(torch.int64)), ctx
        sta, stb = a.get_state(), b.get_state()
        for k in sta:
            assert torch.equal(sta[k], stb[k]), (k,) + ctx
        if negotiate:
            assert torch.equal(dec_a, dec_b), ctx
    assert resets > 2 * E
    assert torch.equal(a.metrics_raw(), b.metrics_raw())
    got_a, got_b = sa.cpu().numpy(), sb.cpu().numpy()
    assert got_a[6] == got_b[6] == resets
    assert np.allclose(got_a, got_b, rtol=1e-12, atol=1e-9)          # float64 atomics: order-dependent in the last bits
    assert np.array_equal(got_a[[0, 3, 6, 7]], got_b[[0, 3, 6, 7]])   # integer-valued statistics are exact


@pytest.mark.gpu
def test_null_contract_probability_matches_oracle(oracle_lib):
    """null_prob > 0 (SeparateContractSubgameStage.reset, two_stage_train.py:159-166): the null / drawn contract parameter of
    every env and episode, grid worlds, feature envs and selfdrive, against the oracle (pinned to the live reference by
    test_deep_differential.py::test_reference_vs_oracle_null_contract_probability)."""
    import torch
    from contracts_b200.batched import BatchedGridEnv
    from contracts_b200.features import BatchedFeatureEnv
    from contracts_b200.selfdrive import BatchedCarEnv
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    E, null_prob = 300, 0.45
    pairs = [
        (BatchedGridEnv("cleanup_new", E, 4, contract="CleanupContract", null_prob=null_prob, seed=3, first_env_id=9),
         oracle_lib.GridOracle("cleanup", E, 4, CLEANUP_MAP, contract="CleanupContract", null_prob=null_prob, seed=3, first_env_id=9)),
        (BatchedFeatureEnv("harvest", E, 5, contract="HarvestFeaturemodLocalContract", null_prob=null_prob, seed=4, first_env_id=2),
         oracle_lib.FeatOracle("harvest", E, 5, HARVEST_MAP, contract="HarvestFeaturemodLocalContract", null_prob=null_prob, seed=4,
                               first_env_id=2)),
        (BatchedCarEnv(E, 6, contract="SelfdriveContractDistprop", null_prob=null_prob, seed=5, first_env_id=1),
         oracle_lib.CarOracle(E, 6, contract="SelfdriveContractDistprop", null_prob=null_prob, seed=5, first_env_id=1)),
    ]
    for env, orc in pairs:
        for ep in range(3):
            env.reset(); orc.reset()
            got, want = env.get_state()["theta"].cpu().numpy(), orc.get_state()["theta"]
            assert np.array_equal(got.view(np.uint64), np.asarray(want, dtype=np.float64).view(np.uint64)), \
                "%s episode %d: theta differs from the oracle" % (type(env).__name__, ep)
            nulls = int((want == 0).sum())
            assert 0.3 * E < nulls < 0.6 * E, nulls
        env.close()

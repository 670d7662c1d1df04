"""GPU: the solver queue of a vectorised sampler (contracts_b200/solver.py, ssd_solver_rows / ssd_solver_resolve).

The twin tests step two identical batches: A with auto-reset and the queue (rows -> value function -> resolve), B with the
route that existed before it (sample all E envs, build every row in torch, ssd_solver_choose, then restore the theta of
the envs that did not restart).  Everything either batch returns must be equal bit for bit.
(Named to sort after test_cuda_kernel_variants.py, whose profiler records must not see this file's kernels.)"""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

S = 6
E_ODD = 37
HORIZON = 7


def _make(kind, E=E_ODD, dtype=None, image_obs=True, seed=4242, first_env_id=5):
    if kind in ("cleanup_new", "harvest_new"):
        from contracts_b200.batched import BatchedGridEnv
        contract = "CleanupContract" if kind == "cleanup_new" else "HarvestFeaturemodLocalContract"
        n = 5 if kind == "cleanup_new" else 4
        return BatchedGridEnv(kind, E, n, horizon=HORIZON, contract=contract, seed=seed, first_env_id=first_env_id,
                              policy_dtype=dtype, image_obs=image_obs, device="cuda:0")
    if kind in ("cleanup", "harvest"):
        from contracts_b200.features import BatchedFeatureEnv
        contract = "CleanupContract" if kind == "cleanup" else "HarvestFeaturemodLocalContract"
        return BatchedFeatureEnv(kind, E, 3, horizon=HORIZON, contract=contract, seed=seed, first_env_id=first_env_id,
                                 policy_dtype=dtype, device="cuda:0")
    from contracts_b200.selfdrive import BatchedCarEnv
    return BatchedCarEnv(E, 3, contract="SelfdriveContractDistprop", seed=seed, first_env_id=first_env_id, policy_dtype=dtype,
                         start_vel=1.5, start_vel_ambulance=2.0, device="cuda:0")


def _actions(env, step):
    if env.kind == "selfdrive":
        return env.random_actions(step, -0.1, 0.1)
    return env.random_actions(step, 8 if env.kind in ("cleanup_new", "cleanup") else 7)


def _theta_t(env):
    st = env.get_state()
    return st["theta"], st["t"]


def _image_feat(env, index):
    """a deterministic number per gathered (env, agent) image: the first 8 values of its observation, weighted"""
    src = env.obs.view(env.E * env.n, -1) if env.policy_dtype is None else env.policy_image.view(env.E * env.n, -1)
    img = src[index]
    acc = torch.zeros(img.shape[0], dtype=torch.float64, device=img.device)
    for j in range(8):
        acc = acc + img[:, j].double() * (0.25 + 0.125 * j)
    return acc


def value_fn(rows, img=None):
    """a deterministic value per row [M, 1 + S, n, W] (+ the per-(env, agent) image feature [M, n]): element-wise ops only,
    so a row's value does not depend on the batch it is in"""
    acc = torch.zeros(rows.shape[:3], dtype=torch.float64, device=rows.device)
    for j in range(rows.shape[3]):
        acc = acc + rows[..., j].double() * (0.5 + 0.1 * j)
    if img is not None:
        acc = acc + img[:, None, :]
    agent = torch.arange(rows.shape[2], dtype=torch.float64, device=rows.device)
    return torch.sin(acc * 13.0 + agent * 0.7)


def _queue_vals(env, out):
    rows = out[0]
    img = None
    if len(out) == 4:
        img = _image_feat(env, out[3]).view(-1, env.n)
    return value_fn(rows, img)


def _all_rows(env, params):
    """today's route: the value-query rows of every env, built in torch ([E, 1 + S, n, W])"""
    E, n, S1 = env.E, env.n, params.shape[1]
    p = params[:, :, None, None].expand(E, S1, n, 1)
    image = getattr(env, "image_obs", False)
    if image:
        if env.policy_dtype is None:
            return torch.cat((p, torch.zeros_like(p)), -1)
        T = env.policy_dtype
        pt = p.float().to(T)
        return torch.cat((pt, torch.zeros_like(pt)), -1).repeat(1, 1, 1, 5)
    if env.policy_dtype is None:
        obs = env.obs[:, None].expand(E, S1, n, env.obs.shape[-1])
        return torch.cat((obs, p, torch.zeros_like(p)), -1)
    W = env.policy_width
    T = env.policy_dtype
    feat = env.policy_obs.view(E, n, W)[:, None, :, :W - 2].expand(E, S1, n, W - 2)
    pt = p.float().to(T)
    return torch.cat((feat, pt, torch.zeros_like(pt)), -1)


def _all_vals(env, rows):
    img = None
    if getattr(env, "image_obs", False):
        idx = torch.arange(env.E * env.n, device=rows.device)
        img = _image_feat(env, idx).view(env.E, env.n)
    return value_fn(rows, img)


def _old_route(env, mask):
    """sample all, value all, choose all, restore the theta of the envs outside `mask` (bool [E])"""
    theta0, _ = _theta_t(env)
    from contracts_b200.batched import solver_choose, solver_sample
    params = solver_sample(env, S)
    rows = _all_rows(env, params)
    best, _ = solver_choose(env, params, _all_vals(env, rows), "majority")
    env.set_contract_params(torch.where(mask, best, theta0))
    return params, rows


def _same(a, b, what):
    a, b = a.contiguous(), b.contiguous()
    assert a.shape == b.shape, what
    assert torch.equal(a.view(torch.uint8) if a.dtype != torch.bool else a, b.view(torch.uint8) if b.dtype != torch.bool else b), what


def _compare_window(qa, out, params_b, rows_b, pending_mask, what):
    cnt, total = [int(x) for x in qa.count.tolist()]
    want = torch.nonzero(pending_mask).flatten()
    assert total == want.numel(), what
    assert cnt == min(total, qa.C), what
    env_ids = qa.env[:cnt].long()
    _same(env_ids, want[:cnt], what + ": window envs")
    assert bool((qa.env[cnt:] == -1).all()), what
    _same(qa.params[:cnt], params_b[env_ids], what + ": candidates")
    _same(out[0][:cnt], rows_b[env_ids], what + ": rows")
    assert not bool(out[0][cnt:].view(torch.uint8).any()), what + ": rows beyond the window"


def _outputs(env):
    out = [env.observation, env.rew, env.done]
    if env.kind != "selfdrive":
        out.append(env.info)
    if getattr(env, "policy_contract", None) is not None:      # the policy image's contract rows
        out.append(env.policy_contract)
    return out


FORMS = [("cleanup_new", None, True), ("cleanup_new", torch.bfloat16, True), ("harvest_new", None, False),
         ("cleanup_new", torch.bfloat16, False)]


def _twin(kind, dtype, image_obs, steps):
    from contracts_b200.solver import SolverQueue
    kw = dict(dtype=dtype) if kind in ("cleanup", "harvest", "selfdrive") else dict(dtype=dtype, image_obs=image_obs)
    A, B = _make(kind, **kw), _make(kind, **kw)
    q = SolverQueue(A, num_samples=S, capacity=A.E)
    A.reset()
    B.reset()
    def solve(what):
        """A: the queue; B: today's route on the envs at t == 0; then everything must agree"""
        _, tb = _theta_t(B)
        pend = tb == 0
        out = q.rows()
        params_b, rows_b = _old_route(B, pend)
        _compare_window(q, out, params_b, rows_b, pend, what)
        q.resolve(_queue_vals(A, out))
        assert int(q.stale.item()) == 0, what
        _same(_theta_t(A)[0], _theta_t(B)[0], what + ": theta")
        for x, y in zip(_outputs(A), _outputs(B)):                   # the theta rows / columns of the observation too
            _same(x, y, what + ": outputs after resolve")

    solve("%s initial" % kind)
    assert q.pending() == 0
    for s in range(steps):
        a = _actions(A, s)
        A.step(a, auto_reset=True)
        B.step(a, auto_reset=True)
        for x, y in zip(_outputs(A), _outputs(B)):
            _same(x, y, "%s step %d outputs" % (kind, s))
        if s < HORIZON and kind != "selfdrive":       # stagger the episodes over the first horizon
            m = (torch.arange(A.E, device="cuda") % HORIZON == s).to(torch.uint8)
            A.reset(m)
            B.reset(m)
        solve("%s step %d" % (kind, s))
    A.close()
    B.close()


@pytest.mark.parametrize("kind,dtype,image_obs", FORMS)
def test_twin_grid(kind, dtype, image_obs, logic_variant):
    _twin(kind, dtype, image_obs, 4 * HORIZON)


@pytest.mark.parametrize("kind", ["cleanup", "harvest"])
@pytest.mark.parametrize("dtype", [None, torch.bfloat16])
def test_twin_features(kind, dtype):
    _twin(kind, dtype, True, 4 * HORIZON)


@pytest.mark.parametrize("dtype", [None, torch.float32])
def test_twin_selfdrive(dtype):
    _twin("selfdrive", dtype, True, 60)


def test_window_matches_oracle(oracle_lib):
    """window entries' candidates and choices against the C oracle's solver_candidates / solver_choose"""
    from contracts_b200.solver import SolverQueue
    A = _make("harvest", E=29)
    q = SolverQueue(A, num_samples=S, capacity=11, rule="max")
    A.reset()
    for s in range(3 * HORIZON):
        if s:
            A.step(_actions(A, s), auto_reset=True)
        out = q.rows()
        vals = _queue_vals(A, out)
        theta, index = q.resolve(vals)
        cnt = int(q.count[0].item())
        ep, env_ids = q.episode.cpu().numpy().view(np.uint32), q.env.cpu().numpy()
        for c in range(cnt):
            want = oracle_lib.solver_candidates(A.seed, A.first_env_id + int(env_ids[c]), int(ep[c]), 0.0,
                                                float(np.float32(10.0)), S)
            assert np.array_equal(q.params[c].cpu().numpy().view(np.uint64), want.view(np.uint64))
            wt, wi = oracle_lib.solver_choose(want, vals[c].cpu().numpy(), "max")
            assert float(theta[c]) == float(wt) and int(index[c]) == int(wi)
    A.close()


def test_run_windows_equal_one_window():
    """after a full reset, run() with C = E / 7 gives every env the theta a single window of C = E gives it"""
    from contracts_b200.solver import SolverQueue
    E = 7 * 19 + 3
    A, B = _make("cleanup", E=E), _make("cleanup", E=E)
    qa, qb = SolverQueue(A, S, capacity=E // 7), SolverQueue(B, S, capacity=E)
    A.reset()
    B.reset()
    assert qa.pending() == E and qb.pending() == E
    f = lambda *out: value_fn(out[0])                       # noqa: E731
    assert qa.run(f) == E
    assert qb.run(f) == E
    assert qa.pending() == 0 and qb.pending() == 0
    _same(_theta_t(A)[0], _theta_t(B)[0], "theta")
    A.close()
    B.close()


def test_stale_entries():
    """a step or a reset between rows and resolve: index -1, theta unchanged, counted in stale"""
    from contracts_b200.solver import SolverQueue
    A = _make("cleanup", E=E_ODD)
    q = SolverQueue(A, S, capacity=16)
    A.reset()
    q.rows()
    th0, _ = _theta_t(A)
    A.step(_actions(A, 0))                                  # every env is at t = 1 now
    theta, index = q.resolve(value_fn(q.query_rows))
    assert bool((index == -1).all()) and int(q.stale.item()) == 16
    _same(theta, th0[q.env.long()], "stale theta")
    _same(_theta_t(A)[0], th0, "theta unchanged")
    # reset some window envs again between the calls: they are stale and stay pending
    A.reset()
    out = q.rows()
    m = torch.zeros(A.E, dtype=torch.uint8, device="cuda")
    m[q.env[:5].long()] = 1
    A.reset(m)
    theta, index = q.resolve(value_fn(out[0]))
    assert int(q.stale.item()) == 5
    assert bool((index[:5] == -1).all()) and bool((index[5:] >= 0).all())
    assert q.pending() == A.E - 11
    A.close()


def test_graph_equals_eager():
    """50 steps of (step, rows, value function, resolve) captured in one CUDA graph = the same steps eagerly"""
    from contracts_b200.solver import SolverQueue
    E = 61
    A, B = _make("harvest", E=E, dtype=torch.bfloat16), _make("harvest", E=E, dtype=torch.bfloat16)
    qa, qb = SolverQueue(A, S, capacity=16), SolverQueue(B, S, capacity=16)

    def substep(env, q):
        env.step(_actions(env, None), auto_reset=True)
        out = q.rows()
        q.resolve(value_fn(out[0]))

    for env, q in ((A, qa), (B, qb)):
        env.reset()
        q.run(lambda *out: value_fn(out[0]))
    for s in range(HORIZON):                                # staggered episodes
        m = (torch.arange(E, device="cuda") % HORIZON == s).to(torch.uint8)
        for env, q in ((A, qa), (B, qb)):
            env.reset(m)
            substep(env, q)
    main, cap = torch.cuda.current_stream(), torch.cuda.Stream()
    cap.wait_stream(main)
    with torch.cuda.stream(cap):
        for _ in range(3):
            substep(A, qa)
    main.wait_stream(cap)
    for _ in range(3):
        substep(B, qb)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=cap):
        for _ in range(50):
            substep(A, qa)
    g.replay()
    for _ in range(50):
        substep(B, qb)
    torch.cuda.synchronize()
    for x, y in zip(_outputs(A) + [qa.theta, qa.index, qa.env], _outputs(B) + [qb.theta, qb.index, qb.env]):
        _same(x, y, "graph vs eager")
    _same(_theta_t(A)[0], _theta_t(B)[0], "theta")
    del g
    A.close()
    B.close()


def test_checkpoint_restore_not_pending():
    """restored envs come back with their theta: not pending, whatever the destination's queue had seen"""
    from contracts_b200.solver import SolverQueue
    A, B = _make("cleanup", dtype=torch.float32), _make("cleanup", dtype=torch.float32)
    qa, qb = SolverQueue(A, S, capacity=A.E), SolverQueue(B, S, capacity=B.E)
    A.reset()
    qa.run(lambda *out: value_fn(out[0]))
    ck = A.checkpoint()
    B.reset()
    assert qb.pending() == B.E
    B.restore(ck)
    assert qb.pending() == 0
    _same(_theta_t(A)[0], _theta_t(B)[0], "theta")
    _same(A.policy_obs, B.policy_obs, "policy rows")
    A.reset()                                               # a new episode is pending again
    assert qa.pending() == A.E
    A.close()
    B.close()


def test_error_surface():
    from contracts_b200 import _lib
    from contracts_b200.solver import SolverQueue
    lib = _lib.load()
    from contracts_b200.features import BatchedFeatureEnv
    plain = BatchedFeatureEnv("cleanup", 5, 2, device="cuda:0")
    with pytest.raises(ValueError):
        SolverQueue(plain)
    assert lib.ssd_solver_enable(plain._h, 1) == -1                          # no contract
    plain.close()

    F = _make("cleanup")
    q = SolverQueue(F, S, capacity=4)
    st = lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)   # noqa: E731

    def win(**kw):
        w = _lib.ssd_solver_window()
        ctypes.memmove(ctypes.byref(w), ctypes.byref(q._win), ctypes.sizeof(w))
        for k, v in kw.items():
            setattr(w, k, v)
        return w

    obs = ctypes.c_void_p(F.obs.data_ptr())
    assert lib.ssd_solver_rows(F._h, ctypes.byref(win()), obs, st()) == 0
    for bad in (dict(struct_size=8), dict(capacity=0), dict(capacity=F.E + 1), dict(num_samples=-1),
                dict(params_dev=q.params.data_ptr() + 4), dict(env_dev=q.env.data_ptr() + 2), dict(count_dev=None),
                dict(rows_dev=q.query_rows.data_ptr() + 8)):
        assert lib.ssd_solver_rows(F._h, ctypes.byref(win(**bad)), obs, st()) == -1, bad
    assert lib.ssd_solver_rows(F._h, ctypes.byref(win()), None, st()) == -1                 # float64 form: obs required
    assert lib.ssd_solver_rows(F._h, ctypes.byref(win()), ctypes.c_void_p(F.obs.data_ptr() + 4), st()) == -1
    vals = torch.zeros((4, S + 1, F.n), dtype=torch.float64, device="cuda")
    vp = ctypes.c_void_p(vals.data_ptr())
    assert lib.ssd_solver_resolve(F._h, ctypes.byref(win()), 1, vp, None, None, None, st()) == 0
    assert lib.ssd_solver_resolve(F._h, ctypes.byref(win()), 7, vp, None, None, None, st()) == -1
    assert lib.ssd_solver_resolve(F._h, ctypes.byref(win()), 1, None, None, None, None, st()) == -1
    assert lib.ssd_solver_resolve(F._h, ctypes.byref(win()), 1, ctypes.c_void_p(vals.data_ptr() + 4), None, None, None, st()) == -1
    assert lib.ssd_solver_resolve(F._h, ctypes.byref(win(struct_size=4)), 1, vp, None, None, None, st()) == -1
    with pytest.raises(ValueError):
        q.resolve(torch.zeros((3, S + 1, F.n), dtype=torch.float64, device="cuda"))
    assert lib.ssd_solver_enable(F._h, 0) == 0
    assert lib.ssd_solver_rows(F._h, ctypes.byref(win()), obs, st()) == -1                   # queue off
    F.close()

    for dtype, image_obs in ((None, True), (torch.bfloat16, True), (None, False)):
        G = _make("cleanup_new", dtype=dtype, image_obs=image_obs)
        qg = SolverQueue(G, S, capacity=4)
        dummy = torch.zeros(8, dtype=torch.float64, device="cuda")
        assert lib.ssd_solver_rows(G._h, ctypes.byref(qg._win), ctypes.c_void_p(dummy.data_ptr()), st()) == -1  # obs given
        assert lib.ssd_solver_rows(G._h, ctypes.byref(qg._win), None, st()) == 0
        G.close()
    P = _make("selfdrive", dtype=torch.float32)
    qp = SolverQueue(P, S, capacity=4)
    dummy = torch.zeros(8, dtype=torch.float64, device="cuda")
    assert lib.ssd_solver_rows(P._h, ctypes.byref(qp._win), ctypes.c_void_p(dummy.data_ptr()), st()) == -1
    P.close()
    torch.cuda.synchronize()

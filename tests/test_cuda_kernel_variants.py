"""GPU: every template instantiation of the grid-world step's kernels against the C oracle.

The step is not one kernel: ssd_create / ssd_set_policy_output pick an observe, reset and logic kernel by env kind, point-list
size (4 or 8 mask rounds), feature_obs, layout specialisation and observation form.  VARIANTS lists configurations and
the instantiations each one launches; every row is rolled out once per observation form and compared bit for bit with
the oracle, and the profiler confirms that the row ran the kernels it names.  tests/test_kernel_variant_inventory.py
checks that the rows name every instantiation in the built library.

Policy forms are compared with the oracle's uint8 windows converted by torch ((x.double() / 255).float().to(T), NCHW) —
never with the library's own policy_inputs kernel."""
import collections
import re

import numpy as np
import pytest

import golden_util as gu
from test_cuda_vs_oracle import CRAMPED_CLEANUP, CRAMPED_HARVEST

pytestmark = pytest.mark.gpu

FORM_ID = {"u8": 0, "f32": 1, "f16": 2, "bf16": 3}       # the FORM template argument of the observe / reset kernels
ALL_FORMS = ("u8", "f32", "f16", "bf16")
CONTRACT = {"cleanup": "CleanupContract", "harvest": "HarvestFeaturemodLocalContract"}
KIND_ID = {"cleanup": 0, "harvest": 1}


def _obs(kind, mw, feat, lay):
    return "grid_obs_kernel<%d, %d, %s, %d, {F}>" % (KIND_ID[kind], mw, "true" if feat else "false", lay)


def _logic(kind, lay):
    return "grid_logic_kernel<%d, %d>" % (KIND_ID[kind], lay)


def _logic8(kind):
    return "grid_logic8_kernel<%d>" % KIND_ID[kind]


def _reset(kind):
    return "grid_reset_kernel<%d, {F}>" % KIND_ID[kind]


REWARD = "grid_reward_kernel"

Variant = collections.namedtuple("Variant", "name kind n map E first logic8 forms kernels")


def _generic(kind, mw, logic):
    """the kernels of a handle without a layout specialisation: the generic observe kernel with and without features"""
    return (logic, _obs(kind, mw, False, 0), _obs(kind, mw, True, 0), _reset(kind)) + ((REWARD,) if kind == "harvest" else ())


# kernels: what reset + a step without and a step with feature_obs launch ({F}: the form's FORM argument)
VARIANTS = [
    # stock cleanup, 8 agents: the layout-specialised logic and observe kernels (the benchmark's configuration)
    Variant("cleanup_n8_stock", "cleanup", 8, "stock", 64, 5, 0, ALL_FORMS,
            (_logic("cleanup", 1), _obs("cleanup", 4, False, 1), _obs("cleanup", 4, True, 0), _reset("cleanup"))),
    Variant("cleanup_n8_stock_octet", "cleanup", 8, "stock", 64, 5, 1, ALL_FORMS,
            (_logic8("cleanup"), _obs("cleanup", 4, False, 1), _obs("cleanup", 4, True, 0), _reset("cleanup"))),
    Variant("cleanup_n5_stock", "cleanup", 5, "stock", 48, 9, 0, ALL_FORMS, _generic("cleanup", 4, _logic("cleanup", 0))),
    Variant("cleanup_n8_cramped", "cleanup", 8, "cramped", 48, 0, 0, ALL_FORMS, _generic("cleanup", 4, _logic("cleanup", 0))),
    # > 128 apple / waste points: 8 mask rounds
    Variant("cleanup_n8_big44x60", "cleanup", 8, "big44x60", 24, 3, 0, ALL_FORMS, _generic("cleanup", 8, _logic("cleanup", 0))),
    Variant("cleanup_n3_big48x64_octet", "cleanup", 3, "big48x64", 24, 3, 1, ALL_FORMS, _generic("cleanup", 8, _logic8("cleanup"))),
    # stock harvest, 4 agents: the layout-specialised kernels (155 apples: 8 mask rounds)
    Variant("harvest_n4_stock", "harvest", 4, "stock", 64, 5, 0, ALL_FORMS,
            (_logic("harvest", 2), _obs("harvest", 8, False, 2), _obs("harvest", 8, True, 0), REWARD, _reset("harvest"))),
    Variant("harvest_n4_stock_octet", "harvest", 4, "stock", 64, 5, 1, ALL_FORMS,
            (_logic8("harvest"), _obs("harvest", 8, False, 2), _obs("harvest", 8, True, 0), REWARD, _reset("harvest"))),
    Variant("harvest_n3_stock", "harvest", 3, "stock", 40, 7, 0, ALL_FORMS, _generic("harvest", 8, _logic("harvest", 0))),
    Variant("harvest_n8_stock", "harvest", 8, "stock", 40, 0, 0, ALL_FORMS, _generic("harvest", 8, _logic("harvest", 0))),
    Variant("harvest_n6_big40x63", "harvest", 6, "big40x63", 24, 3, 0, ALL_FORMS, _generic("harvest", 8, _logic("harvest", 0))),
    # <= 128 apples: 4 mask rounds
    Variant("harvest_n8_cramped", "harvest", 8, "cramped", 48, 0, 0, ALL_FORMS, _generic("harvest", 4, _logic("harvest", 0))),
    Variant("harvest_n5_random_octet", "harvest", 5, "random", 48, 2, 1, ALL_FORMS, _generic("harvest", 4, _logic8("harvest"))),
] + [
    # agent counts of the policy forms: each n gives another chunk plan (agents per staged chunk, halfword head / tail
    # stores); an odd E puts env blocks at every even residue mod 16.  The half types share a plan: bf16 at n = 1 and 7 only.
    Variant("policy_cleanup_n%d" % n, "cleanup", n, "stock", 37, 11, 0, ("f32", "f16") + (("bf16",) if n in (1, 7) else ()),
            (_logic("cleanup", 1), _obs("cleanup", 4, False, 1), _obs("cleanup", 4, True, 0), _reset("cleanup")) if n == 8
            else _generic("cleanup", 4, _logic("cleanup", 0)))
    for n in range(1, 9)
] + [
    # one agent, no contract: no contract rows are written
    Variant("policy_harvest_n1", "harvest", 1, "stock", 37, 11, 0, ("f32", "f16", "bf16"), _generic("harvest", 8, _logic("harvest", 0))),
]


def variant_kernels(v, form):
    return {k.format(F=FORM_ID[form]) for k in v.kernels}


def _map(v):
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    if v.map == "stock":
        return CLEANUP_MAP if v.kind == "cleanup" else HARVEST_MAP
    if v.map == "cramped":
        return CRAMPED_CLEANUP if v.kind == "cleanup" else CRAMPED_HARVEST
    if v.map == "random":
        return gu.random_map(np.random.RandomState(8), v.kind, v.n)
    H, W = (int(x) for x in v.map[3:].split("x"))
    return gu.big_map(v.kind, H, W, H * W)


_GRID_KERNEL = re.compile(r"^(?:void )?(grid_(?:obs|reset|logic|logic8|reward)_kernel(?:<[^>]*>)?)")


def _launched(fn):
    """the grid-world kernels (as 'grid_obs_kernel<0, 8, true, 0, 2>') that fn launched, from the profiler's CUDA records"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()] + [k.name for e in prof.events() for k in getattr(e, "kernels", ())]
    launched = {m.group(1) for m in map(_GRID_KERNEL.match, names) if m}
    assert launched, "the profiler recorded no grid-world kernel (CUDA records: %r)" % sorted(set(names))[:20]
    return launched


def _contract_rows(theta, n, dtype):
    """(float32(theta), 0) x 5 per agent, T [E n, 10]"""
    import torch
    th = torch.from_numpy(np.asarray(theta, dtype=np.float64).astype(np.float32))
    rows = torch.stack([th, torch.zeros_like(th)] * 5, dim=1)
    return rows.to(dtype).repeat_interleave(n, dim=0)


def _equal(name, got, want, rows_per_env, ctx):
    """bit-exact comparison (every value is finite); names the first differing envs"""
    import torch
    assert got.shape == want.shape, "%s shape %r != %r at %s" % (name, tuple(got.shape), tuple(want.shape), ctx)
    if torch.equal(got, want):
        return
    bad = (got != want).reshape(got.shape[0] // rows_per_env, -1).any(1).nonzero().flatten().tolist()
    raise AssertionError("%s differs at %s in %d envs, first %r" % (name, ctx, len(bad), bad[:10]))


class Rollout:
    """One oracle and CUDA envs of the same configuration, one per observation form, driven with the same calls and
    compared with the oracle after each: observations (every env), rewards, base rewards, transfers, infos, dones,
    feature_obs, state, decisions, contract rows, and metrics (finish)."""

    def __init__(self, oracle_lib, kind, n, amap, E, first, forms, horizon, seed):
        import torch
        from contracts_b200.batched import BatchedGridEnv
        self.kind, self.n, self.E, self.horizon = kind, n, E, horizon
        self.contract = CONTRACT[kind] if n >= 2 else None
        self.nact = 9 if kind == "cleanup" else 8
        self.orc = oracle_lib.GridOracle(kind, E, n, amap, horizon=horizon, contract=self.contract, seed=seed, first_env_id=first)
        dtypes = {"u8": None, "f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}
        self.envs = [BatchedGridEnv(kind + "_new", E, n, amap, horizon=horizon, contract=self.contract, seed=seed, first_env_id=first,
                                    policy_dtype=dtypes[f]) for f in forms]
        self.forms = forms
        self.decs = [torch.zeros(E, dtype=torch.uint8, device="cuda") for _ in forms]
        self.rng = np.random.RandomState(seed)
        self.want = None                             # the oracle's current windows, uint8 [E, n, 15, 15, 3]
        self.finished = 0

    def actions(self):
        return self.rng.randint(0, self.nact, size=(self.E, self.n))

    def check_obs(self, ctx):
        import torch
        want = torch.from_numpy(self.want).cuda()
        theta = self.orc.get_state()["theta"] if self.contract else None
        for f, env in zip(self.forms, self.envs):
            if env.policy_dtype is None:
                _equal("obs", env.obs, want, 1, "%s %s" % (f, ctx))
                continue
            assert env.obs is None
            _equal("policy image", env.policy_image, gu.policy_image(want, env.policy_dtype), self.n, "%s %s" % (f, ctx))
            if self.contract:
                _equal("contract rows", env.policy_contract.cpu(), _contract_rows(theta, self.n, env.policy_dtype), self.n,
                       "%s %s" % (f, ctx))
            else:
                assert env.policy_contract is None

    def check_state(self, ctx):
        so = self.orc.get_state()
        for f, env in zip(self.forms, self.envs):
            sc = env.get_state()
            for k in ("map", "pos", "ori", "t", "theta"):
                gu.assert_same(k, sc[k].cpu().numpy(), so[k], "%s %s" % (f, ctx))

    def check_outputs(self, o, wf, ctx):
        for f, env in zip(self.forms, self.envs):
            c = "%s %s" % (f, ctx)
            gu.assert_same("rew", env.rew.cpu().numpy(), o["rew"], c)
            gu.assert_same("base_rew", env.base_rew.cpu().numpy(), o["base_rew"], c)
            gu.assert_same("transfers", env.transfers.cpu().numpy(), o["transfers"], c)
            gu.assert_same("info", env.info.cpu().numpy()[..., :3], o["info"][..., :3], c)
            gu.assert_same("done", env.done.cpu().numpy(), o["done"], c)
            if wf:
                gu.assert_same("feature_obs", env.feature_obs.cpu().numpy(), o["feature_obs"], c)

    def reset(self, mask=None, ctx="reset"):
        import torch
        m = None if mask is None else torch.as_tensor(mask.astype(np.uint8)).cuda()
        for env in self.envs:
            env.reset(m)
        r = self.orc.reset(mask)
        if mask is None:
            self.want = r
        else:
            self.want[mask.astype(bool)] = r[mask.astype(bool)]
        self.check_obs(ctx)
        self.check_state(ctx)

    def step(self, a, wf, ctx):
        import torch
        a_dev = torch.as_tensor(a.astype(np.uint8)).cuda()
        for env in self.envs:
            env.step(a_dev, want_features=wf)
        o = self.orc.step(a, want_features=wf)
        self.want = o["obs"]
        self.check_outputs(o, wf, ctx)
        self.check_obs(ctx)
        self.check_state(ctx)
        return o["done"]

    def set_t(self, t):
        import torch
        for env in self.envs:
            env.set_state(t=torch.as_tensor(t, dtype=torch.int32).cuda())
        self.orc.set_state(t=t)

    def auto_step(self, a, wf, ctx):
        """step(auto_reset=True, negotiation=...); on the oracle: step, reset(done), negotiate on every env, and theta of
        the finished envs from the negotiation (the agreement draw is the same masked or not)"""
        import torch
        prop, acc = self.rng.uniform(0.0, 0.2, self.E), self.rng.uniform(0.3, 1.0, (self.E, self.n))
        a_dev = torch.as_tensor(a.astype(np.uint8)).cuda()
        prop_d, acc_d = torch.as_tensor(prop).cuda(), torch.as_tensor(acc).cuda()
        for env, dec in zip(self.envs, self.decs):
            env.step(a_dev, want_features=wf, auto_reset=True, negotiation=(prop_d, acc_d, dec) if self.contract else None)
        o = self.orc.step(a, want_features=wf)
        done = o["done"].astype(bool)
        self.want = o["obs"]
        self.check_outputs(o, wf, ctx)
        if done.any():
            self.finished += int(done.sum())
            r = self.orc.reset(o["done"])
            self.want[done] = r[done]
            if self.contract:
                old = self.orc.get_state()["theta"]
                want_dec = self.orc.negotiate(prop, acc)
                self.orc.set_state(theta=np.where(done, self.orc.get_state()["theta"], old))
                for f, dec in zip(self.forms, self.decs):
                    gu.assert_same("decisions", dec.cpu().numpy()[done], want_dec[done], "%s %s" % (f, ctx))
        self.check_obs(ctx)
        self.check_state(ctx)

    def finish(self, ctx="end"):
        want = self.orc.metrics_raw()
        for f, env in zip(self.forms, self.envs):
            gu.assert_same("metrics", env.metrics_raw().cpu().numpy(), want, "%s %s" % (f, ctx))


HORIZON = 40


@pytest.mark.parametrize("v,form", [(v, f) for v in VARIANTS for f in v.forms], ids=lambda x: x if isinstance(x, str) else x.name)
def test_variant_matches_oracle(oracle_lib, monkeypatch, v, form):
    """reset, 60 steps (feature_obs every other step, masked resets of finished envs), then HORIZON + 5 auto-reset steps
    with negotiation and staggered episodes; the first reset and steps are profiled"""
    monkeypatch.setenv("SSD_LOGIC8", str(v.logic8))
    r = Rollout(oracle_lib, v.kind, v.n, _map(v), v.E, v.first, (form,), HORIZON, seed=1000 + VARIANTS.index(v))
    a0, a1 = r.actions(), r.actions()

    def first_calls():
        r.reset()
        r.step(a0, False, "step 0")
        r.step(a1, True, "step 1")
    launched = _launched(first_calls)
    assert launched == variant_kernels(v, form), "launched %s, the table lists %s" % (sorted(launched), sorted(variant_kernels(v, form)))
    for t in range(2, 60):
        done = r.step(r.actions(), t % 2 == 1, "step %d" % t)
        if done.any():
            mask = done.copy()
            mask[::3] = 0                           # the others keep running past the horizon
            if mask.any():
                r.reset(mask, "masked reset after step %d" % t)
    r.set_t(np.arange(v.E) % HORIZON)
    for t in range(HORIZON + 5):
        r.auto_step(r.actions(), t % 3 == 0, "auto-reset step %d" % t)
    assert r.finished >= v.E
    r.finish()


# ---- the observe kernel's schedule: static grid-stride envs, then a dynamic tail from a global counter that the last CTA
# re-arms; sizes chosen relative to the persistent grid (W = grid x 8 warps)
_GRID = {}
_RESET_LINE = re.compile(r"reset kernel: \d+ CTAs x \d+ warps = (\d+) warps; octet logic kernel: \d+ CTAs x \d+ envs = (\d+) envs/round")


def persistent_grids(capfd, monkeypatch, v):
    """(W, Wr, G8) of the configuration of VARIANTS row v: the observe kernel's warps, the reset kernels' warps and the
    octet logic kernel's envs per round, from the line SSD_DEBUG prints at create (a probe batch larger than every grid;
    the grids depend on kind, agents and map, not on the observation form)"""
    key = (v.kind, v.n, v.map)
    if key not in _GRID:
        from contracts_b200.batched import BatchedGridEnv
        monkeypatch.setenv("SSD_DEBUG", "1")
        E = 1 << 16
        capfd.readouterr()
        probe = BatchedGridEnv(v.kind + "_new", E, v.n, _map(v), contract=CONTRACT[v.kind] if v.n >= 2 else None)
        err = capfd.readouterr().err
        probe.close()
        monkeypatch.delenv("SSD_DEBUG")
        m = re.search(r"observe kernel: (\d+) warps/CTA, .* grid (\d+);", err)
        assert m, "SSD_DEBUG printed no observe-kernel grid: %r" % err
        r = _RESET_LINE.search(err)
        assert r, "SSD_DEBUG printed no reset / octet grid: %r" % err
        grids = (int(m.group(1)) * int(m.group(2)), int(r.group(1)), int(r.group(2)))
        assert max(grids) < E, "the probe batch does not fill the persistent grids %r" % (grids,)
        with capfd.disabled():
            print("[persistent grids] %s n=%d %s map: W = %d observe warps, Wr = %d reset warps, G8 = %d octet envs/round" %
                  ((v.kind, v.n, v.map) + grids))
        _GRID[key] = grids
    return _GRID[key]


def _persistent_warps(capfd, monkeypatch, v=VARIANTS[0]):
    """warps of the observe kernel's persistent grid (stock cleanup n = 8 unless another VARIANTS row is given)"""
    return persistent_grids(capfd, monkeypatch, v)[0]


SIZES = {"1": lambda W: 1, "W-1": lambda W: W - 1, "W": lambda W: W, "W+1": lambda W: W + 1, "2W+1": lambda W: 2 * W + 1,
         "5W+17": lambda W: 5 * W + 17}


@pytest.fixture(params=["0", "unset", "100"])
def obs_static_pct(request, monkeypatch):
    """SSD_OBS_STATIC_PCT (read when the handle is created): 0 = every env from the counter, 100 = every env static"""
    if request.param == "unset":
        monkeypatch.delenv("SSD_OBS_STATIC_PCT", raising=False)
    else:
        monkeypatch.setenv("SSD_OBS_STATIC_PCT", request.param)
    return request.param


# the observe kernel's layouts: stock cleanup n = 8 (LAY = 1; its sizes carry no prefix), stock harvest n = 4 (LAY = 2) and
# the generic kernel with 8 mask words (LAY = 0, MW = 8)
SCHEDULE_ROWS = ("cleanup_n8_stock", "harvest_n4_stock", "cleanup_n8_big44x60")


@pytest.mark.parametrize("size", [(row + "/" if row != SCHEDULE_ROWS[0] else "") + s for row in SCHEDULE_ROWS for s in SIZES])
def test_observe_schedule_matches_oracle(oracle_lib, capfd, monkeypatch, obs_static_pct, size):
    """each layout of the observe kernel, uint8 and bf16: 20 back-to-back auto-reset steps, every env compared with the
    oracle; E relative to that configuration's own persistent grid"""
    row, _, size = size.rpartition("/")
    v = next(x for x in VARIANTS if x.name == (row or SCHEDULE_ROWS[0]))
    E = SIZES[size](_persistent_warps(capfd, monkeypatch, v))
    r = Rollout(oracle_lib, v.kind, v.n, _map(v), E, 7, ("u8", "bf16"), 25, seed=77)
    r.reset()
    r.set_t((24 - np.arange(E)) % 25)                # env e finishes in step e mod 25
    for t in range(20):
        r.auto_step(r.actions(), False, "E %d auto-reset step %d" % (E, t))
    assert r.finished > 0
    r.finish()

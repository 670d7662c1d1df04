"""GPU: the grid-world step and reset kernels against the C oracle across the rounds of their persistent grids.

Every grid-world kernel makes one warp, octet or CTA serve env after env, and each env inherits the shared-memory state
(tiles T / T2, stage and spawn scratch, view descriptors, the per-warp map of the global reset) of the one before:
  - grid_obs_kernel: a persistent grid of W warps; each warp takes obs_static_iters envs grid-stride, then more from a
    counter that the last CTA re-arms;
  - grid_feature_kernel / grid_global_kernel: the same grid, grid-stride;
  - grid_logic8_kernel: groups of 32 envs, `grp += gridDim.x` (G8 envs per round);
  - grid_reset_kernel, grid_reset_features_kernel, grid_reset_global_kernel: Wr warps, each taking its envs 32 at a time
    through a ballot (`i0 += 32` once E > 32 Wr).
W, Wr and G8 are read for each configuration from the line SSD_DEBUG prints at create, and the batches below are sized
against them, so that every warp (octet group, reset chunk) serves more than one env.  Every env is compared by bit
pattern with the oracle after every call.

Which kernels a configuration launches depends on kind, map, agents, form and want_features, not on E (the logic kernel
is forced with SSD_LOGIC8), so the rows name their kernels from the tables that test_cuda_kernel_variants,
test_grid_feature_obs and test_grid_global_obs pin to what is launched; test_every_instantiation_has_a_multi_round_row
checks on the CPU that these rows name every instantiation.  No torch.profiler here: test_grid_feature_obs.py records that
profiler records were lost late in a B200 session."""
import collections
import re
import time

import numpy as np
import pytest
import torch

from test_cuda_kernel_variants import CONTRACT, KIND_ID, VARIANTS, Rollout, _map, persistent_grids, variant_kernels
from test_grid_feature_obs import FEATURE_KERNELS, flat_rows, reset_rows
from test_grid_global_obs import GLOBAL_KERNELS, conv

FIRST = 7 * 16384                       # first_env_id of rank 7 of a sharded 16384-env-per-GPU run
DTYPES = {"u8": None, "f64": None, "f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}
FEATURE_OUT = {"f32": 0, "f16": 1, "bf16": 2, "f64": 3}     # OUT of the feature form's kernels (SSD_POLICY_* / SSD_FEATURE_F64)
GLOBAL_OUT = {"f32": 0, "f16": 1, "bf16": 2, "u8": 4}       # OUT of the global form's kernels (SSD_POLICY_* / SSD_GLOBAL_U8)


def _variant(name):
    return next(v for v in VARIANTS if v.name == name)


def _mask_words(v):
    """MW of a VARIANTS row: the mask words of the observe kernel the row's table entry names"""
    return int(re.match(r"grid_obs_kernel<\d+, (\d+),", v.kernels[1]).group(1))


def _report(capfd, text):
    """print past the capture that reads SSD_DEBUG's lines"""
    if capfd is None:
        print(text)
        return
    with capfd.disabled():
        print(text)


def _wall(capfd, t0, what):
    _report(capfd, "[%s] %.1f s" % (what, time.perf_counter() - t0))


# ---- bit-exact comparison on the device ---------------------------------------------------------------------------------
def _same_bits(name, got, want, ctx, rows_per_env=1):
    """got and want (device tensors, env-major) by bit pattern; names the first differing envs"""
    assert tuple(got.shape) == tuple(want.shape) and got.dtype == want.dtype, \
        "%s: %s %r != %s %r at %s" % (name, got.dtype, tuple(got.shape), want.dtype, tuple(want.shape), ctx)
    if got.numel() == 0:
        return
    rows = got.shape[0] // rows_per_env
    g = got.contiguous().view(torch.uint8).reshape(rows, -1)
    w = want.contiguous().view(torch.uint8).reshape(rows, -1)
    bad = (g != w).any(1).nonzero().flatten()
    assert bad.numel() == 0, "%s differs from the oracle at %s in %d envs, first %r" % (name, ctx, bad.numel(), bad[:10].tolist())


class AltRollout(Rollout):
    """Rollout's calls and checks for the feature form (family "feature": float64 rows or the policy's flat T rows, under
    the configuration's contract) and the global form ("global": uint8 view or T [E, 3, H, W], no contract).  Step rows
    are compared with the oracle's feature_obs / global_view(), reset rows with reset_rows of the oracle's state — for at
    most `sample` of the envs a call resets when given (reset_rows is a Python loop), always including the last ones.
    The outputs, state, decisions and metrics are Rollout's checks."""

    def __init__(self, oracle_lib, family, kind, n, amap, E, first, forms, horizon, seed, sample=None):
        from contracts_b200.batched import BatchedGridEnv
        self.family, self.amap, self.sample = family, amap, sample
        self.kind, self.n, self.E, self.horizon = kind, n, E, horizon
        self.contract = CONTRACT[kind] if family == "feature" and n >= 2 else None
        self.nact = 9 if kind == "cleanup" else 8
        self.orc = oracle_lib.GridOracle(kind, E, n, amap, horizon=horizon, contract=self.contract, seed=seed, first_env_id=first)
        self.envs = [BatchedGridEnv(kind + "_new", E, n, amap, horizon=horizon, contract=self.contract, seed=seed,
                                    first_env_id=first, policy_dtype=DTYPES[f], image_obs=family != "feature",
                                    global_obs=family == "global") for f in forms]
        self.forms = forms
        self.decs = [torch.zeros(E, dtype=torch.uint8, device="cuda") for _ in forms]
        self.rng = np.random.RandomState(seed)
        self.rows = np.zeros((E, n, self.orc.F))      # feature form: the oracle's float64 rows ...
        self.known = np.zeros(E, bool)                # ... of these envs
        self.finished = 0

    def _reset_rows(self, sel):
        idx = np.nonzero(sel)[0]
        keep = idx
        if self.sample is not None and idx.size > self.sample:
            keep = np.union1d(idx[::-(-idx.size // self.sample)], idx[-16:])
        self.known[idx] = False
        if keep.size:
            st = self.orc.get_state()
            self.rows[keep] = reset_rows(self.kind, self.amap, {k: st[k][keep] for k in ("map", "pos", "ori")})
            self.known[keep] = True

    def check_obs(self, ctx):
        if self.family == "global":
            view = torch.from_numpy(self.orc.global_view()).cuda()
            for f, env in zip(self.forms, self.envs):
                got, want = (env.obs, view) if f == "u8" else (env.policy_obs, conv(view, DTYPES[f]))
                _same_bits("global rows", got, want, "%s %s" % (f, ctx))
            return
        known = torch.from_numpy(self.known).cuda()
        rows = torch.from_numpy(self.rows).cuda()
        theta = torch.from_numpy(self.orc.get_state()["theta"]).cuda()
        for f, env in zip(self.forms, self.envs):
            if f == "f64":
                got, want = env.obs, rows
            else:
                got = env.policy_obs.view(self.E, self.n, -1)
                want = flat_rows(rows, theta, self.contract is not None, DTYPES[f]).view(self.E, self.n, -1)
            _same_bits("feature rows", got[known], want[known], "%s %s" % (f, ctx))

    def reset(self, mask=None, ctx="reset"):
        m = None if mask is None else torch.as_tensor(np.asarray(mask).astype(np.uint8)).cuda()
        for env in self.envs:
            env.reset(m)
        self.orc.reset(None if mask is None else np.asarray(mask).astype(np.uint8))
        if self.family == "feature":
            self._reset_rows(np.ones(self.E, bool) if mask is None else np.asarray(mask).astype(bool))
        self.check_obs(ctx)
        self.check_state(ctx)

    def _after_step(self, o):
        if self.family == "feature":
            self.rows, self.known[:] = o["feature_obs"], True

    def step(self, a, wf, ctx):
        """wf is Rollout's feature_obs flag: the feature and global forms write no feature_obs copy"""
        a_dev = torch.as_tensor(a.astype(np.uint8)).cuda()
        for env in self.envs:
            env.step(a_dev)
        o = self.orc.step(a, want_features=self.family == "feature")
        self._after_step(o)
        self.check_outputs(o, False, ctx)
        self.check_obs(ctx)
        self.check_state(ctx)
        return o["done"]

    def auto_step(self, a, wf, ctx):
        prop, acc = self.rng.uniform(0.0, 0.2, self.E), self.rng.uniform(0.3, 1.0, (self.E, self.n))
        a_dev = torch.as_tensor(a.astype(np.uint8)).cuda()
        prop_d, acc_d = torch.as_tensor(prop).cuda(), torch.as_tensor(acc).cuda()
        for env, dec in zip(self.envs, self.decs):
            env.step(a_dev, auto_reset=True, negotiation=(prop_d, acc_d, dec) if self.contract else None)
        o = self.orc.step(a, want_features=self.family == "feature")
        self._after_step(o)
        self.check_outputs(o, False, ctx)
        done = o["done"].astype(bool)
        if done.any():
            self.finished += int(done.sum())
            self.orc.reset(o["done"])
            if self.contract:
                old = self.orc.get_state()["theta"]
                want_dec = self.orc.negotiate(prop, acc)
                self.orc.set_state(theta=np.where(done, self.orc.get_state()["theta"], old))
                for f, dec in zip(self.forms, self.decs):
                    _same_bits("decisions", dec[torch.from_numpy(done).cuda()], torch.from_numpy(want_dec[done]).cuda(),
                               "%s %s" % (f, ctx))
            if self.family == "feature":
                self._reset_rows(done)
        self.check_obs(ctx)
        self.check_state(ctx)

    def close(self):
        for env in self.envs:
            env.close()


def _one_env_per_warp(E, warps):
    """a mask with one env of each of `warps` grid-stride warps (env w + k warps, k varying over the warp's envs)"""
    m = np.zeros(E, bool)
    for w in range(min(warps, E)):
        count = len(range(w, E, warps))
        m[w + warps * ((7 * w + 3) % count)] = True
    return m


def _multi_round_schedule(r, W, Wr, name):
    """reset, six steps (feature_obs on odd steps where the form has it) with masked resets of the last observe round only
    and of one env per reset warp, then staggered auto-reset steps with negotiation until every env has restarted"""
    E = r.E
    masks = {2: ("last observe round", np.arange(E) >= (-(-E // W) - 1) * W), 4: ("one env per reset warp", _one_env_per_warp(E, Wr))}
    r.reset(None, "%s reset" % name)
    for t in range(6):
        r.step(r.actions(), t % 2 == 1, "%s step %d" % (name, t))
        if t in masks:
            what, m = masks[t]
            r.reset(m, "%s masked reset (%s) after step %d" % (name, what, t))
    r.set_t(np.arange(E) % r.horizon)
    for t in range(r.horizon + 2):
        r.auto_step(r.actions(), t % 3 == 0, "%s auto-reset step %d" % (name, t))
    assert r.finished >= E, "%s: %d restarts for %d envs" % (name, r.finished, E)
    r.finish("%s end" % name)


# ---- a. every window-form instantiation past one round ------------------------------------------------------------------
H_ROUNDS = 10


@pytest.mark.gpu
@pytest.mark.parametrize("v", VARIANTS, ids=[v.name for v in VARIANTS])
def test_window_forms_past_one_round(oracle_lib, capfd, monkeypatch, v):
    """every VARIANTS row in each of its forms at E = 2W + 17 with its logic kernel: every observe warp takes envs from the
    static and the dynamic part of the schedule, and some reset warps serve two envs"""
    t0 = time.perf_counter()
    W, Wr, G8 = persistent_grids(capfd, monkeypatch, v)
    E = 2 * W + 17
    assert E >= 2 * W and E > Wr
    monkeypatch.setenv("SSD_LOGIC8", str(v.logic8))
    r = Rollout(oracle_lib, v.kind, v.n, _map(v), E, FIRST, v.forms, H_ROUNDS, seed=2000 + VARIANTS.index(v))
    _multi_round_schedule(r, W, Wr, v.name)
    _report(capfd, "[%s %s] E = %d: W = %d (up to %d envs per observe warp), Wr = %d (up to %d envs per reset warp), G8 = %d" %
            (v.name, "/".join(v.forms), E, W, -(-E // W), Wr, -(-E // Wr), G8))
    _wall(capfd, t0, v.name)


# ---- b. the feature and global forms past one round ---------------------------------------------------------------------
AltRow = collections.namedtuple("AltRow", "variant family")

# the configurations the feature / global form runs past one round: both kinds with 4 and 8 mask words
ALT_ROWS = [
    AltRow("cleanup_n8_stock", "feature"), AltRow("cleanup_n8_stock", "global"),            # cleanup, MW 4
    AltRow("cleanup_n8_big44x60", "feature"), AltRow("cleanup_n8_big44x60", "global"),      # cleanup, MW 8
    AltRow("harvest_n4_stock", "feature"), AltRow("harvest_n4_stock", "global"),            # harvest, MW 8
    AltRow("harvest_n8_cramped", "feature"), AltRow("harvest_n8_cramped", "global"),        # harvest, MW 4
]
ALT_FORMS = {"feature": ("f64", "f32", "f16", "bf16"), "global": ("u8", "f32", "f16", "bf16")}


def alt_kernels(row):
    """the feature / global step and reset instantiations a row runs in its family's forms"""
    v = _variant(row.variant)
    k, mw = KIND_ID[v.kind], _mask_words(v)
    if row.family == "feature":
        return {"grid_feature_kernel<%d, %d, %d>" % (k, mw, FEATURE_OUT[f]) for f in ALT_FORMS["feature"]} | \
               {"grid_reset_features_kernel<%d, %d>" % (k, FEATURE_OUT[f]) for f in ALT_FORMS["feature"]}
    return {"grid_global_kernel<%d, %d, %d>" % (k, mw, GLOBAL_OUT[f]) for f in ALT_FORMS["global"]} | \
           {"grid_reset_global_kernel<%d, %d>" % (k, GLOBAL_OUT[f]) for f in ALT_FORMS["global"]}


@pytest.mark.gpu
@pytest.mark.parametrize("row", ALT_ROWS, ids=["%s-%s" % r for r in ALT_ROWS])
def test_alt_forms_past_one_round(oracle_lib, capfd, monkeypatch, logic_variant, row):
    """the feature form (float64 and T rows, contract) or the global form (uint8 and T views) at E = 2W + 17, both logic
    kernels: the schedule of test_window_forms_past_one_round"""
    t0 = time.perf_counter()
    v = _variant(row.variant)
    W, Wr, G8 = persistent_grids(capfd, monkeypatch, v)
    E = 2 * W + 17
    assert E >= 2 * W and E > Wr
    r = AltRollout(oracle_lib, row.family, v.kind, v.n, _map(v), E, FIRST, ALT_FORMS[row.family], H_ROUNDS,
                   seed=3000 + ALT_ROWS.index(row))
    name = "%s %s %s" % (row.variant, row.family, logic_variant)
    _multi_round_schedule(r, W, Wr, name)
    _report(capfd, "[%s] E = %d: W = %d (up to %d envs per warp), Wr = %d (up to %d envs per reset warp), MW = %d" %
            (name, E, W, -(-E // W), Wr, -(-E // Wr), _mask_words(v)))
    r.close()
    _wall(capfd, t0, name)


# ---- d. the octet logic kernel past one round ---------------------------------------------------------------------------
OCTET_ROWS = {"cleanup": "cleanup_n8_stock", "harvest": "harvest_n4_stock"}
OCTET_SIZES = {"G8-1": lambda G: G - 1, "G8": lambda G: G, "G8+1": lambda G: G + 1, "2G8+1": lambda G: 2 * G + 1}
H_OCTET = 8


@pytest.mark.gpu
@pytest.mark.parametrize("kind,size", [(k, s) for k in OCTET_ROWS for s in OCTET_SIZES] + [("harvest", "24576-default")])
def test_octet_logic_past_one_round(oracle_lib, capfd, monkeypatch, kind, size):
    """grid_logic8_kernel (SSD_LOGIC8=1) at E around multiples of G8, and harvest n = 4 at 24576 envs under the default
    selection (the largest batch ssd_create gives the octet kernel): staggered auto-reset with negotiation in the float64
    feature form, whose rows cost least to compare (reset rows of a sample of the restarted envs); rewards, transfers,
    infos, dones, decisions, state and metrics of every env"""
    t0 = time.perf_counter()
    v = _variant(OCTET_ROWS[kind])
    W, Wr, G8 = persistent_grids(capfd, monkeypatch, v)
    if size == "24576-default":
        monkeypatch.delenv("SSD_LOGIC8", raising=False)
        E = 24576
    else:
        monkeypatch.setenv("SSD_LOGIC8", "1")
        E = OCTET_SIZES[size](G8)
    rounds = -(-E // G8)
    _report(capfd, "[octet %s %s] E = %d, G8 = %d: %d round(s) of the octet kernel%s" %
            (kind, size, E, G8, rounds, " (the default selection's largest batch spans more than one round)" if rounds > 1 and
             size == "24576-default" else ""))
    r = AltRollout(oracle_lib, "feature", v.kind, v.n, _map(v), E, FIRST, ("f64",), H_OCTET, seed=4000 + E, sample=256)
    r.reset(None, "E %d reset" % E)
    r.set_t(np.arange(E) % H_OCTET)
    for t in range(H_OCTET + 2):
        r.auto_step(r.actions(), False, "E %d auto-reset step %d" % (E, t))
    assert r.finished >= E
    r.finish("E %d end" % E)
    r.close()
    _wall(capfd, t0, "octet %s %s" % (kind, size))


# ---- e. reset kernels past one chunk ------------------------------------------------------------------------------------
RESET_FAMILIES = {"windows": ("u8", "bf16"), "feature": ("f64",), "global": ("u8",)}


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(RESET_FAMILIES))
def test_reset_kernels_past_one_chunk(oracle_lib, capfd, monkeypatch, family):
    """stock harvest n = 4 at E = 32 Wr + 17 (reset warps 0..16 take a second chunk of 32 envs): a full reset, then masked
    resets of every env, of the second chunk's envs only, of one env per reset warp and of none, each followed by a step"""
    t0 = time.perf_counter()
    v = _variant("harvest_n4_stock")
    W, Wr, G8 = persistent_grids(capfd, monkeypatch, v)
    E = 32 * Wr + 17
    assert E > 32 * Wr
    forms = RESET_FAMILIES[family]
    if family == "windows":
        r = Rollout(oracle_lib, v.kind, v.n, _map(v), E, FIRST, forms, 1000, seed=5000)
    else:
        r = AltRollout(oracle_lib, family, v.kind, v.n, _map(v), E, FIRST, forms, 1000, seed=5000, sample=2048)
    chunk = np.arange(E) // Wr                       # the chunk of its warp an env is in, times 32
    masks = [("every env", np.ones(E, bool)), ("the second chunk", chunk >= 32),
             ("one env per reset warp", _one_env_per_warp(E, Wr)), ("no env", np.zeros(E, bool))]
    _report(capfd, "[reset %s] E = %d, Wr = %d: %d envs in the second chunk" % (family, E, Wr, int(masks[1][1].sum())))
    r.reset(None, "full reset")
    r.step(r.actions(), False, "step 0")
    for what, m in masks:
        r.reset(m, "masked reset (%s)" % what)
        r.step(r.actions(), False, "step after the masked reset (%s)" % what)
    r.finish()
    if family != "windows":
        r.close()
    _wall(capfd, t0, "reset %s" % family)


# ---- f. harvest at the benchmark's size ---------------------------------------------------------------------------------
BENCH_E = 16384                                      # bench.py's harvest16k: envs per GPU, n = 4
BENCH_FAMILIES = {"windows": ("u8", "f32", "f16", "bf16"), "feature": ("f64", "bf16"), "global": ("u8", "bf16")}
H_BENCH = 12


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(BENCH_FAMILIES))
def test_harvest_benchmark_size(oracle_lib, monkeypatch, family):
    """stock harvest n = 4 at 16384 envs with the default logic selection, in every form: staggered auto-reset (with
    negotiation where there is a contract) until every env has restarted, every env compared at every step (the windows
    with feature_obs on every third step)"""
    t0 = time.perf_counter()
    monkeypatch.delenv("SSD_LOGIC8", raising=False)
    v = _variant("harvest_n4_stock")
    forms = BENCH_FAMILIES[family]
    if family == "windows":
        r = Rollout(oracle_lib, v.kind, v.n, _map(v), BENCH_E, FIRST, forms, H_BENCH, seed=73907)
    else:
        r = AltRollout(oracle_lib, family, v.kind, v.n, _map(v), BENCH_E, FIRST, forms, H_BENCH, seed=73907)
    r.reset(None, "harvest16k reset")
    r.set_t(np.arange(BENCH_E) % H_BENCH)
    for t in range(H_BENCH + 2):
        r.auto_step(r.actions(), t % 3 == 0, "harvest16k auto-reset step %d" % t)
    assert r.finished >= BENCH_E
    r.finish("harvest16k end")
    if family != "windows":
        r.close()
    _wall(None, t0, "harvest16k %s" % family)


# ---- g. no instantiation without a multi-round row ----------------------------------------------------------------------
def test_every_instantiation_has_a_multi_round_row():
    """CPU: the kernels this file's rows run (every VARIANTS row in each form, ALT_ROWS in their family's forms) are every
    instantiation of the VARIANTS, FEATURE_KERNELS and GLOBAL_KERNELS tables, which the cuobjdump inventories pin to the
    library"""
    named = set().union(*(variant_kernels(v, f) for v in VARIANTS for f in v.forms), *(alt_kernels(r) for r in ALT_ROWS))
    tables = set().union(*(variant_kernels(v, f) for v in VARIANTS for f in v.forms)) | set(FEATURE_KERNELS) | set(GLOBAL_KERNELS)
    assert sorted(tables - named) == [], "instantiations without a multi-round row"
    assert sorted(named - tables) == [], "rows name kernels the tables do not list"

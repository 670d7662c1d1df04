"""Replay a golden fixture (reference output, tests/golden/*.npz) against a backend.

A backend adapter exposes, for ONE environment:
    reset() -> obs uint8 [n,15,15,3]
    step(actions int[n], want_features) -> dict(obs, rew, base_rew, transfers, info [n,4], done, feature_obs|None)
    state() -> dict(map [H,W] uint8 chars, pos [n,2], ori [n], theta float64)
    metrics_raw() -> float64 [56]
Every comparison is bit-exact (float64 compared through their uint64 bit patterns).
"""
import glob
import hashlib
import os

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


OTHER_SCHEMAS = ("negotiate_", "selfdrive_", "features_", "flatobs_", "solver_", "joint_", "render_")


def fixture_names(prefix=None):
    """Step-replay fixtures (default) or the fixtures of another schema (`prefix`)."""
    names = sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))
    if prefix is None:
        return [n for n in names if not n.startswith(OTHER_SCHEMAS)]
    return [n for n in names if n.startswith(prefix)]


def load(name):
    d = np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)
    return {k: d[k] for k in d.files}


def shaping_kwargs(fx):
    """use_collective_reward / inequity_averse_reward / alpha / beta of a fixture (absent in older fixtures)."""
    mode = int(fx["reward_mode"]) if "reward_mode" in fx else 0
    if not mode:
        return {}
    return dict(use_collective_reward=bool(mode & 1), inequity_averse_reward=bool(mode & 2),
                alpha=float(fx["alpha"]), beta=float(fx["beta"]))


def contract_name(fx):
    if not bool(fx["contract"]):
        return None
    return "CleanupContract" if str(fx["kind"]) == "cleanup" else "HarvestFeaturemodLocalContract"


class _Stored:
    """The reference's side of a comparison when the reference does not run: its outputs are only known through the
    digests stored in tests/golden/reference_tapes.json (see Tape).  Indexing and membership keep the test bodies as they
    are; every comparison against it is checked through the active tape."""

    def __getitem__(self, key):
        return self

    def __contains__(self, key):
        return True


STORED = _Stored()
TAPE = None                 # the active Tape, set by a fixture of the differential tests


class Tape:
    """Ordered digest of every value a reference comparison checks (name, shape and the bits assert_same compares).
    A checkpoint is taken every EVERY values and at the end; against `stored` checkpoints each one must match, so a
    divergence is located to within EVERY comparisons."""
    EVERY = 1000

    def __init__(self, test_id, stored=None):
        self.test_id, self.stored = test_id, stored
        self.h, self.count, self.marks, self.last_ctx = hashlib.sha256(), 0, [], None
        self.diverged = False

    def feed(self, name, got, ctx):
        got = np.asarray(got)
        canon = bits(got) if got.dtype.kind == "f" else np.ascontiguousarray(got.astype(np.int64))
        self.h.update(("%s|%r|" % (name, got.shape)).encode())
        self.h.update(canon.tobytes())
        self.count += 1
        self.last_ctx = ctx
        if self.count % self.EVERY == 0:
            self._mark()

    def _mark(self):
        d = self.h.hexdigest()[:16]
        i = len(self.marks)
        self.marks.append(d)
        if self.stored is not None:
            self.diverged = True                    # until this checkpoint is found equal
            assert i < len(self.stored), "%s: more comparisons than the reference's recorded run" % self.test_id
            assert self.stored[i] == d, ("%s: the values of comparisons %d..%d (the last at %s) differ from the reference's "
                                         "recorded outputs" % (self.test_id, i * self.EVERY + 1, self.count, self.last_ctx))
            self.diverged = False

    def finish(self):
        if self.diverged:                           # already reported by the failing comparison
            return
        if self.count % self.EVERY:
            self._mark()
        if self.stored is not None:
            assert len(self.marks) == len(self.stored), "%s: fewer comparisons than the reference's recorded run" % self.test_id


def _f64(x):
    return x if x is STORED else np.float64(x)


def bits(x):
    return np.ascontiguousarray(np.asarray(x, dtype=np.float64)).view(np.uint64)


def assert_same(name, got, want, ctx):
    if TAPE is not None:
        TAPE.feed(name, got, ctx)
    if want is STORED:
        return
    got, want = np.asarray(got), np.asarray(want)
    if got.dtype.kind == "f" or want.dtype.kind == "f":
        ok = np.array_equal(bits(got), bits(want)) and got.shape == want.shape
    else:
        ok = np.array_equal(got.astype(np.int64), want.astype(np.int64))
    if not ok:
        raise AssertionError("%s mismatch at %s\n got: %r\nwant: %r" % (name, ctx, got, want))


def equality(totals):
    """compute_equality (cleanup_new.py:422-434) from the per-agent reward sums, same operation order."""
    eq, total = 0, 0
    for i in totals:
        for j in totals:
            eq += abs(i - j)
        total += i
    if total == 0:
        total = 0.001
    return 1 - eq / (2 * len(totals) * total)


def sustainability(totals, tsums):
    """compute_sustainability (cleanup_new.py:436-445) from the per-agent sum r and sum t*r."""
    return np.mean([ts / max(tot, 1) for tot, ts in zip(totals, tsums)])


def metrics_from_raw(kind, n, contract, raw):
    """env.metrics (minus equality/sustainability, checked separately) from the raw accumulators."""
    m = {"total_apples_eaten": raw[0], "raw_env_rewards": raw[2], "transfers": raw[3]}
    if kind == "cleanup":
        m["dirt_cleaned"] = raw[4]
        for i in range(n):
            m["a%d-waste_cleaned" % i] = raw[8 + i]
    else:
        m["low_density_apples_eaten"] = raw[1]
        for i in range(n):
            m["a%d-apples_consumed" % i] = raw[8 + i]
            m["a%d-close_apples_consumed" % i] = raw[16 + i]
    return m


def check_episode_metrics(kind, n, contract, raw, want, ctx):
    """env.metrics of the reference at the end of an episode (`want`: name -> value) against a backend's raw
    accumulators, bit for bit, incl. equality / sustainability when the episode ended."""
    raw = np.asarray(raw, dtype=np.float64)
    assert raw[5] == 0, "backend error flags %r" % raw[5]
    got = metrics_from_raw(kind, n, contract, raw)
    for k, v in got.items():
        assert_same("metric " + k, np.float64(v), _f64(want[k]), ctx)
    if "equality" in want:          # episode ended: cleanup_new.py:264-266, two_stage_train.py:97-99
        totals, tsums = list(raw[24:24 + n]), list(raw[32:32 + n])
        assert_same("equality", np.float64(equality(totals)), _f64(want["equality"]), ctx)
        assert_same("sustainability", np.float64(sustainability(totals, tsums)), _f64(want["sustainability"]), ctx)
        if "transfer_equality" in want:
            totals, tsums = list(raw[40:40 + n]), list(raw[48:48 + n])
            assert_same("transfer_equality", np.float64(equality(totals)), _f64(want["transfer_equality"]), ctx)
            assert_same("transfer_sustainability", np.float64(sustainability(totals, tsums)),
                        _f64(want["transfer_sustainability"]), ctx)


def replay(backend, fx, check_features=True):
    kind, n = str(fx["kind"]), int(fx["n"])
    episodes, steps = fx["actions"].shape[:2]
    keys = [str(k) for k in fx["metric_keys"]]
    for ep in range(episodes):
        obs = backend.reset()
        st = backend.state()
        ctx = "reset ep %d" % ep
        assert_same("reset map", st["map"], fx["reset_map"][ep], ctx)
        assert_same("reset pos", st["pos"], fx["reset_pos"][ep], ctx)
        assert_same("reset ori", st["ori"], fx["reset_ori"][ep], ctx)
        assert_same("reset obs", obs, fx["reset_obs"][ep], ctx)
        if bool(fx["contract"]):
            assert_same("reset theta", st["theta"], fx["reset_theta"][ep], ctx)
        for t in range(steps):
            ctx = "ep %d step %d" % (ep, t)
            o = backend.step(fx["actions"][ep, t], check_features)
            st = backend.state()
            assert_same("pos", st["pos"], fx["pos"][ep, t], ctx)
            assert_same("ori", st["ori"], fx["ori"][ep, t], ctx)
            assert_same("map", st["map"], fx["map"][ep, t], ctx)
            assert_same("obs", o["obs"], fx["obs"][ep, t], ctx)
            assert_same("base_rew", o["base_rew"], fx["base_rew"][ep, t], ctx)
            assert_same("transfers", o["transfers"], fx["transfers"][ep, t], ctx)
            assert_same("rew", o["rew"], fx["rew"][ep, t], ctx)
            assert_same("eaten_apples", o["info"][:, 0], fx["eaten_apples"][ep, t], ctx)
            assert_same("cleaned|eaten_close", o["info"][:, 1], fx["info1"][ep, t], ctx)
            assert_same("done", int(o["done"]), int(fx["done"][ep, t]), ctx)
            if check_features and o.get("feature_obs") is not None:
                assert_same("feature_obs", o["feature_obs"], fx["feature_obs"][ep, t], ctx)
        want = dict(zip(keys, fx["metrics"][ep]))
        check_episode_metrics(kind, n, bool(fx["contract"]), backend.metrics_raw(), want, "ep %d" % ep)


def auto_reset_step(orc, actions, done_prev):
    """One step of a batch with the next-step auto-reset, on a FeatOracle / CarOracle of all its envs: the envs that
    finished in the previous step (done_prev, bool [E]) restart instead of stepping (reset observation, zero rewards,
    transfers and infos, done cleared, their actions ignored); the others step.  Returns the step's outputs."""
    done_prev = np.asarray(done_prev, dtype=bool)
    restart = orc.reset(done_prev) if done_prev.any() else None
    o = orc.step(actions, skip=done_prev)
    if restart is not None:
        o["obs"][done_prev] = restart[done_prev]
    return o


class OracleBackend:
    def __init__(self, oracle_mod, fx):
        self.o = oracle_mod.GridOracle(str(fx["kind"]), 1, int(fx["n"]), [str(r) for r in fx["ascii_map"]],
                                       horizon=int(fx["horizon"]), contract=contract_name(fx),
                                       seed=int(fx["seed"]), first_env_id=int(fx["env_id"]), **shaping_kwargs(fx))

    def reset(self):
        return self.o.reset()[0]

    def step(self, actions, want_features):
        r = self.o.step(np.asarray(actions)[None], want_features)
        return {k: (None if v is None else v[0]) for k, v in r.items()}

    def state(self):
        return {k: v[0] for k, v in self.o.get_state().items()}

    def metrics_raw(self):
        return self.o.metrics_raw()[0]


class CudaBackend:
    """Env `index` of a small BatchedGridEnv whose global id equals the fixture's env_id."""

    def __init__(self, fx, num_envs=3, index=1, padded_obs=False):
        from contracts_b200.batched import BatchedGridEnv
        kind = "cleanup_new" if str(fx["kind"]) == "cleanup" else "harvest_new"
        self.i = index
        first = (int(fx["env_id"]) - index) & 0xFFFFFFFF
        self.env = BatchedGridEnv(kind, num_envs, int(fx["n"]), [str(r) for r in fx["ascii_map"]],
                                  horizon=int(fx["horizon"]), contract=contract_name(fx), seed=int(fx["seed"]),
                                  first_env_id=first, padded_obs=padded_obs, **shaping_kwargs(fx))
        self.n = int(fx["n"])

    def reset(self):
        return self.env.reset()[self.i].cpu().numpy()

    def step(self, actions, want_features):
        import torch
        a = torch.zeros((self.env.E, self.n), dtype=torch.uint8)
        a[:] = torch.as_tensor(np.asarray(actions).astype(np.uint8))
        obs, rew, done, info = self.env.step(a.cuda(), want_features=want_features)
        i = self.i
        return {"obs": obs[i].cpu().numpy(), "rew": rew[i].cpu().numpy(), "base_rew": self.env.base_rew[i].cpu().numpy(),
                "transfers": self.env.transfers[i].cpu().numpy(), "info": info[i].cpu().numpy(),
                "done": int(done[i].item()),
                "feature_obs": self.env.feature_obs[i].cpu().numpy() if want_features else None}

    def state(self):
        return {k: v[self.i].cpu().numpy() for k, v in self.env.get_state().items()}

    def metrics_raw(self):
        return self.env.metrics_raw()[self.i].cpu().numpy()


def random_map(rng, kind, n):
    """A walled H x W map with random interior content: at least n spawn points and one cell of every dynamic kind;
    inner walls, dead ends and agents packed next to each other make contested moves and blocked beams frequent."""
    H, W = int(rng.randint(6, 15)), int(rng.randint(6, 15))
    g = np.full((H, W), "@", dtype="<U1")
    inner = [(r, c) for r in range(1, H - 1) for c in range(1, W - 1)]
    rng.shuffle(inner)
    chars = {"cleanup": (["P", "H", "R", "S", "B", " ", "@"], [.22, .16, .08, .06, .2, .2, .08]),
             "harvest": (["P", "A", " ", "@"], [.25, .35, .3, .1])}[kind]
    must = ["P"] * n + (["H", "R", "S", "B"] if kind == "cleanup" else ["A"])
    for i, (r, c) in enumerate(inner):
        g[r, c] = must[i] if i < len(must) else rng.choice(chars[0], p=chars[1])
    return ["".join(row) for row in g]


def big_map(kind, H, W, seed):
    """A random walled map near the size limits (48 x 64, 200+ apple / waste points: the 8-word mask variants of the kernels)."""
    rng = np.random.RandomState(seed)
    g = np.full((H, W), " ", dtype="<U1")
    g[0, :] = g[-1, :] = g[:, 0] = g[:, -1] = "@"
    inner = [(r, c) for r in range(1, H - 1) for c in range(1, W - 1)]
    rng.shuffle(inner)
    kinds = (("P", 24), ("@", 60), ("B", 200), ("H", 90), ("R", 120), ("S", 30)) if kind == "cleanup" else (("P", 24), ("@", 60), ("A", 240))
    k = 0
    for ch, cnt in kinds:
        for r, c in inner[k:k + cnt]:
            g[r, c] = ch
        k += cnt
    return ["".join(row) for row in g]


def policy_image(want_u8, dtype, chunk=8192):
    """the reference's windows uint8 [E, n, 15, 15, 3] (a device tensor) as the policy image T [E n, 3, 15, 15], in chunks
    of envs so that the float64 intermediate stays small"""
    import torch
    out = []
    for e0 in range(0, want_u8.shape[0], chunk):
        x = want_u8[e0:e0 + chunk]
        out.append((x.double() / 255).float().to(dtype).reshape(-1, 15, 15, 3).permute(0, 3, 1, 2))
    return torch.cat(out)

"""The C oracle's step with a skip mask (feat_oracle_step_skip / car_oracle_step_skip), which emulates a batch's next-step
auto-reset at any batch size (golden_util.auto_reset_step): reset(done_prev) + step(skip=done_prev) on one oracle of E envs
must equal one single-env oracle per env, stepped or reset one by one, bit for bit.  CPU only."""
import numpy as np
import pytest

import golden_util as gu

E = 13
CONTRACT = {"cleanup": "CleanupContract", "harvest": "HarvestFeaturemodLocalContract"}


def _maps(kind):
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    return CLEANUP_MAP if kind == "cleanup" else HARVEST_MAP


def _compare(batch_out, singles_out, keys, ctx):
    for k in keys:
        gu.assert_same(k, batch_out[k], np.stack([o[k][0] for o in singles_out]), ctx)


@pytest.mark.parametrize("kind,n", [("cleanup", 3), ("harvest", 4)])
def test_feature_skip_step_equals_single_envs(oracle_lib, kind, n):
    H, first, c = 9, 40, CONTRACT[kind]
    batch = oracle_lib.FeatOracle(kind, E, n, _maps(kind), horizon=H, contract=c, seed=21, first_env_id=first)
    singles = [oracle_lib.FeatOracle(kind, 1, n, _maps(kind), horizon=H, contract=c, seed=21, first_env_id=first + i)
               for i in range(E)]
    gu.assert_same("reset obs", batch.reset(), np.concatenate([s.reset() for s in singles]), "reset")
    rng = np.random.default_rng(5)
    nact = 9 if kind == "cleanup" else 8
    done_prev = np.zeros(E, bool)
    restarts = 0
    for t in range(4 * H):
        if t == 4:                                   # stagger the episodes; a masked reset clears a pending restart
            m = np.arange(E) % 3 == 0
            gu.assert_same("masked reset obs", batch.reset(m)[m], np.concatenate([singles[i].reset() for i in np.nonzero(m)[0]]),
                           "step %d" % t)
            done_prev[m] = False
        a = rng.integers(0, nact, size=(E, n))
        o = gu.auto_reset_step(batch, a, done_prev)
        outs = []
        for i, s in enumerate(singles):
            if done_prev[i]:
                outs.append({"obs": s.reset(), "rew": np.zeros((1, n)), "base_rew": np.zeros((1, n)),
                             "transfers": np.zeros((1, n)), "info": np.zeros((1, n, 4), np.int32), "done": np.zeros(1, np.uint8)})
            else:
                outs.append(s.step(a[i][None]))
        ctx = "%s step %d" % (kind, t)
        _compare(o, outs, ("obs", "rew", "base_rew", "transfers", "info", "done"), ctx)
        sts = [s.get_state() for s in singles]
        _compare(batch.get_state(), sts, ("pos", "ori", "cells", "theta", "t"), ctx)
        gu.assert_same("episode", batch.episode, np.concatenate([s.episode for s in singles]), ctx)
        restarts += int(done_prev.sum())
        done_prev = o["done"].astype(bool)
    assert restarts >= E
    gu.assert_same("metrics", batch.metrics_raw(), np.concatenate([s.metrics_raw() for s in singles]), "end")


def test_selfdrive_skip_step_equals_single_envs(oracle_lib):
    n, first = 3, 7
    kw = dict(contract=True, seed=33)
    batch = oracle_lib.CarOracle(E, n, first_env_id=first, **kw)
    singles = [oracle_lib.CarOracle(1, n, first_env_id=first + i, **kw) for i in range(E)]
    gu.assert_same("reset obs", batch.reset(), np.concatenate([s.reset() for s in singles]), "reset")
    rng = np.random.default_rng(6)
    done_prev = np.zeros(E, bool)
    restarts = 0
    for t in range(300):
        if t == 30:
            m = np.arange(E) % 4 == 1
            gu.assert_same("masked reset obs", batch.reset(m)[m], np.concatenate([singles[i].reset() for i in np.nonzero(m)[0]]),
                           "step %d" % t)
            done_prev[m] = False
        a = rng.uniform(-0.1, 0.1, (E, n)).astype(np.float32)
        o = gu.auto_reset_step(batch, a, done_prev)
        outs = []
        for i, s in enumerate(singles):
            if done_prev[i]:
                outs.append({"obs": s.reset(), "rew": np.zeros((1, n)), "base_rew": np.zeros((1, n)),
                             "transfers": np.zeros((1, n)), "info": np.zeros((1, n, 4)), "done": np.zeros((1, n + 1), np.uint8)})
            else:
                outs.append(s.step(a[i][None]))
        ctx = "selfdrive step %d" % t
        _compare(o, outs, ("obs", "rew", "base_rew", "transfers", "info", "done"), ctx)
        _compare(batch.get_state(), [s.get_state() for s in singles], ("pos", "vel", "theta", "transfers", "t"), ctx)
        restarts += int(done_prev.sum())
        done_prev = o["done"][:, n].astype(bool)
    assert restarts >= E


def test_skip_leaves_rows_and_state_untouched(oracle_lib):
    """a skipped env is not stepped: its state stays and its output rows keep what the caller passed (zeros)"""
    orc = oracle_lib.FeatOracle("cleanup", E, 2, _maps("cleanup"), horizon=50, contract="CleanupContract", seed=3)
    orc.reset()
    before = orc.get_state()
    skip = np.zeros(E, bool)
    skip[[0, 5, E - 1]] = True
    o = orc.step(np.full((E, 2), 2), skip=skip)
    after = orc.get_state()
    for k in ("pos", "ori", "cells", "theta", "t"):
        gu.assert_same(k, after[k][skip], before[k][skip], "skipped")
    assert (after["t"][~skip] == 1).all()
    for k in ("obs", "rew", "base_rew", "transfers", "info", "done"):
        assert not o[k][skip].any(), k
    with pytest.raises(ValueError):
        orc.step(np.zeros((E, 2)), skip=np.zeros(E - 1, bool))

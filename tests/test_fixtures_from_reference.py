"""Needs a checkout of the original project (SSD_REFERENCE_ROOT): the committed fixtures are what the UNMODIFIED
reference produces today — a sample of every fixture family is regenerated through oracle/make_golden.py and compared
array by array."""
import numpy as np
import pytest

import golden_util as gu
from oracle import ref_stubs

pytestmark = pytest.mark.skipif(ref_stubs.live_reference() is None,
                                reason="SSD_REFERENCE_ROOT does not name a checkout of the original project")

SAMPLES = [("run_scenario", "cleanup_n5_short_horizon"), ("run_scenario", "harvest_cramped_n6_collective_inequity"),
           ("run_negotiate", "negotiate_cleanup_n2"), ("run_solver", "solver_cleanup_n2_majority"),
           ("run_joint", "joint_cleanup_n3_global"), ("run_render", "render_cleanup_open_n6")]


@pytest.mark.parametrize("fn,name", SAMPLES, ids=[n for _, n in SAMPLES])
def test_fixture_is_reproduced_by_the_reference(fn, name):
    from oracle import make_golden
    fresh = getattr(make_golden, fn)(name)
    stored = gu.load(name)
    assert set(stored.keys()) <= set(fresh.keys())              # older fixtures predate some metadata keys
    for k in stored:
        a, b = np.asarray(fresh[k]), stored[k]
        assert a.shape == b.shape, k
        if a.dtype.kind == "f":
            assert np.array_equal(a.astype(np.float64).view(np.uint64), b.astype(np.float64).view(np.uint64)), k
        else:
            assert np.array_equal(a, b), k

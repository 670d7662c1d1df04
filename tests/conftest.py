import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: needs a checkout of the original project (SSD_REFERENCE_ROOT)")


def has_reference():
    from oracle import ref_stubs
    return ref_stubs.live_reference() is not None


@pytest.fixture(scope="session")
def oracle_lib():
    from oracle import oracle
    oracle.build()
    return oracle


@pytest.fixture(params=["logic_thread", "logic_octet"])
def logic_variant(request, monkeypatch):
    """The gridworld decision logic has two kernels — one thread per env (ssd_grid2.cuh, large batches) and eight lanes
    per env (ssd_grid3.cuh, batches that do not fill the GPU); ssd_create picks by batch size.  Tests that use this
    fixture run once with each forced (SSD_LOGIC8 is read when the handle is created)."""
    monkeypatch.setenv("SSD_LOGIC8", "1" if request.param == "logic_octet" else "0")
    return request.param

"""CPU: the solver queue's C ABI (ssd_solver_window, ssd_solver_enable / _rows / _resolve) as the bindings declare it,
and its loud failure without a GPU."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_fields(struct):
    text = open(os.path.join(ROOT, "include", "ssd_b200.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (struct, struct), text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return [re.sub(r"\[.*\]|[\*\s]", "", d.strip().split()[-1]) for d in body.split(";") if d.strip()]


def test_window_struct_matches_header():
    """ctypes mirror has the header's field order; three int32 then five pointers (8-byte aligned, 56 bytes)."""
    from contracts_b200 import _lib
    assert _header_fields("ssd_solver_window") == [f[0] for f in _lib.ssd_solver_window._fields_]
    assert ctypes.sizeof(_lib.ssd_solver_window) == 56
    assert _lib.ssd_solver_window.env_dev.offset == 16 and _lib.ssd_solver_window.rows_dev.offset == 48


def test_entry_points_declared():
    from contracts_b200 import _lib
    text = open(os.path.join(ROOT, "include", "ssd_b200.h")).read()
    for name in ("ssd_solver_enable", "ssd_solver_rows", "ssd_solver_resolve"):
        assert name in _lib.EXPORTS
        assert re.search(r"\bint %s\(" % name, text), name


def test_entry_points_reject_null_handle():
    """No device needed: a NULL handle is SSD_EINVAL for every entry point, with or without a window."""
    from contracts_b200 import _lib
    lib = _lib.load()
    win = _lib.ssd_solver_window(struct_size=ctypes.sizeof(_lib.ssd_solver_window), num_samples=1, capacity=1)
    assert lib.ssd_solver_enable(None, 1) == -1
    assert lib.ssd_solver_rows(None, ctypes.byref(win), None, None) == -1
    assert lib.ssd_solver_rows(None, None, None, None) == -1
    assert lib.ssd_solver_resolve(None, ctypes.byref(win), 1, None, None, None, None, None) == -1


def test_queue_fails_loudly_without_gpu():
    """Without a GPU the batch a queue needs cannot be built: an SsdError, not a CPU fallback."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from contracts_b200 import _lib
    from contracts_b200.features import BatchedFeatureEnv
    with pytest.raises(_lib.SsdError):
        BatchedFeatureEnv("cleanup", 3, 2, contract="CleanupContract")


def test_queue_validates_before_the_device():
    """The Python queue rejects a batch without a contract and a bad capacity before any device call."""
    from contracts_b200.solver import SolverQueue

    class Fake:
        contract, E, n = None, 4, 2
    with pytest.raises(ValueError):
        SolverQueue(Fake())
    Fake.contract = "CleanupContract"
    with pytest.raises(ValueError):
        SolverQueue(Fake(), capacity=5)
    with pytest.raises(ValueError):
        SolverQueue(Fake(), rule="min")

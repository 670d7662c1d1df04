"""CPU: the grid worlds' global output C ABI (ssd_global_out, ssd_set_global_output) as the bindings declare it."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_global_out_struct_matches_header():
    """ctypes mirror of ssd_global_out has the field order and size of the header's declaration; SSD_GLOBAL_U8 agrees."""
    from contracts_b200 import _lib
    text = open(os.path.join(ROOT, "include", "ssd_b200.h")).read()
    body = re.search(r"typedef struct ssd_global_out \{(.*?)\} ssd_global_out;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = [re.sub(r"[\*\s]", "", d.strip().split()[-1]) for d in body.split(";") if d.strip()]
    assert fields == [f[0] for f in _lib.ssd_global_out._fields_]
    assert ctypes.sizeof(_lib.ssd_global_out) == 16
    assert [o for o in (_lib.ssd_global_out.struct_size.offset, _lib.ssd_global_out.dtype.offset, _lib.ssd_global_out.obs_dev.offset)] == [0, 4, 8]
    assert int(re.search(r"#define SSD_GLOBAL_U8 (\d+)", text).group(1)) == _lib.GLOBAL_U8
    assert _lib.GLOBAL_U8 not in _lib.POLICY_DTYPE.values() and _lib.GLOBAL_U8 != _lib.FEATURE_F64
    assert "ssd_set_global_output" in _lib.EXPORTS


def test_set_global_output_rejects_null_handle():
    """No device needed: a NULL handle is SSD_EINVAL, with or without a struct."""
    from contracts_b200 import _lib
    lib = _lib.load()
    out = _lib.ssd_global_out(struct_size=ctypes.sizeof(_lib.ssd_global_out), dtype=_lib.GLOBAL_U8, obs_dev=None)
    assert lib.ssd_set_global_output(None, None) == -1
    assert lib.ssd_set_global_output(None, ctypes.byref(out)) == -1


def test_global_obs_needs_a_device():
    """Without a GPU the batched env fails loudly (no CPU fallback), before any form check could pass silently."""
    import pytest
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from contracts_b200 import _lib
    from contracts_b200.batched import BatchedGridEnv
    with pytest.raises(_lib.SsdError):
        BatchedGridEnv("cleanup_new", 4, 2, global_obs=True)

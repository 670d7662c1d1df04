"""CPU: the grid worlds' feature output C ABI (ssd_feature_out, ssd_set_feature_output) as the bindings declare it."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_feature_out_struct_matches_header():
    """ctypes mirror of ssd_feature_out has the field order and size of the header's declaration; SSD_FEATURE_F64 agrees."""
    from contracts_b200 import _lib
    text = open(os.path.join(ROOT, "include", "ssd_b200.h")).read()
    body = re.search(r"typedef struct ssd_feature_out \{(.*?)\} ssd_feature_out;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = [re.sub(r"[\*\s]", "", d.strip().split()[-1]) for d in body.split(";") if d.strip()]
    assert fields == [f[0] for f in _lib.ssd_feature_out._fields_]
    assert ctypes.sizeof(_lib.ssd_feature_out) == 16
    assert int(re.search(r"#define SSD_FEATURE_F64 (\d+)", text).group(1)) == _lib.FEATURE_F64
    assert _lib.FEATURE_F64 not in _lib.POLICY_DTYPE.values()
    assert "ssd_set_feature_output" in _lib.EXPORTS


def test_set_feature_output_rejects_null_handle():
    """No device needed: a NULL handle is SSD_EINVAL, with or without a struct."""
    from contracts_b200 import _lib
    lib = _lib.load()
    out = _lib.ssd_feature_out(struct_size=ctypes.sizeof(_lib.ssd_feature_out), dtype=_lib.FEATURE_F64, obs_dev=None)
    assert lib.ssd_set_feature_output(None, None) == -1
    assert lib.ssd_set_feature_output(None, ctypes.byref(out)) == -1

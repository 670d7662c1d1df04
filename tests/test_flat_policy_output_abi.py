"""CPU: the flat policy output's C ABI (ssd_flat_policy_out, ssd_set_flat_policy_output) as the bindings declare it."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_flat_policy_out_struct_matches_header():
    """ctypes mirror of ssd_flat_policy_out has the field order and size of the header's declaration."""
    from contracts_b200 import _lib
    text = open(os.path.join(ROOT, "include", "ssd_b200.h")).read()
    body = re.search(r"typedef struct ssd_flat_policy_out \{(.*?)\} ssd_flat_policy_out;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = [re.sub(r"[\*\s]", "", d.strip().split()[-1]) for d in body.split(";") if d.strip()]
    assert fields == [f[0] for f in _lib.ssd_flat_policy_out._fields_]
    assert ctypes.sizeof(_lib.ssd_flat_policy_out) == 16


def test_set_flat_policy_output_rejects_null_handle():
    """No device needed: a NULL handle is SSD_EINVAL, with or without a struct."""
    from contracts_b200 import _lib
    lib = _lib.load()
    out = _lib.ssd_flat_policy_out(struct_size=ctypes.sizeof(_lib.ssd_flat_policy_out), dtype=2, obs_dev=None)
    assert lib.ssd_set_flat_policy_output(None, None) == -1
    assert lib.ssd_set_flat_policy_output(None, ctypes.byref(out)) == -1

"""CPU: every grid-world kernel instantiation in the built library has a row in the oracle-comparison table.

test_cuda_kernel_variants.VARIANTS names the instantiations each configuration launches; a template instantiation added
to the library without a configuration that runs it fails here."""
import os
import re
import shutil
import subprocess

import pytest

from test_cuda_kernel_variants import VARIANTS, variant_kernels

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "contracts_b200", "libssd_b200.so")
FAMILIES = ("grid_obs_kernel", "grid_reset_kernel", "grid_logic_kernel", "grid_logic8_kernel")


def _cuobjdump():
    """cuobjdump beside the nvcc that contracts_b200/build.py uses"""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        nvcc = shutil.which("nvcc") or nvcc
    path = os.path.join(os.path.dirname(nvcc), "cuobjdump")
    return path if os.path.exists(path) else shutil.which("cuobjdump")


def demangle(sym):
    """'_Z15grid_obs_kernelILi1ELi8ELb0ELi0ELi3EEv...' -> 'grid_obs_kernel<1, 8, false, 0, 3>' (None for other symbols)"""
    m = re.match(r"_Z\d+(%s)I((?:L[ib]\d+E)+)E" % "|".join(FAMILIES), sym)
    if not m:
        return None
    args = [("true" if v == "1" else "false") if t == "b" else v for t, v in re.findall(r"L([ib])(\d+)E", m.group(2))]
    return "%s<%s>" % (m.group(1), ", ".join(args))


def test_demangle():
    assert demangle("_Z15grid_obs_kernelILi1ELi8ELb0ELi2ELi3EEv10GridParams6StepIOPj") == "grid_obs_kernel<1, 8, false, 2, 3>"
    assert demangle("_Z18grid_logic8_kernelILi0EEv10GridParams6StepIOPj") == "grid_logic8_kernel<0>"
    assert demangle("_Z17grid_reset_kernelILi1ELi0EEv10GridParamsPKhPhx6StepIOPv") == "grid_reset_kernel<1, 0>"
    assert demangle("_Z18grid_reward_kernel10GridParams6StepIOPKj") is None


def test_every_instantiation_has_a_variant_row():
    if not os.path.exists(LIB):
        pytest.skip("contracts_b200/libssd_b200.so is not built (__graft_entry__.build())")
    tool = _cuobjdump()
    if tool is None:
        pytest.skip("cuobjdump not found beside nvcc")
    out = subprocess.run([tool, "-symbols", LIB], check=True, capture_output=True, text=True).stdout
    entries = [line.split()[-1] for line in out.splitlines() if "STO_ENTRY" in line]
    built = {k for k in map(demangle, entries) if k}
    assert built, "no grid-world kernel entries in %s" % LIB
    listed = {k for v in VARIANTS for f in v.forms for k in variant_kernels(v, f) if k.startswith(FAMILIES)}
    missing, stale = sorted(built - listed), sorted(listed - built)
    assert not missing, "instantiations without a VARIANTS row (tests/test_cuda_kernel_variants.py): %s" % missing
    assert not stale, "VARIANTS names kernels the library does not have: %s" % stale

"""Groups of contexts (pmdi_group_*, pmdi(chains=C)) without a GPU: the group kernel is built for sm_100a within the
register budget of one 512-thread CTA per SM and carried inside the library, and bad input is refused before any
device is touched."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import pmdi_b200  # noqa: F401
from pmdi_b200 import capi

CUBIN = os.path.join(os.path.dirname(capi.LIB_PATH), "pmdi_spec_group.cubin")


def test_group_kernels_fit_one_cta_per_sm_and_ship_in_the_library():
    capi.build()
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([tool, "--dump-resource-usage", CUBIN], capture_output=True, text=True).stdout
    for k in ("k_sweep_spec_group", "k_sweep_spec_group_dbg"):
        m = re.search(r"Function %s:\s*\n\s*REG:(\d+) STACK:(\d+)" % k, out)
        assert m, f"{k} not found in {CUBIN}"
        assert int(m.group(1)) <= 128
    # the group module holds the group kernels and nothing else (a kernel next to them would change their code)
    assert sorted(re.findall(r"Function (\w+):", out)) == ["k_sweep_spec_group", "k_sweep_spec_group_dbg"]
    blob = open(capi.LIB_PATH, "rb").read()
    assert open(CUBIN, "rb").read() in blob


def _create(members, n):
    h = C.c_void_p()
    rc = capi.lib().pmdi_group_create(C.byref(h), members, n)
    return rc, h, capi.lib().pmdi_last_error().decode()


@pytest.mark.parametrize("n", [0, 17, -1])
def test_group_create_rejects_member_counts(n):
    arr = (C.c_void_p * 17)()
    rc, h, msg = _create(arr, n)
    assert rc == 1 and not h.value and "n_members" in msg


def test_group_create_rejects_null_input():
    rc, h, msg = _create(None, 2)
    assert rc == 1 and not h.value and "members is NULL" in msg
    rc, h, msg = _create((C.c_void_p * 2)(), 2)
    assert rc == 1 and not h.value and "member 0" in msg
    assert capi.lib().pmdi_group_run(None) == 1
    assert capi.lib().pmdi_group_destroy(None) == 0


def test_group_without_device_fails_loudly():
    if capi.device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(capi.PmdiError, match="no CPU fallback"):
        capi.Group([capi.Context([np.zeros((10, 2))], [capi.GAUSSIAN], 3, 4)])


@pytest.mark.parametrize("kw,match", [
    (dict(distributed=True), "distributed"),
    (dict(outputFile=["a.csv"]), "3 paths"),
    (dict(K=5), "K <= 4"),
])
def test_pmdi_chains_argument_errors(tmp_path, kw, match):
    from pmdi_b200.pmdi import pmdi
    K = kw.pop("K", 2)
    data = [np.random.default_rng(k).normal(size=(30, 3)) for k in range(K)]
    out = kw.pop("outputFile", [str(tmp_path / f"c{c}.csv") for c in range(3)])
    with pytest.raises(ValueError, match=match):
        pmdi(data, [capi.GAUSSIAN] * K, 4, 8, 0.25, 2, out, chains=3, **kw)

"""Groups of contexts with user-defined cluster types, checked without a GPU: the run-time compile of the group kernels
("spec-group" program, NVRTC cross-compiles for sm_100a) through pmdi_group_type_check, its argument errors, and the
argument errors of pmdi_ctx_set_engine and pmdi(chains=C) with user types that need no device."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import pmdi_b200  # noqa: F401
from pmdi_b200 import capi

import multi_user_types as mu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(code, env=None):
    """`code` in a fresh interpreter: the registry of cluster types and the program cache are per process."""
    e = dict(os.environ, **(env or {}))
    e["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "tests")])
    return subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=e, cwd=ROOT)


@pytest.mark.parametrize("named_cluster", [False, True], ids=["own_names", "both_Cluster"])
def test_group_type_check_compiles_the_spec_group_program(named_cluster):
    """A Gaussian and a NegBinom in one group program; then again from the cache."""
    code = ("import pmdi_b200; from pmdi_b200 import capi; import multi_user_types as mu\n"
            f"tags = mu.register(capi, named_cluster={named_cluster})\n"
            "capi.group_type_check(tags)\n"
            "capi.group_type_check(tags)\n")
    r = _run(code, {"PMDI_JIT_LOG": "1"})
    assert r.returncode == 0, r.stderr[-4000:]
    names = "'GaussianCluster_u', 'NegBinomCluster_u'" if named_cluster else "'MyGaussian', 'MyNegBinom'"
    assert re.search(r"nvrtc compiled %s for the spec-group engine in [0-9.]+ s" % names, r.stderr), r.stderr
    assert "nvrtc cache hit: %s, spec-group engine" % names in r.stderr, r.stderr


def test_words_mismatch_fails_the_group_compile_naming_the_type():
    tag = capi.register_cluster_type("TwoWords", mu.WORDS_MISMATCH, "TwoWords", capi.F64)
    with pytest.raises(capi.PmdiError) as e:
        capi.group_type_check([tag])
    msg = str(e.value)
    assert "static assertion failed" in msg and "cluster type 'TwoWords'" in msg and "WORDS is not 1" in msg


def test_group_type_check_argument_errors():
    L = capi.lib()
    assert L.pmdi_group_type_check(None, 1) == 1
    assert "tags is NULL" in L.pmdi_last_error().decode()
    tags = (C.c_int32 * 9)(*([16] * 9))
    for n in (0, -1, 9):
        assert L.pmdi_group_type_check(tags, n) == 1
        assert "1 <= n <= 8" in L.pmdi_last_error().decode()
    for bad in (0, 2, 15, 10_000):  # built-in tags and unregistered ones
        assert L.pmdi_group_type_check((C.c_int32 * 1)(bad), 1) == 1
        assert "tags[0] is not a registered user type" in L.pmdi_last_error().decode()


def test_set_engine_on_a_null_context_fails():
    L = capi.lib()
    assert L.pmdi_ctx_set_engine(None, 2) == 1
    assert "NULL context" in L.pmdi_last_error().decode()


def test_context_rejects_an_unknown_engine_name():
    with pytest.raises(ValueError, match="engine"):
        capi.Context([np.zeros((10, 2))], [capi.GAUSSIAN], 3, 4, engine="dense")


def test_pmdi_chains_accept_user_types(tmp_path):
    """chains > 1 with a user type is no longer refused by its arguments: without a device it fails where every
    pmdi() run does, at the first context."""
    if capi.device_count() > 0:
        pytest.skip("a CUDA device is present")
    from pmdi_b200.pmdi import pmdi
    counts, expr, _ = mu.planted(n=30)
    out = [str(tmp_path / f"c{c}.csv") for c in range(3)]
    with pytest.raises(capi.PmdiError, match="no CPU fallback"):
        pmdi([counts, expr], list(mu.pmdi_types()), 4, 8, 0.25, 2, out, chains=3)

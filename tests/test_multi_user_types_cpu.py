"""Several user-defined cluster types in one context, checked without a GPU: the run-time compile of a two-type program
for each engine (NVRTC cross-compiles for sm_100a), the compiler's check of WORDS, the statically compiled sweep
kernels' resources, and UserCluster objects handed to another process."""
import os
import pickle
import re
import shutil
import subprocess
import sys

import pytest

import pmdi_b200  # noqa: F401
from pmdi_b200 import capi

import multi_user_types as mu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(code, env=None):
    """`code` in a fresh interpreter: the registry of cluster types is per process."""
    e = dict(os.environ, **(env or {}))
    e["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "tests")])
    return subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=e, cwd=ROOT)


@pytest.mark.parametrize("engine", ["pool", "spec"])
def test_two_types_named_cluster_compile_into_one_program(engine):
    """A Gaussian and a NegBinom that both call their struct `Cluster`, in one program of each engine."""
    code = ("import pmdi_b200; from pmdi_b200 import capi; import multi_user_types as mu\n"
            "mu.register(capi, named_cluster=True)\n"
            "capi.cluster_type_check(-1)\n")
    r = _run(code, {"PMDI_ENGINE": engine, "PMDI_JIT_LOG": "1"})
    assert r.returncode == 0, r.stderr[-4000:]
    assert re.search(r"nvrtc compiled 'GaussianCluster_u', 'NegBinomCluster_u' for the %s engine" % engine, r.stderr), r.stderr


def test_words_text_that_disagrees_with_the_struct_is_a_compile_error_naming_the_type():
    """The first `WORDS = ` of the text (a comment here) says 1, the struct has 2: the arena would be sized for 1."""
    tag = capi.register_cluster_type("TwoWords", mu.WORDS_MISMATCH, "TwoWords", capi.F64)
    with pytest.raises(capi.PmdiError) as e:
        capi.cluster_type_check(tag)
    msg = str(e.value)
    assert "static assertion failed" in msg and "cluster type 'TwoWords'" in msg and "WORDS is not 1" in msg


def test_static_sweep_kernels_keep_their_resources():
    """User-type code is compiled only into run-time programs: the statically compiled sweep kernels keep the
    register count and stack frame of the measured build (spec 128 / 352 B, pool 128 / 528 B)."""
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    capi.build()
    out = subprocess.run([tool, "--dump-resource-usage", capi.LIB_PATH], capture_output=True, text=True).stdout
    for name, stack in (("k_sweep_spec", 352), ("k_sweep_pool", 528)):
        m = re.search(r"Function %s:\s*\n\s*REG:(\d+) STACK:(\d+)" % name, out)
        assert m, f"{name} not found in the library"
        assert (int(m.group(1)), int(m.group(2))) == (128, stack), name


def test_user_cluster_registers_itself_in_another_process():
    """A rank of a distributed run gets the UserCluster objects pickled: reading `tag` there registers the type in
    that process, under the tag that process gives it."""
    from pmdi_b200 import pmdi as host
    ng = host.UserCluster("MyNegBinom", mu.USER_NEGBINOM, integer_data=True)
    blob = pickle.dumps(ng).hex()
    code = ("import pickle, pmdi_b200; from pmdi_b200 import capi; import user_types as ut\n"
            "first = capi.register_cluster_type('MyPoisson', ut.USER_POISSON, 'MyPoisson', capi.I64)\n"
            f"t = pickle.loads(bytes.fromhex('{blob}'))\n"
            "assert t.tag == first + 1 and t.tag == t.tag, t.tag\n")
    r = _run(code)
    assert r.returncode == 0, r.stderr[-4000:]

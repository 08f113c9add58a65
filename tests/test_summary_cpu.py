"""Posterior summaries without a GPU: the CSV reader, argument errors raised before any device call, the exported
symbols, and the resources of the summary kernels."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import pmdi_b200  # noqa: F401
from pmdi_b200 import capi
from pmdi_b200 import pmdi as host

SUMMARY_EXPORTS = ["pmdi_summary_create", "pmdi_summary_add", "pmdi_summary_rows", "pmdi_summary_psm",
                   "pmdi_summary_ls", "pmdi_summary_agreement", "pmdi_summary_destroy", "pmdi_parse_allocations"]


def _write(path, K, n, names, allocs, seed=0):
    rng = np.random.default_rng(seed)
    with open(path, "w") as f:
        f.write(host.csv_header(K, n, names) + "\n")
        for r, a in enumerate(allocs):
            phi = rng.gamma(1.0, 0.2, K * (K - 1) // 2) if K > 1 else np.zeros(1)
            f.write(host.csv_row(rng.gamma(2.0, 1.0, K), phi, 1.25e-5 * r, a) + "\n")


@pytest.mark.parametrize("K,n", [(1, 9), (3, 17)])
def test_read_chains_infers_the_layout_and_equals_read_allocations(tmp_path, K, n):
    rng = np.random.default_rng(K)
    names = [f"set_n{k}" for k in range(K)]  # "_n" inside a name too
    paths = []
    for c in range(2):
        p = str(tmp_path / f"c{c}.csv")
        _write(p, K, n, names, rng.integers(1, 257, (11, n, K)), seed=c)
        paths.append(p)
    if K == 1:
        assert host.csv_header(K, n, names).split(",")[1] == "phi_1_1"
    for burnin, thin in ((0, 1), (3, 2)):
        chains, got_names = host.read_chains(paths, burnin, thin)
        assert got_names == names and len(chains) == 2
        for p, a in zip(paths, chains):
            ref = host.read_allocations(p, K, n, burnin, thin)
            assert a.dtype == np.int64 and a.shape == ref.shape
            np.testing.assert_array_equal(a, ref)
    one, _ = host.read_chains(paths[0])
    assert len(one) == 1


def test_read_chains_refuses_a_malformed_file(tmp_path):
    p = tmp_path / "bad.csv"
    p.write_text(host.csv_header(1, 2, ["x"]) + "\n2.0,0.0,0.1,1.0,2.5\n")
    with pytest.raises(ValueError, match="not an integer"):
        host.read_chains(str(p))
    q = tmp_path / "other.csv"
    q.write_text("a,b,c\n1,2,3\n")
    with pytest.raises(ValueError, match="header"):
        host.read_chains(str(q))


def test_parse_allocations_reads_integer_labels_and_refuses_the_rest():
    text = b"2.0,1.5e-5,7.0,256.0,10\n2.0,0.0,1.0,2.0,30.0\n"
    np.testing.assert_array_equal(capi.parse_allocations(text, 2, 2, 3), [[7, 256, 10], [1, 2, 30]])
    np.testing.assert_array_equal(capi.parse_allocations(text.rstrip(b"\n"), 2, 2, 3), [[7, 256, 10], [1, 2, 30]])
    for bad, rows, what in ((b"2.0,1.0,7.5,1.0,1.0", 1, "expected ','"), (b"2.0,1.0,7.0,1.0", 1, "expected ','"),
                            (b"2.0,1.0,7.0,1.0,1.0,1.0", 1, "more columns"), (b"2.0,1.0,-7.0,1.0,1.0", 1, "integer label"),
                            (b"2.0\n", 1, "fewer columns"), (b"2.0,1.0,7.0,1.0,1.0\n", 2, "fewer")):
        with pytest.raises(ValueError, match=what):
            capi.parse_allocations(bad, rows, 2, 3)


@pytest.mark.parametrize("kw", [dict(K=0), dict(K=9), dict(n_obs=0), dict(n_obs=65536), dict(N=257), dict(N=0),
                                dict(chains=0), dict(chains=65), dict(burnin=-1), dict(thin=0)])
def test_python_argument_errors_come_before_the_device(kw):
    args = dict(K=2, n_obs=10, N=5, chains=1, burnin=0, thin=1)
    args.update(kw)
    with pytest.raises(ValueError):
        capi.PosteriorSummary(**args)


@pytest.mark.parametrize("K,n,N,chains", [(0, 10, 5, 1), (9, 10, 5, 1), (1, 65536, 5, 1), (1, 10, 257, 1),
                                          (1, 10, 5, 0), (1, 10, 5, 65)])
def test_summary_create_preconditions(K, n, N, chains):
    h = C.c_void_p()
    assert capi.lib().pmdi_summary_create(C.byref(h), 0, K, n, N, chains) == 1 and not h.value
    assert capi.lib().pmdi_last_error()


def test_pmdi_refuses_summary_with_distributed():
    class S:
        K, n, N, chains = 1, 12, 3, 1
    data = [np.zeros((12, 2))]
    with pytest.raises(ValueError, match="distributed"):
        host.pmdi(data, [host.GaussianCluster], 3, 4, 0.5, 1, "/dev/null", distributed=True, summary=S())


def test_library_exports_the_summary_calls():
    capi.build()
    L = capi.lib()
    for s in SUMMARY_EXPORTS:
        assert s in capi.EXPORTS and hasattr(L, s)


def test_summary_kernels_use_no_stack():
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    capi.build()
    out = subprocess.run([tool, "--dump-resource-usage", capi.LIB_PATH], capture_output=True, text=True).stdout
    found = re.findall(r"Function (\w*k_summary_\w+):\s*\n\s*REG:(\d+) STACK:(\d+)", out)
    names = {re.search(r"k_summary_[a-z]+", f).group(0) for f, _, _ in found}
    assert names == {"k_summary_count", "k_summary_put", "k_summary_get", "k_summary_psm", "k_summary_ls",
                     "k_summary_agree"}
    for f, regs, stack in found:
        assert int(stack) == 0, f

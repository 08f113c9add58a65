"""Several user-defined cluster types in one context, and user types on the speculative engine, on one GPU.  The
user restatements of the built-in Gaussian and NegBinom types must reproduce the built-ins: allocations, ancestors,
selected particle, final allocations, cluster sizes and resampling count bit for bit, log-probabilities and
log-weights to 1e-9 (the built-ins hoist terms into per-size tables, the user types sum per-feature terms)."""
import numpy as np
import pytest

import multi_user_types as mu
import user_types as ut
from helpers import C, G, NB, problem, tapes_for

pytestmark = pytest.mark.gpu


def _sweep(pr, types, tapes):
    from pmdi_b200 import capi
    with capi.Context(pr["data"], types, pr["N"], pr["P"]) as ctx:
        return ctx.sweep(pr["s"], pr["order"], pr["n1"], pr["Pi"], pr["phi"], seed=3, it=2, tapes=tapes, debug=True)


def _assert_same(a, b):
    np.testing.assert_array_equal(a["alloc"], b["alloc"])
    np.testing.assert_array_equal(a["anc"], b["anc"])
    np.testing.assert_array_equal(a["s"], b["s"])
    np.testing.assert_array_equal(a["cluster_n"], b["cluster_n"])
    assert a["p_star"] == b["p_star"] and a["n_resamples"] == b["n_resamples"] and a["n_resamples"] > 0
    np.testing.assert_allclose(b["lp"], a["lp"], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(b["lw"], a["lw"], rtol=1e-9, atol=1e-9)


def test_user_gaussian_on_the_spec_engine_reproduces_the_builtin(monkeypatch):
    from pmdi_b200 import capi
    monkeypatch.setenv("PMDI_ENGINE", "spec")
    tag = capi.register_cluster_type("MyGaussian", ut.USER_GAUSSIAN, "MyGaussian", capi.F64)
    pr = problem(sets=[(G, 130, 0), (NB, 70, 0), (G, 40, 0)], n=110, N=9, P=48, seed=6)
    tapes = tapes_for(pr)
    a = _sweep(pr, pr["types"], tapes)
    b = _sweep(pr, [tag, pr["types"][1], tag], tapes)
    assert a["engine"] == "spec" and b["engine"] == "spec"
    _assert_same(a, b)


@pytest.mark.parametrize("named_cluster", [False, True], ids=["own_names", "both_Cluster"])
@pytest.mark.parametrize("engine", ["pool", "spec"])
def test_two_user_types_in_one_context_reproduce_the_builtins(engine, named_cluster, monkeypatch):
    """[user Gaussian, user NegBinom, Categorical] against [Gaussian, NegBinom, Categorical]; then the same with two
    sources whose structs are both named `Cluster`."""
    from pmdi_b200 import capi
    monkeypatch.setenv("PMDI_ENGINE", engine)
    tg, tn = mu.register(capi, named_cluster)
    pr = problem(sets=[(G, 130, 0), (NB, 70, 0), (C, 40, 3)], n=110, N=9, P=48, seed=6)
    tapes = tapes_for(pr)
    a = _sweep(pr, pr["types"], tapes)
    b = _sweep(pr, [tg, tn, pr["types"][2]], tapes)
    assert a["engine"] == engine and b["engine"] == engine
    _assert_same(a, b)


def test_default_engine_for_user_types_on_one_gpu_is_pool(monkeypatch):
    from pmdi_b200 import capi
    monkeypatch.delenv("PMDI_ENGINE", raising=False)
    tg, tn = mu.register(capi)
    pr = problem(sets=[(G, 64, 0), (NB, 33, 0)], n=64, N=5, P=32, seed=2)
    assert _sweep(pr, [tg, tn], None)["engine"] == "pool"
    monkeypatch.setenv("PMDI_ENGINE", "dense")   # the dense engine has no user hooks
    assert _sweep(pr, [tg, tn], None)["engine"] == "pool"


def test_second_context_with_the_same_types_does_not_recompile(monkeypatch, capfd):
    """Checked through the compile log the library writes to stderr with PMDI_JIT_LOG set."""
    from pmdi_b200 import capi
    monkeypatch.setenv("PMDI_JIT_LOG", "1")
    monkeypatch.setenv("PMDI_ENGINE", "spec")
    tg, tn = mu.register(capi)
    pr = problem(sets=[(G, 64, 0), (NB, 33, 0)], n=64, N=5, P=32, seed=2)
    a = _sweep(pr, [tg, tn], None)
    capfd.readouterr()
    b = _sweep(pr, [tg, tn], None)
    err = capfd.readouterr().err
    assert "pmdi: nvrtc cache hit: 'MyGaussian', 'MyNegBinom', spec engine" in err, err
    assert "nvrtc compiled" not in err, err
    np.testing.assert_array_equal(a["alloc"], b["alloc"])


def test_pmdi_with_two_user_types_recovers_planted_clusters(tmp_path):
    from pmdi_b200 import pmdi as host
    counts, expr, z = mu.planted()
    out = tmp_path / "o.csv"
    host.pmdi([counts, expr], list(mu.pmdi_types()), 6, 32, 0.25, 30, str(out), seed=1)
    alloc = host.read_allocations(str(out), 2, len(z), burnin=10)
    psm = host.posterior_similarity(alloc)
    same = z[:, None] == z[None, :]
    for k in range(2):
        assert psm[k][same].mean() > 0.85 and psm[k][~same].mean() < 0.1, k

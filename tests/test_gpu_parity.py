"""GPU parity: libpmdi_cuda.so (through the C-ABI) against the CPU oracle on the same inputs.

Bars (BASELINE.json north_star): allocations, ancestors and the selected particle bit-exact in
deterministic mode (shared uniforms); per-step log-probs and log-weights within 1e-5 relative
(measured: ~1e-13).
"""
import numpy as np
import pytest

from helpers import C, G, NB, problem, tapes_for

pytestmark = pytest.mark.gpu

RTOL = 1e-5  # north_star tolerance for floating-point outputs


# the speculative engine (the default for K <= 4), the copy-on-write pool (the default above) and the dense form,
# selected by PMDI_ENGINE
ENGINES = ["spec", "pool", "dense"]


def _run_both(pr, tapes=None, seed=11, it=3, lw0=0.0, flags=None, engine="pool"):
    import os
    from oracle import oracle as orc
    import pmdi_b200.capi as capi
    os.environ["PMDI_ENGINE"] = engine
    o = orc.Oracle(pr["data"], pr["types"], pr["N"], pr["P"])
    ctx = capi.Context(pr["data"], pr["types"], pr["N"], pr["P"])
    if flags is not None:
        for k, f in enumerate(flags):
            o.set_flags(k, f)
            ctx.set_flags(k, f)
    ref = o.sweep(pr["s"], pr["order"], pr["n1"], pr["Pi"], pr["phi"], mode=orc.MODE_DENSE,
                  logweight_init=lw0, seed=seed, it=it, tapes=tapes, debug=True)
    got = ctx.sweep(pr["s"], pr["order"], pr["n1"], pr["Pi"], pr["phi"], logweight_init=lw0,
                    seed=seed, it=it, tapes=tapes, debug=True)
    ctx.close()
    os.environ.pop("PMDI_ENGINE", None)
    assert got["engine"] == engine
    return ref, got


def _assert_parity(pr, ref, got):
    np.testing.assert_array_equal(got["alloc"], ref["alloc"])
    np.testing.assert_array_equal(got["anc"], ref["anc"])
    assert got["p_star"] == ref["p_star"]
    np.testing.assert_array_equal(got["s"], ref["s"])
    np.testing.assert_array_equal(got["cluster_n"], ref["cluster_n"])
    assert got["n_resamples"] == ref["n_resamples"]
    np.testing.assert_allclose(got["lp"], ref["lp"], rtol=RTOL, atol=1e-9)
    np.testing.assert_allclose(got["lw"], ref["lw"], rtol=RTOL, atol=1e-9)
    np.testing.assert_allclose(got["logweight"], ref["logweight"], rtol=RTOL, atol=1e-9)
    # structural invariants of test/runtests.jl:147 in dense form
    assert (got["cluster_n"].sum(axis=2) == pr["n"]).all()


CASES = {
    "gauss_small": dict(sets=[(G, 4, 0)], n=60, N=6, P=8),
    "gauss_iris_shape": dict(sets=[(G, 4, 0)], n=150, N=10, P=32),
    "gauss_wide": dict(sets=[(G, 300, 0)], n=80, N=8, P=48),
    "cat": dict(sets=[(C, 70, 3)], n=80, N=8, P=32),
    "negbinom": dict(sets=[(NB, 90, 0)], n=80, N=8, P=32),
    "mixed_k3": dict(sets=[(G, 130, 0), (C, 65, 3), (NB, 100, 0)], n=120, N=12, P=64),
    "mixed_k2_manyP": dict(sets=[(G, 64, 0), (NB, 33, 0)], n=64, N=5, P=700),
    "gauss_N40": dict(sets=[(G, 20, 0), (G, 10, 0)], n=100, N=40, P=40),
}


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("name", list(CASES))
def test_sweep_matches_oracle_philox(name, engine):
    pr = problem(**CASES[name], seed=3)
    ref, got = _run_both(pr, engine=engine)
    _assert_parity(pr, ref, got)


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("name", ["gauss_small", "mixed_k3"])
def test_sweep_matches_oracle_tapes(name, engine):
    """Deterministic mode proper: the uniforms are fed in as tapes."""
    pr = problem(**CASES[name], seed=4)
    ref, got = _run_both(pr, tapes=tapes_for(pr), lw0=1.0, engine=engine)
    _assert_parity(pr, ref, got)
    if name == "mixed_k3":
        assert ref["n_resamples"] > 0  # the resampling path is exercised


@pytest.mark.parametrize("engine", ENGINES)
def test_sweep_with_feature_flags(engine):
    pr = problem(**CASES["mixed_k3"], seed=6)
    rng = np.random.default_rng(0)
    flags = [(rng.random(d.shape[1]) < 0.6).astype(np.uint8) for d in pr["data"]]
    ref, got = _run_both(pr, flags=flags, engine=engine)
    _assert_parity(pr, ref, got)


@pytest.mark.parametrize("engine", ["pool", "dense"])
@pytest.mark.parametrize("name", ["gauss_wide", "mixed_k3", "mixed_k2_manyP"])
@pytest.mark.parametrize("qb", ["1", "8"])
def test_parity_for_other_item_sizes(name, qb, engine, monkeypatch):
    """The number of 256-feature blocks per work item is chosen per workload / per step (whole rows when
    there are many rows per warp); parity must not depend on it.  Only the dense engine's work items read
    PMDI_QB, so the spec engine is left out here: the other tests of this file run it on these cases."""
    monkeypatch.setenv("PMDI_QB", qb)
    pr = problem(**CASES[name], seed=5)
    ref, got = _run_both(pr, lw0=1.0, engine=engine)
    _assert_parity(pr, ref, got)


DISTINCT = ["gauss_iris_shape", "mixed_k3", "mixed_k2_manyP", "gauss_N40"]


def _assert_evaluates_each_distinct_cluster_once(name, engine):
    from oracle import oracle as orc
    pr = problem(**CASES[name], seed=7)
    ref, got = _run_both(pr, lw0=1.0, engine=engine)
    _assert_parity(pr, ref, got)
    o = orc.Oracle(pr["data"], pr["types"], pr["N"], pr["P"])
    dd = o.sweep(pr["s"], pr["order"], pr["n1"], pr["Pi"], pr["phi"], mode=orc.MODE_DEDUP, logweight_init=1.0,
                 seed=11, it=3)
    np.testing.assert_array_equal(dd["s"], got["s"])
    # evaluation runs one observation ahead of the resampling decision: rows that a resampling removes were
    # evaluated once more than in the reference; the kernel counts them
    assert sum(got["rows_evaluated"]) - got["rows_evaluated_ahead"] == dd["n_ops"]
    assert sum(got["rows_referenced"]) >= sum(got["rows_evaluated"]) - pr["K"] * (pr["n"] - pr["n1"] + 1)


@pytest.mark.parametrize("name", DISTINCT)
def test_pool_evaluates_each_distinct_cluster_once(name):
    """The copy-on-write pool performs exactly the reference's calc_logprob calls: one per distinct
    cluster per (observation, dataset) - the oracle's de-duplicated mode counts them the way
    src/__pmdi.jl:187 does (n_operations)."""
    _assert_evaluates_each_distinct_cluster_once(name, "pool")


@pytest.mark.parametrize("name", DISTINCT)
def test_spec_evaluates_each_distinct_cluster_once(name):
    """The same count for the speculative engine, whose evaluation CTAs walk the live-row list one
    observation ahead of the resampling decision."""
    _assert_evaluates_each_distinct_cluster_once(name, "spec")


def test_sstar_compat_flag():
    """pmdi()'s own (unpermuted) trajectory emission, src/pmdi.jl:321-324."""
    from oracle import oracle as orc
    import pmdi_b200.capi as capi
    pr = problem(**CASES["mixed_k3"], seed=9)
    o = orc.Oracle(pr["data"], pr["types"], pr["N"], pr["P"])
    ref = o.sweep(pr["s"], pr["order"], pr["n1"], pr["Pi"], pr["phi"],
                  mode=orc.MODE_DENSE | orc.MODE_SSTAR_COMPAT, seed=2, it=1)
    with capi.Context(pr["data"], pr["types"], pr["N"], pr["P"]) as ctx:
        got = ctx.sweep(pr["s"], pr["order"], pr["n1"], pr["Pi"], pr["phi"], seed=2, it=1, sstar_compat=True)
    assert ref["n_resamples"] > 0
    np.testing.assert_array_equal(got["s"], ref["s"])
    assert got["p_star"] == ref["p_star"]


EDGE = {
    "smallest_N_P_empty_prefix": dict(sets=[(G, 3, 0), (C, 2, 2)], n=12, N=2, P=2, rho=0.1),
    "one_step": dict(sets=[(NB, 5, 0)], n=10, N=3, P=4, rho=0.999),
    "ragged_widths": dict(sets=[(G, 1, 0), (G, 257, 0), (C, 63, 5), (NB, 65, 0)], n=40, N=4, P=9),
    "N_equals_n": dict(sets=[(G, 6, 0)], n=16, N=16, P=12),
}


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("name", list(EDGE))
def test_edge_cases(name, engine):
    pr = problem(**EDGE[name], seed=10)
    ref, got = _run_both(pr, lw0=1.0, engine=engine)
    _assert_parity(pr, ref, got)


@pytest.mark.parametrize("name", __import__("helpers").GOLDEN)
def test_cuda_matches_golden_fixture(name):
    """Committed fixtures (tests/golden/make_golden.py): no oracle at run time."""
    from helpers import assert_matches_golden, load_golden
    import pmdi_b200.capi as capi
    pr, tapes, z = load_golden(name)
    with capi.Context(pr["data"], pr["types"], pr["N"], pr["P"]) as ctx:
        got = ctx.sweep(pr["s"], pr["order"], pr["n1"], pr["Pi"], pr["phi"], seed=int(z["seed"]),
                        it=int(z["it"]), tapes=tapes, debug=True, logweight_init=float(z["lw0"]))
    assert_matches_golden(got, z, rtol=RTOL)


def test_chained_sweeps_match_oracle():
    """Three MCMC iterations through one context (state is rebuilt per sweep, src/pmdi.jl:165-172)."""
    from oracle import oracle as orc
    import pmdi_b200.capi as capi
    pr = problem(**CASES["mixed_k3"], seed=11)
    o = orc.Oracle(pr["data"], pr["types"], pr["N"], pr["P"])
    rng = np.random.default_rng(3)
    s_ref = s_got = pr["s"]
    with capi.Context(pr["data"], pr["types"], pr["N"], pr["P"]) as ctx:
        for it in range(3):
            order = rng.permutation(pr["n"]) + 1
            ref = o.sweep(s_ref, order, pr["n1"], pr["Pi"], pr["phi"], seed=8, it=it, logweight_init=float(it > 0))
            got = ctx.sweep(s_got, order, pr["n1"], pr["Pi"], pr["phi"], seed=8, it=it, logweight_init=float(it > 0))
            np.testing.assert_array_equal(got["s"], ref["s"])
            assert got["p_star"] == ref["p_star"]
            s_ref, s_got = ref["s"], got["s"]


def test_argument_errors_are_reported():
    import pmdi_b200.capi as capi
    pr = problem(**CASES["gauss_small"], seed=3)
    with capi.Context(pr["data"], pr["types"], pr["N"], pr["P"]) as ctx:
        bad = pr["order"].copy()
        bad[0] = bad[1]
        with pytest.raises(capi.PmdiError, match="permutation"):
            ctx.sweep(pr["s"], bad, pr["n1"], pr["Pi"], pr["phi"])
        s_bad = pr["s"].copy()
        s_bad[0, 0] = pr["N"] + 1
        with pytest.raises(capi.PmdiError, match="label"):
            ctx.sweep(s_bad, pr["order"], pr["n1"], pr["Pi"], pr["phi"])
        with pytest.raises(capi.PmdiError, match="n1"):
            ctx.sweep(pr["s"], pr["order"], 0, pr["Pi"], pr["phi"])

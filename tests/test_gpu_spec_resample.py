"""The speculative engine's resampling event against the CPU oracle, with the bounds checks of the instrumented kernel
(debug=True: a row id outside its pool or a list longer than its storage ends the sweep with an error), and with its
pool accounting at the end of every sweep on one GPU: every row id of a dataset must be in exactly one place - the free
stack, one evaluation CTA's free-id cache, the live-row list with the rows' children, or the empty row and its child -
so a leaked row or one freed or handed out twice fails the sweep (error 97).

The problems and seeds are chosen so that the oracle's run resamples at the places where the event's bookkeeping
differs (each test asserts from the oracle's output that it did):
  - early: after step 1 (after step 0 every particle carries the same weight, so the ESS test never fires there);
  - after two or more consecutive steps: the event runs on a list the previous event rebuilt;
  - after the second-to-last step: no ids were handed out for the step after the next;
  - after the last step: the final resampling, which only moves the row maps.
"""
import os

import numpy as np
import pytest

from helpers import C, G, problem, tapes_for

pytestmark = pytest.mark.gpu

RTOL = 1e-5

SHARP = dict(sets=[(G, 200, 0), (C, 200, 3)], n=24, N=6, P=64)
CASES = {  # name: (problem, where the oracle resamples)
    "early_and_runs": (dict(**SHARP, rho=0.05, seed=3), ("early", "consecutive")),
    "last_step": (dict(**SHARP, rho=0.05, seed=4), ("last",)),
    "runs_to_the_end": (dict(**SHARP, rho=0.25, seed=3), ("consecutive", "second_to_last", "last")),
    "second_to_last": (dict(sets=[(G, 20, 0), (G, 10, 0)], n=100, N=40, P=40, seed=2), ("second_to_last",)),
}


def _resampled(ref):
    return ref["anc"].any(axis=1)  # the oracle records ancestors at the steps that resampled


def _reached(res, what):
    return {"early": bool(res[1]),
            "consecutive": any(res[i] and res[i + 1] for i in range(len(res) - 1)),
            "second_to_last": bool(res[-2]),
            "last": bool(res[-1])}[what]


def _oracle(pr, **kw):
    from oracle import oracle as orc
    o = orc.Oracle(pr["data"], pr["types"], pr["N"], pr["P"])
    return o.sweep(pr["s"], pr["order"], pr["n1"], pr["Pi"], pr["phi"], mode=orc.MODE_DENSE, debug=True, **kw)


def _ctx(pr):
    import pmdi_b200.capi as capi
    return capi.Context(pr["data"], pr["types"], pr["N"], pr["P"], engine="spec")


def _assert_parity(got, ref):
    np.testing.assert_array_equal(got["alloc"], ref["alloc"])
    np.testing.assert_array_equal(got["anc"], ref["anc"])
    assert got["p_star"] == ref["p_star"]
    np.testing.assert_array_equal(got["s"], ref["s"])
    np.testing.assert_array_equal(got["cluster_n"], ref["cluster_n"])
    assert got["n_resamples"] == ref["n_resamples"]
    np.testing.assert_allclose(got["lp"], ref["lp"], rtol=RTOL, atol=1e-9)
    np.testing.assert_allclose(got["lw"], ref["lw"], rtol=RTOL, atol=1e-9)
    np.testing.assert_allclose(got["logweight"], ref["logweight"], rtol=RTOL, atol=1e-9)


@pytest.mark.parametrize("name", list(CASES))
def test_resampling_event_matches_oracle(name):
    spec, where = CASES[name]
    pr = problem(**spec)
    kw = dict(logweight_init=1.0, seed=11, it=3, tapes=tapes_for(pr))
    ref = _oracle(pr, **kw)
    res = _resampled(ref)
    for w in where:
        assert _reached(res, w), f"{name}: the oracle did not resample {w} ({res.astype(int)})"
    with _ctx(pr) as ctx:
        got = ctx.sweep(pr["s"], pr["order"], pr["n1"], pr["Pi"], pr["phi"], debug=True, **kw)
    assert got["engine"] == "spec"
    _assert_parity(got, ref)


def test_chained_sweeps_with_resamplings():
    """Tens of sweeps through one context, each with several resamplings, the allocations carried from sweep to
    sweep.  Every sweep runs the checked kernel, whose pool accounting fails the sweep on a row the events leaked or
    freed twice; a row freed while still referenced changes the results the oracle checks."""
    from oracle import oracle as orc
    pr = problem(**SHARP, rho=0.05, seed=1)
    o = orc.Oracle(pr["data"], pr["types"], pr["N"], pr["P"])
    rng = np.random.default_rng(3)
    s_ref = s_got = pr["s"]
    events = 0
    with _ctx(pr) as ctx:
        for it in range(24):
            order = rng.permutation(pr["n"]) + 1
            kw = dict(seed=8, it=it, logweight_init=float(it > 0))
            ref = o.sweep(s_ref, order, pr["n1"], pr["Pi"], pr["phi"], **kw)
            got = ctx.sweep(s_got, order, pr["n1"], pr["Pi"], pr["phi"], debug=True, **kw)
            np.testing.assert_array_equal(got["s"], ref["s"])
            assert got["p_star"] == ref["p_star"]
            assert got["n_resamples"] == ref["n_resamples"]
            events += got["n_resamples"]
            s_ref, s_got = ref["s"], got["s"]
    assert events >= 24 * 3


def test_group_member_resamples_as_alone():
    """Two contexts in one group launch: each member's sweep, resamplings included, equals the same context swept
    alone."""
    import pmdi_b200.capi as capi
    prs = [problem(**SHARP, rho=0.05, seed=3), problem(**SHARP, rho=0.25, seed=3)]
    args = [dict(s=pr["s"], order_obs=pr["order"], n1=pr["n1"], Pi=pr["Pi"], phi=pr["phi"], seed=5, it=2,
                 logweight_init=1.0) for pr in prs]
    ctxs = [_ctx(pr) for pr in prs]
    with capi.Group(ctxs) as grp:
        got = grp.sweep(args)
    for ctx, pr, a, g in zip(ctxs, prs, args, got):
        assert g["n_resamples"] > 0
        with _ctx(pr) as alone:
            alone.upload(**a)
            alone.run()
            r = alone.download()
        assert r["n_resamples"] == g["n_resamples"] and r["p_star"] == g["p_star"]
        np.testing.assert_array_equal(r["s"], g["s"])
        np.testing.assert_array_equal(r["logweight"], g["logweight"])
        ctx.close()

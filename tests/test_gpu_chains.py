"""Groups: several contexts (chains) swept in one launch of the spec engine (pmdi_group_*, capi.Group,
pmdi(chains=C)).  A member's results must be those of the member swept alone - bit for bit - whatever share of the
SMs it runs on; mixed members must match the oracle as a single context does."""
import os

import numpy as np
import pytest

from helpers import C, G, NB, problem, tapes_for

pytestmark = pytest.mark.gpu

EXACT = ["s", "p_star", "label_counts", "pair_agree", "contingency", "rows_evaluated", "rows_added",
         "n_resamples", "cluster_n"]
RTOL = 1e-5

SAME = dict(sets=[(G, 130, 0), (C, 65, 3), (NB, 100, 0)], n=120, N=12, P=64)


def _ctx(pr):
    import pmdi_b200.capi as capi
    return capi.Context(pr["data"], pr["types"], pr["N"], pr["P"])


def _args(pr, seed=11, it=3, lw0=1.0, tapes=None, debug=False, s=None, order=None):
    return dict(s=pr["s"] if s is None else s, order_obs=pr["order"] if order is None else order, n1=pr["n1"],
                Pi=pr["Pi"], phi=pr["phi"], seed=seed, it=it, logweight_init=lw0, tapes=tapes, debug=debug)


def _alone(ctx, a):
    ctx.upload(**a)
    ctx.run()
    return ctx.download()


def _assert_same(got, ref):
    for k in EXACT:
        np.testing.assert_array_equal(np.asarray(got[k]), np.asarray(ref[k]), err_msg=k)
    np.testing.assert_allclose(got["logweight"], ref["logweight"], rtol=1e-12, atol=0)


def _members():
    """Three members with one problem and three seeds, one that resamples often (fed-in tapes), one settled."""
    same = problem(**SAME, seed=3)
    heavy = problem(**SAME, seed=4)
    settled = problem(sets=[(G, 4, 0)], n=150, N=10, P=32, seed=5)
    return [(same, _args(same, seed=s)) for s in (11, 12, 13)] + \
        [(heavy, _args(heavy, tapes=tapes_for(heavy))), (settled, _args(settled, seed=2, lw0=0.0))]


def test_group_equals_alone():
    import pmdi_b200.capi as capi
    members = _members()
    ctxs = [_ctx(pr) for pr, _ in members]
    with capi.Group(ctxs) as grp:
        got = grp.sweep([a for _, a in members])
        assert got[3]["n_resamples"] > 0  # the resampling path ran inside the group
        for ctx, (pr, a), g in zip(ctxs, members, got):
            assert g["engine"] == "spec" and g["sweep_kernel_ms"] > 0
            _assert_same(g, _alone(ctx, a))      # alone on the member's share of the SMs
            with _ctx(pr) as fresh:              # alone on the whole GPU
                _assert_same(g, _alone(fresh, a))
    for ctx in ctxs:
        ctx.close()


def _oracle(pr, a):
    from oracle import oracle as orc
    o = orc.Oracle(pr["data"], pr["types"], pr["N"], pr["P"])
    return o.sweep(a["s"], a["order_obs"], a["n1"], a["Pi"], a["phi"], mode=orc.MODE_DENSE,
                   logweight_init=a["logweight_init"], seed=a["seed"], it=a["it"], tapes=a["tapes"], debug=True)


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


MIXED = [  # (problem, tapes?) - K 1..4, other N, P, n and types, the edge shapes of test_gpu_parity.py
    (dict(sets=[(G, 130, 0), (C, 65, 3), (NB, 100, 0)], n=120, N=12, P=64), True),
    (dict(sets=[(G, 20, 0), (G, 10, 0)], n=100, N=40, P=40), False),
    (dict(sets=[(G, 3, 0), (C, 2, 2)], n=12, N=2, P=2, rho=0.1), True),
    (dict(sets=[(NB, 5, 0)], n=10, N=3, P=4, rho=0.999), False),
    (dict(sets=[(G, 1, 0), (G, 257, 0), (C, 63, 5), (NB, 65, 0)], n=40, N=4, P=9), True),
    (dict(sets=[(C, 70, 3)], n=80, N=8, P=32), False),
]


def test_mixed_group_matches_oracle():
    import pmdi_b200.capi as capi
    prs = [problem(**cfg, seed=10 + i) for i, (cfg, _) in enumerate(MIXED)]
    args = [_args(pr, seed=20 + i, tapes=tapes_for(pr) if t else None, debug=True)
            for i, (pr, (_, t)) in enumerate(zip(prs, MIXED))]
    # one member without debug capture: it runs the instrumented twin with the others and captures nothing
    plain = problem(**SAME, seed=9)
    ctxs = [_ctx(pr) for pr in prs + [plain]]
    with capi.Group(ctxs) as grp:
        got = grp.sweep(args + [_args(plain, seed=5)])
    for pr, a, g in zip(prs, args, got):
        _assert_parity(g, _oracle(pr, a))
    with _ctx(plain) as fresh:
        _assert_same(got[-1], _alone(fresh, _args(plain, seed=5)))
    assert "lp" not in got[-1]
    for ctx in ctxs:
        ctx.close()


def test_cfg2_member_matches_dedup_oracle():
    """A cfg2-shaped member (shrunk evaluation side) beside a small one, against the oracle's de-duplicated
    corrected mode as tests/test_gpu_fullparity.py checks a single context."""
    import fullsize
    import pmdi_b200.capi as capi
    cfg = fullsize.make("cfg2_multiomics_fresh")
    hy = cfg["hy"]
    other = problem(**SAME, seed=3)
    big, small = capi.Context(cfg["data"], cfg["types"], cfg["N"], cfg["P"]), _ctx(other)
    grp = capi.Group([big, small, _ctx(other)])

    def run(s, order, it, lw0, debug):
        big.upload(s, order, cfg["n1"], hy["Pi"], hy["phi"], seed=77, it=it, logweight_init=lw0, debug=debug)
        for c in grp.contexts[1:]:
            c.upload(**_args(other))
        grp.run()
        for c in grp.contexts[1:]:
            c.download()
        return big.download()

    out = fullsize.compare(cfg, run)
    fullsize.assert_parity(out)
    grp.close()
    for c in grp.contexts:
        c.close()


def test_chained_group_sweeps_with_a_solo_sweep_between():
    """Five group sweeps with the allocations chained, member 0 swept alone after the second: the barrier counters
    and step tags run on across group and solo sweeps; results equal the same sequence on fresh contexts."""
    import pmdi_b200.capi as capi
    prs = [problem(**SAME, seed=3), problem(sets=[(G, 4, 0)], n=150, N=10, P=32, seed=5)]
    rng = np.random.default_rng(1)
    orders = [[rng.permutation(pr["n"]) + 1 for pr in prs] for _ in range(6)]
    ctxs = [_ctx(pr) for pr in prs]
    refs = [_ctx(pr) for pr in prs]
    s_g = [pr["s"] for pr in prs]
    s_r = list(s_g)
    with capi.Group(ctxs) as grp:
        for it in range(5):
            got = grp.sweep([_args(pr, seed=8, it=it, lw0=float(it > 0), s=s, order=orders[it][i])
                             for i, (pr, s) in enumerate(zip(prs, s_g))])
            ref = [_alone(c, _args(pr, seed=8, it=it, lw0=float(it > 0), s=s, order=orders[it][i]))
                   for i, (c, pr, s) in enumerate(zip(refs, prs, s_r))]
            for g, r in zip(got, ref):
                _assert_same(g, r)
            s_g, s_r = [g["s"] for g in got], [r["s"] for r in ref]
            if it == 1:  # member 0 alone, between two group sweeps
                a = _args(prs[0], seed=9, it=7, s=s_g[0], order=orders[5][0])
                g0, r0 = _alone(ctxs[0], a), _alone(refs[0], a)
                _assert_same(g0, r0)
                s_g[0], s_r[0] = g0["s"], r0["s"]
    for c in ctxs + refs:
        c.close()


def _chain_data():
    from pmdi_b200 import synth
    data, types, _ = synth.make_data([(G, 6, 0), (C, 5, 3)], 60, 3, 2)
    return data, types


def _csv(path, K):
    from pmdi_b200.pmdi import n_hyper_columns
    rows = [line.split(",") for line in open(path).read().splitlines()]
    ll = n_hyper_columns(K) - 1
    return [r[:ll] + r[ll + 1:] for r in rows]


@pytest.mark.parametrize("feature_select", [False, True])
def test_pmdi_chains_equal_single_runs(tmp_path, feature_select):
    from pmdi_b200.pmdi import pmdi
    data, types = _chain_data()
    kw = dict(N=5, particles=32, rho=0.25, iter=4)
    outs = [str(tmp_path / f"chain{c}.csv") for c in range(3)]
    fsel = [str(tmp_path / f"fs{c}.csv") for c in range(3)] if feature_select else None
    stats = pmdi(data, types, outputFile=outs, featureSelect=fsel, seed=40, chains=3, **kw)
    assert len(stats) == 3 and all(s["iterations"] == 4 for s in stats)
    for c in range(3):
        one, fs_one = str(tmp_path / f"one{c}.csv"), (str(tmp_path / f"fs_one{c}.csv") if feature_select else None)
        pmdi(data, types, outputFile=one, featureSelect=fs_one, seed=40 + c, **kw)
        assert _csv(outs[c], 2) == _csv(one, 2)
        if feature_select:
            assert open(fsel[c]).read() == open(fs_one).read()


def test_refusals():
    import pmdi_b200.capi as capi
    from pmdi_b200 import synth
    import user_types
    pr = problem(**SAME, seed=3)
    a, b, c = _ctx(pr), _ctx(pr), _ctx(pr)
    with capi.Group([a, b]):
        with pytest.raises(capi.PmdiError, match="already in a group"):
            capi.Group([b, c])
    with pytest.raises(capi.PmdiError, match="same context"):
        capi.Group([a, a])
    data5, types5, _ = synth.make_data([(G, 3, 0)] * 5, 40, 3, 1)
    with capi.Context(data5, types5, 4, 8) as k5:
        with pytest.raises(capi.PmdiError, match="spec engine"):
            capi.Group([a, k5])
    tag = capi.register_cluster_type("ChainsGaussian", user_types.USER_GAUSSIAN, "MyGaussian")
    with capi.Context([pr["data"][0]], [tag], pr["N"], pr["P"]) as u:
        with pytest.raises(capi.PmdiError, match="user-defined"):
            capi.Group([a, u])
    os.environ["PMDI_ENGINE"] = "pool"
    try:
        with pytest.raises(capi.PmdiError, match="pool engine"):
            capi.Group([a, b])
    finally:
        os.environ.pop("PMDI_ENGINE")
    with capi.Context(pr["data"], pr["types"], pr["N"], pr["P"], rank=0, n_ranks=2) as sh:
        with pytest.raises(capi.PmdiError, match="sharded"):
            capi.Group([a, sh])
    # 16 members with 2048 particles and N = 40: a share of 9 SMs leaves one proposal CTA, whose tables do not fit
    big = problem(sets=[(G, 4, 0)], n=100, N=40, P=2048, seed=1)
    many = [_ctx(big) for _ in range(16)]
    with pytest.raises(capi.PmdiError, match="member 0"):
        capi.Group(many)
    for m in many:
        m.close()
    # nothing changed: a refused member still sweeps alone as a fresh context does
    ref = _alone(c, _args(pr))
    _assert_same(_alone(a, _args(pr)), ref)
    _assert_same(_alone(b, _args(pr)), ref)
    for x in (a, b, c):
        x.close()


def test_destroying_a_member_detaches_it():
    """pmdi_ctx_destroy of a member detaches it; the group refuses to run, the other members sweep alone."""
    import pmdi_b200.capi as capi
    pr = problem(**SAME, seed=3)
    a, b = _ctx(pr), _ctx(pr)
    grp = capi.Group([a, b])
    grp.sweep([_args(pr), _args(pr)])
    a.close()
    b.upload(**_args(pr))
    with pytest.raises(capi.PmdiError, match="destroyed"):
        grp.run()
    grp.close()
    with _ctx(pr) as fresh:
        _assert_same(_alone(b, _args(pr)), _alone(fresh, _args(pr)))
    b.close()

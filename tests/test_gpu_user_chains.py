"""Groups with user-defined cluster types (pmdi_ctx_set_engine, pmdi_group_* with the run-time compiled group kernels,
pmdi(chains=C) with UserCluster types).  A member's results must be those of the member swept alone - bit for bit -
on its share of the SMs and on a fresh spec context with the whole GPU; the user restatements of the built-in types
must reproduce the built-ins inside a group as they do alone."""
import numpy as np
import pytest

import multi_user_types as mu
from helpers import C, G, NB, problem, tapes_for

pytestmark = pytest.mark.gpu

EXACT = ["s", "p_star", "label_counts", "pair_agree", "contingency", "rows_evaluated", "rows_added",
         "n_resamples", "cluster_n"]
# [user Gaussian, user NegBinom, Categorical]: the shape of tests/test_gpu_multi_user_types.py
SHAPE = dict(sets=[(G, 130, 0), (NB, 70, 0), (C, 40, 3)], n=110, N=9, P=48)


def _user_ctx(pr, tags, engine="spec"):
    from pmdi_b200 import capi
    tg, tn = tags
    return capi.Context(pr["data"], [tg, tn, pr["types"][2]], pr["N"], pr["P"], engine=engine)


def _builtin_ctx(pr):
    from pmdi_b200 import capi
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
    """One problem at three seeds, one member with tapes that force resampling, one settled member."""
    same = problem(**SHAPE, seed=3)
    heavy = problem(**SHAPE, seed=4)
    settled = problem(sets=[(G, 4, 0), (NB, 3, 0), (C, 3, 2)], n=150, N=10, P=32, seed=5)
    return [(same, _args(same, seed=s)) for s in (11, 12, 13)] + \
        [(heavy, _args(heavy, tapes=tapes_for(heavy))), (settled, _args(settled, seed=2, lw0=0.0))]


def test_group_equals_alone():
    from pmdi_b200 import capi
    tags = mu.register(capi)
    members = _members()
    ctxs = [_user_ctx(pr, tags) for pr, _ in members]
    with capi.Group(ctxs) as grp:
        got = grp.sweep([a for _, a in members])
        assert got[3]["n_resamples"] > 0  # the resampling path ran inside the group
        for ctx, (pr, a), g in zip(ctxs, members, got):
            assert g["engine"] == "spec" and g["sweep_kernel_ms"] > 0
            _assert_same(g, _alone(ctx, a))            # alone on the member's share of the SMs
            with _user_ctx(pr, tags) as fresh:         # a fresh spec context on the whole GPU
                _assert_same(g, _alone(fresh, a))
    for ctx in ctxs:
        ctx.close()


def test_user_members_reproduce_the_builtins():
    """The group's user members against built-in contexts swept alone with debug capture (the built-ins are tied to
    the oracle by tests/test_gpu_chains.py and tests/test_gpu_parity.py)."""
    from pmdi_b200 import capi
    tags = mu.register(capi)
    prs = [problem(**SHAPE, seed=6 + i) for i in range(3)]
    args = [_args(pr, seed=3 + i, it=2, tapes=tapes_for(pr, seed=5 + i), debug=True) for i, pr in enumerate(prs)]
    ctxs = [_user_ctx(pr, tags) for pr in prs]
    with capi.Group(ctxs) as grp:
        got = grp.sweep(args)
    for pr, a, g in zip(prs, args, got):
        with _builtin_ctx(pr) as b:
            ref = b.sweep(**a)
        assert ref["engine"] == "spec" and ref["n_resamples"] > 0
        for k in ("alloc", "anc", "s", "cluster_n"):
            np.testing.assert_array_equal(g[k], ref[k], err_msg=k)
        assert g["p_star"] == ref["p_star"] and g["n_resamples"] == ref["n_resamples"]
        np.testing.assert_allclose(g["lp"], ref["lp"], rtol=1e-9, atol=1e-9)
        np.testing.assert_allclose(g["lw"], ref["lw"], rtol=1e-9, atol=1e-9)
    for ctx in ctxs:
        ctx.close()


def test_builtin_members_ride_in_a_user_group_with_two_structs_named_cluster():
    from pmdi_b200 import capi
    tags = mu.register(capi, named_cluster=True)
    pu = problem(**SHAPE, seed=7)
    pb = problem(sets=[(G, 130, 0), (C, 65, 3), (NB, 100, 0)], n=120, N=12, P=64, seed=3)
    pg = problem(sets=[(G, 4, 0)], n=150, N=10, P=32, seed=5)
    members = [(_user_ctx(pu, tags), _args(pu, seed=4, tapes=tapes_for(pu))), (_builtin_ctx(pb), _args(pb)),
               (_user_ctx(pu, tags), _args(pu, seed=5)), (_builtin_ctx(pg), _args(pg, seed=2, lw0=0.0))]
    fresh = [lambda: _user_ctx(pu, tags), lambda: _builtin_ctx(pb), lambda: _user_ctx(pu, tags),
             lambda: _builtin_ctx(pg)]
    with capi.Group([c for c, _ in members]) as grp:
        got = grp.sweep([a for _, a in members])
    assert got[0]["n_resamples"] > 0
    for (ctx, a), g, make in zip(members, got, fresh):
        with make() as f:
            _assert_same(g, _alone(f, a))
        ctx.close()


def test_chained_group_sweeps_with_a_solo_sweep_between():
    """Five group sweeps with the allocations chained, member 0 swept alone after the second: results equal the same
    sequence on fresh contexts."""
    from pmdi_b200 import capi
    tags = mu.register(capi)
    prs = [problem(**SHAPE, seed=3), problem(**SHAPE, seed=8)]
    rng = np.random.default_rng(1)
    orders = [[rng.permutation(pr["n"]) + 1 for pr in prs] for _ in range(6)]
    ctxs = [_user_ctx(pr, tags) for pr in prs]
    refs = [_user_ctx(pr, tags) for pr in prs]
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


def _csv(path, K):
    from pmdi_b200.pmdi import n_hyper_columns
    rows = [line.split(",") for line in open(path).read().splitlines()]
    ll = n_hyper_columns(K) - 1
    return [r[:ll] + r[ll + 1:] for r in rows]


@pytest.mark.parametrize("feature_select", [False, True])
def test_pmdi_chains_with_user_types_equal_single_spec_runs(tmp_path, feature_select, monkeypatch):
    from pmdi_b200.pmdi import pmdi
    counts, expr, _ = mu.planted(n=60)
    types = list(mu.pmdi_types())
    kw = dict(N=5, particles=32, rho=0.25, iter=4)
    outs = [str(tmp_path / f"chain{c}.csv") for c in range(3)]
    fsel = [str(tmp_path / f"fs{c}.csv") for c in range(3)] if feature_select else None
    monkeypatch.delenv("PMDI_ENGINE", raising=False)
    stats = pmdi([counts, expr], types, outputFile=outs, featureSelect=fsel, seed=40, chains=3, **kw)
    assert len(stats) == 3 and all(s["iterations"] == 4 for s in stats)
    monkeypatch.setenv("PMDI_ENGINE", "spec")
    for c in range(3):
        one, fs_one = str(tmp_path / f"one{c}.csv"), (str(tmp_path / f"fs_one{c}.csv") if feature_select else None)
        pmdi([counts, expr], types, outputFile=one, featureSelect=fs_one, seed=40 + c, **kw)
        assert _csv(outs[c], 2) == _csv(one, 2)
        if feature_select:
            assert open(fsel[c]).read() == open(fs_one).read()


def test_refusals_and_lifecycle(monkeypatch, capfd):
    from pmdi_b200 import capi
    monkeypatch.delenv("PMDI_ENGINE", raising=False)
    tags = mu.register(capi)
    named = mu.register(capi, named_cluster=True)
    pr = problem(**SHAPE, seed=3)
    a, b = _user_ctx(pr, tags), _user_ctx(pr, tags)
    # a user member on its one-GPU default, the pool engine
    with _user_ctx(pr, tags, engine=None) as p:
        with pytest.raises(capi.PmdiError, match=r"member 1: has a user-defined .*pmdi_ctx_set_engine"):
            capi.Group([a, p])
    # another type list (here: the same types under other names and sources)
    with _user_ctx(pr, named) as o:
        with pytest.raises(capi.PmdiError, match=r"member 1: its user-defined cluster types .* differ"):
            capi.Group([a, o])
    # the engine is fixed once the context is prepared
    with _user_ctx(pr, tags) as s:
        _alone(s, _args(pr))
        assert capi.lib().pmdi_ctx_set_engine(s.h, 1) == 1
        assert "already been prepared for the spec engine" in capi.lib().pmdi_last_error().decode()
    ref = [_alone(c, _args(pr)) for c in (a, b)]  # refused members are unchanged
    # a second group with the same types loads the first one's program
    monkeypatch.setenv("PMDI_JIT_LOG", "1")
    with capi.Group([a, b]) as g1:
        g1.sweep([_args(pr), _args(pr)])
    capfd.readouterr()
    grp = capi.Group([a, b])
    err = capfd.readouterr().err
    assert "pmdi: nvrtc cache hit: 'MyGaussian', 'MyNegBinom', spec-group engine" in err, err
    assert "nvrtc compiled" not in err, err
    got = grp.sweep([_args(pr), _args(pr)])
    for g, r in zip(got, ref):
        _assert_same(g, r)
    # destroying a member detaches it: the group refuses to run, the other member sweeps alone
    a.close()
    b.upload(**_args(pr))
    with pytest.raises(capi.PmdiError, match="destroyed"):
        grp.run()
    grp.close()
    with _user_ctx(pr, tags) as fresh:
        _assert_same(_alone(b, _args(pr)), _alone(fresh, _args(pr)))
    b.close()

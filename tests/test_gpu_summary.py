"""Posterior summaries on the GPU (pmdi_summary_*, capi.PosteriorSummary): pair counts and PSMs against numpy bit for
bit, the least-squares consensus and the chains' agreement against direct numpy evaluations, and pmdi(summary=)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

LABELS = np.array([1, 2, 3, 255, 256])


def _rows(rng, rows, n, K, N=256):
    """rows x (n, K) allocations with labels 1 and 256 present and enough agreement to count."""
    a = rng.choice(LABELS, size=(rows, n, K))
    if K > 1:
        a[..., 1] = rng.integers(1, N + 1, size=(rows, n))
    return a.astype(np.int64)


def _overall(psm):
    acc = psm[0].copy()
    for p in psm[1:]:
        acc = acc + p
    return acc / len(psm)


def _ari(a, b):
    from scipy.special import comb
    ct = np.zeros((a.max() + 1, b.max() + 1))
    for i, j in zip(a, b):
        ct[i, j] += 1
    s = comb(ct, 2).sum()
    sa, sb = comb(ct.sum(1), 2).sum(), comb(ct.sum(0), 2).sum()
    e = sa * sb / comb(len(a), 2)
    return (s - e) / (0.5 * (sa + sb) - e)


def _separable(n, seed=0):
    """Planted clusters that every feature separates (as in test_gpu_pmdi.py)."""
    rng = np.random.default_rng(seed)
    z = np.arange(n) % 3
    x = rng.normal(0, 1, (n, 10)) + 6.0 * z[:, None]
    xnb = rng.poisson(np.array([1.0, 30.0, 900.0])[z][:, None] * np.ones((n, 40))).astype(np.int64)
    xc = np.where(rng.random((n, 30)) < 0.05, rng.integers(1, 4, (n, 30)), (z + 1)[:, None]).astype(np.int64)
    xc[0, :] = 3
    return [x, xnb, xc], z


def _ls_numpy(samples, pi):
    n = pi.shape[0]
    iu = np.triu_indices(n, 1)
    p = pi[iu]
    return np.array([(((s[:, None] == s[None, :])[iu]) - p) @ (((s[:, None] == s[None, :])[iu]) - p)
                     for s in samples])


@pytest.mark.parametrize("n,rows,K,chains", [(1, 1, 1, 1), (2, 3, 2, 1), (127, 5, 3, 3), (129, 257, 4, 1),
                                             (129, 257, 1, 3), (1000, 5, 2, 3), (1000, 257, 1, 1)])
def test_psm_equals_numpy_bit_for_bit(n, rows, K, chains):
    from pmdi_b200 import capi
    from pmdi_b200 import pmdi as host
    rng = np.random.default_rng(n * 7 + rows + K)
    data = [_rows(rng, rows, n, K) for _ in range(chains)]
    with capi.PosteriorSummary(K, n, 256, chains=chains) as S:
        # adds interleaved between the chains: single rows and blocks
        for r in range(0, rows, 2):
            for c in range(chains):
                S.add(c, data[c][r] if r + 1 >= rows else data[c][r:r + 2])
        assert [S.rows(c) for c in range(chains)] == [rows] * chains
        for c in range(chains):
            ref = host.posterior_similarity(data[c])
            for k in range(K):
                np.testing.assert_array_equal(S.psm(k, chain=c), ref[k])
            np.testing.assert_array_equal(S.psm(None, chain=c), _overall(ref))
        pooled = host.posterior_similarity(np.concatenate(data))
        for k in range(K):
            got = S.psm(k)
            np.testing.assert_array_equal(got, pooled[k])
            assert (np.diag(got) == 1.0).all()
            np.testing.assert_array_equal(S.psm(k, dtype=np.float32), got.astype(np.float32))
        np.testing.assert_array_equal(S.psm(), _overall(pooled))


def test_psm_within_one_ulp_of_context_psm():
    from pmdi_b200 import capi
    n, K, N, rows = 129, 2, 8, 37
    rng = np.random.default_rng(3)
    a = rng.integers(1, N + 1, size=(rows, n, K))
    ctx = capi.Context([np.zeros((n, 1))] * K, [capi.GAUSSIAN] * K, N, 4)
    old = ctx.psm(a)
    ctx.close()
    with capi.PosteriorSummary(K, n, N) as S:
        S.add(0, a)
        for k in range(K):
            np.testing.assert_array_max_ulp(S.psm(k), old[k], 1)


def _planted(rng, n, N, rows, noise=0.1):
    base = rng.integers(1, N + 1, n)
    out = np.repeat(base[None], rows, axis=0)
    flip = rng.random((rows, n)) < noise
    out[flip] = rng.integers(1, N + 1, flip.sum())
    return base, out


def test_least_squares_matches_numpy_with_a_planted_tie():
    from pmdi_b200 import capi
    n, N, K, chains, rows = 150, 5, 2, 3, 40
    rng = np.random.default_rng(11)
    base, _ = _planted(rng, n, N, 1)
    data = []
    for c in range(chains):
        d = np.stack([_planted(rng, n, N, rows, 0.15)[1] for _ in range(K)], axis=2)
        d[:, :, 0] = np.where(rng.random((rows, n)) < 0.15, rng.integers(1, N + 1, (rows, n)), base)
        data.append(d)
    # the planted tie: the base partition twice, in chain 1 row 5 and chain 2 row 2 (and nothing else is closer)
    data[1][5, :, 0] = base
    data[2][2, :, 0] = base
    with capi.PosteriorSummary(K, n, N, chains=chains) as S:
        for c in range(chains):
            S.add(c, data[c])
        allrows = np.concatenate(data)
        for k in range(K):
            part, loss, best = S.least_squares(k)
            ref = _ls_numpy(allrows[:, :, k], S.psm(k))
            np.testing.assert_allclose(loss, ref, rtol=1e-12, atol=0)
            i = int(np.argmin(loss))
            assert loss[i] == loss.min() and best == (i // rows, i % rows)
            np.testing.assert_array_equal(part, allrows[i, :, k])
            assert np.isclose(ref[i], ref.min(), rtol=1e-12)
            if k == 0:
                assert best == (1, 5) and loss[rows + 5] == loss[2 * rows + 2]
            _, loss2, best2 = S.least_squares(k)
            np.testing.assert_array_equal(loss2, loss)  # the same bits on every call
            assert best2 == best


def test_least_squares_and_counts_do_not_depend_on_how_samples_are_chunked():
    """3,300 rows cross chunk (256) and least-squares batch (3,072) boundaries; one summary gets them in one call,
    the other in pieces with read-outs in between (each read-out counts a partial chunk)."""
    from pmdi_b200 import capi
    n, N, rows = 40, 4, 3300
    rng = np.random.default_rng(5)
    a = np.stack([_planted(rng, n, N, rows, 0.3)[1]], axis=2)
    with capi.PosteriorSummary(1, n, N) as S1, capi.PosteriorSummary(1, n, N) as S2:
        S1.add(0, a)
        at = 0
        for step in (1, 3, 250, 7, 1000, 2039):
            S2.add(0, a[at:at + step])
            at += step
            S2.psm(0)
        assert at == rows
        np.testing.assert_array_equal(S1.psm(0), S2.psm(0))
        p1, l1, b1 = S1.least_squares(0)
        p2, l2, b2 = S2.least_squares(0)
        np.testing.assert_array_equal(l1, l2)
        assert b1 == b2 and (p1 == p2).all()
        np.testing.assert_allclose(l1[::97], _ls_numpy(a[::97, :, 0], S1.psm(0)), rtol=1e-12)


def test_agreement_matches_numpy_for_three_chains():
    from pmdi_b200 import capi
    from pmdi_b200 import pmdi as host
    n, K, N = 300, 2, 6
    rng = np.random.default_rng(8)
    data = [np.stack([_planted(rng, n, N, r, 0.2 + 0.1 * c)[1] for _ in range(K)], axis=2)
            for c, r in enumerate((20, 33, 7))]
    with capi.PosteriorSummary(K, n, N, chains=3) as S:
        for c in (2, 0, 1):
            S.add(c, data[c])
        mx, mean = S.agreement()
    psm = [host.posterior_similarity(d) for d in data]
    iu = np.triu_indices(n, 1)
    for p, (a, b) in enumerate([(0, 1), (0, 2), (1, 2)]):
        for k in range(K):
            d = np.abs(psm[a][k] - psm[b][k])[iu]
            assert mx[p, k] == d.max()
            np.testing.assert_allclose(mean[p, k], d.mean(), rtol=1e-12)


def test_pmdi_summary_equals_generate_psm_of_its_files(tmp_path):
    from pmdi_b200 import capi
    from pmdi_b200 import pmdi as host
    n, K, N, iters = 90, 3, 6, 24
    data, z = _separable(n)
    outs = [str(tmp_path / f"c{c}.csv") for c in range(2)]
    with capi.PosteriorSummary(K, n, N, chains=2, burnin=3, thin=2) as S:
        host.pmdi(data, [host.GaussianCluster, host.NegBinomCluster, host.CategoricalCluster], N, 32, 0.25, iters,
                  outs, thin=2, seed=4, chains=2, summary=S)
        assert [S.rows(c) for c in range(2)] == [len(range(3, 1 + iters // 2, 2))] * 2
        got = np.stack([S.psm(k) for k in range(K)] + [S.psm()])
        ref = host.generate_psm(outs, burnin=3, thin=2)
        assert ref.shape == (K + 1, n, n)
        np.testing.assert_array_equal(got, ref)
        chains, names = host.read_chains(outs, burnin=3, thin=2)
        np.testing.assert_array_equal(ref[0], host.posterior_similarity(np.concatenate(chains))[0])
        for k in range(K):
            part, _, _ = S.least_squares(k)
            assert _ari(part, z) > 0.9, k
        cons = host.consensus_partition(outs, burnin=3, thin=2)
        assert cons.shape == (n, K) and all(_ari(cons[:, k], z) > 0.9 for k in range(K))
        mx, mean = host.chain_agreement(outs, burnin=3, thin=2)
        np.testing.assert_array_equal(mx, S.agreement()[0])


def test_refusals():
    from pmdi_b200 import capi
    with pytest.raises(capi.PmdiError, match="bytes"):
        capi.PosteriorSummary(8, 65535, 256, chains=64)
    with capi.PosteriorSummary(2, 10, 5, chains=2) as S:
        good = np.ones((10, 2), dtype=np.int64)
        bad0, bad6 = good.copy(), good.copy()
        bad0[3, 1] = 0
        bad6[9, 0] = 6
        for bad in (bad0, bad6):
            with pytest.raises(capi.PmdiError, match="outside 1..5"):
                S.add(0, bad)
        assert S.rows(0) == 0
        with pytest.raises(ValueError):
            S.add(2, good)
        s = np.asfortranarray(good)
        assert capi.lib().pmdi_summary_add(S.h, 2, s.ctypes.data_as(C.c_void_p), 1) == 1
        assert capi.lib().pmdi_summary_add(S.h, -1, s.ctypes.data_as(C.c_void_p), 1) == 1
        with pytest.raises(capi.PmdiError, match="no rows"):
            S.psm(0)
        S.add(1, good)
        assert S.rows(1) == 1 and S.rows(0) == 0
        with pytest.raises(capi.PmdiError, match="no rows"):
            S.agreement()

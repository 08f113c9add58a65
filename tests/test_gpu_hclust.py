"""Hierarchical consensus clustering on the GPU (pmdi_summary_hclust, capi.PosteriorSummary.hclust,
pmdi.consensus_allocations): Z equals the exact CPU reference (tests/hclust_ref.py) bit for bit, whatever the tile
boundaries, the chains and the chunks the rows came in."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import hclust_ref  # noqa: E402

pytestmark = pytest.mark.gpu

LINKAGES = hclust_ref.LINKAGES


def _planted(rng, n, N, rows, K, noise):
    """rows x (n, K) labels around a planted partition per dataset: few labels, few rows, ties everywhere."""
    out = np.empty((rows, n, K), dtype=np.int64)
    for k in range(K):
        base = rng.integers(1, N + 1, n)
        a = np.repeat(base[None], rows, axis=0)
        flip = rng.random((rows, n)) < noise
        a[flip] = rng.integers(1, N + 1, flip.sum())
        out[..., k] = a
    return out


def _ref(S, k, linkage):
    """The reference's Z from the summary's own PSMs: counts = PSM x rows (summed over the datasets for Overall)."""
    R = sum(S.rows(c) for c in range(S.chains))
    ks = range(S.K) if k is None else [k]
    A = sum(hclust_ref.counts_from_psm(S.psm(q), R) for q in ks)
    return hclust_ref.linkage_counts(A, R * len(ks), linkage)


def _check(S, k, linkage):
    from scipy.cluster import hierarchy
    Z = S.hclust(k, linkage=linkage)
    ref, _, rescans = _ref(S, k, linkage)
    np.testing.assert_array_equal(Z, ref)  # bit for bit, heights included
    assert S.last_rescans == rescans
    assert hierarchy.is_valid_linkage(Z)
    return Z


@pytest.mark.parametrize("n", [2, 127, 128, 129, 300, 1000, 3000])
def test_z_equals_the_reference_per_dataset_and_overall(n):
    from pmdi_b200 import capi
    rng = np.random.default_rng(n)
    K = 2
    a = _planted(rng, n, 6, 9, K, 0.3)
    with capi.PosteriorSummary(K, n, 6) as S:
        S.add(0, a)
        for k in (0, 1, None):
            for linkage in LINKAGES:
                if n == 3000 and k == 1:
                    continue  # dataset 0 and Overall at the largest size keep the test short
                _check(S, k, linkage)


def test_identical_rows_give_zero_heights():
    from pmdi_b200 import capi
    n = 200
    a = np.ones((3, n, 1), dtype=np.int64)
    with capi.PosteriorSummary(1, n, 2) as S:
        S.add(0, a)
        for linkage in LINKAGES:
            Z = _check(S, 0, linkage)
            assert (Z[:, 2] == 0.0).all() and Z[-1, 3] == n


def test_rows_in_chains_and_chunks_give_the_same_z():
    """The same 300 rows as one chain, as four chains, and added in pieces across the 256-row chunk boundary; a second
    call gives the same bits; more rows and a new call match the reference on all the rows."""
    from pmdi_b200 import capi
    n, K, N = 150, 2, 5
    rng = np.random.default_rng(7)
    a = _planted(rng, n, N, 300, K, 0.4)
    with capi.PosteriorSummary(K, n, N) as S1, capi.PosteriorSummary(K, n, N, chains=4) as S4, \
            capi.PosteriorSummary(K, n, N) as Sp:
        S1.add(0, a)
        for c, part in enumerate(np.array_split(a, 4)):
            S4.add(c, part)
        at = 0
        for step in (1, 200, 60, 39):
            Sp.add(0, a[at:at + step])
            at += step
            Sp.psm(0)  # a read-out counts the partial chunk
        assert at == 300
        for k in (0, None):
            for linkage in LINKAGES:
                Z1 = _check(S1, k, linkage)
                np.testing.assert_array_equal(S4.hclust(k, linkage=linkage), Z1)
                np.testing.assert_array_equal(Sp.hclust(k, linkage=linkage), Z1)
                np.testing.assert_array_equal(S1.hclust(k, linkage=linkage), Z1)
        S1.add(0, _planted(rng, n, N, 40, K, 0.2))
        for linkage in LINKAGES:
            _check(S1, None, linkage)


def test_one_observation_and_cut_tree_against_scipy():
    from scipy.cluster import hierarchy
    from pmdi_b200 import capi
    from pmdi_b200 import pmdi as host
    with capi.PosteriorSummary(1, 1, 3) as S:
        S.add(0, np.ones((4, 1, 1), dtype=np.int64))
        Z = S.hclust(0, linkage="average")
        assert Z.shape == (0, 4)
        np.testing.assert_array_equal(host.cut_tree(Z, 1), [1])
    rng = np.random.default_rng(2)
    n = 90
    with capi.PosteriorSummary(1, n, 4) as S:
        S.add(0, _planted(rng, n, 4, 500, 1, 0.5))  # many rows: few exact ties
        for linkage in LINKAGES:
            Z = S.hclust(0, linkage=linkage)
            assert hierarchy.is_valid_linkage(Z)
            for c in range(1, n + 1):
                if c in (1, n) or Z[n - c - 1, 2] < Z[n - c, 2]:
                    np.testing.assert_array_equal(host.cut_tree(Z, c),
                                                  hierarchy.cut_tree(Z, n_clusters=c).ravel() + 1)


def test_refusals():
    from pmdi_b200 import capi
    with capi.PosteriorSummary(1, 10, 3) as S:
        with pytest.raises(capi.PmdiError, match="no rows"):
            S.hclust(0, linkage="single")
        S.add(0, np.ones((1, 10, 1), dtype=np.int64))
        assert capi.lib().pmdi_summary_hclust(S.h, 0, 3, None, None) == 1
        assert capi.lib().pmdi_summary_hclust(S.h, 1, 0, None, None) == 1
        assert capi.lib().pmdi_summary_hclust(S.h, 0, 0, None, None) == 1  # Z_out NULL


def test_consensus_allocations_equals_the_reference_cut(tmp_path):
    from pmdi_b200 import pmdi as host
    n, K, N, iters = 90, 2, 6, 20
    rng = np.random.default_rng(3)
    z = np.arange(n) % 3
    data = [rng.normal(0, 1, (n, 4)) + 6.0 * z[:, None],
            np.where(rng.random((n, 20)) < 0.05, rng.integers(1, 4, (n, 20)), (z + 1)[:, None]).astype(np.int64)]
    outs = [str(tmp_path / f"c{c}.csv") for c in range(2)]
    host.pmdi(data, [host.GaussianCluster, host.CategoricalCluster], N, 32, 0.25, iters, outs, seed=5, chains=2)
    chains, _ = host.read_chains(outs, burnin=2)
    allrows = np.concatenate(chains)
    R = allrows.shape[0]
    psm = host.posterior_similarity(allrows)
    for dataset in (0, None):
        ks = range(K) if dataset is None else [dataset]
        A = sum(hclust_ref.counts_from_psm(psm[q], R) for q in ks)
        for linkage in LINKAGES:
            Z, _, _ = hclust_ref.linkage_counts(A, R * len(ks), linkage)
            for c in (1, 3, 7):
                got = host.consensus_allocations(outs, c, linkage, dataset=dataset, burnin=2)
                np.testing.assert_array_equal(got, host.cut_tree(Z, c))

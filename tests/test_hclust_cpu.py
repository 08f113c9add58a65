"""Hierarchical consensus clustering without a GPU: the exact CPU reference (tests/hclust_ref.py) against scipy's
linkage on tie-free matrices, the tie rule on a hand-built matrix, cut_tree against scipy's, and argument errors
refused before any device is touched."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
from scipy.cluster import hierarchy
from scipy.spatial.distance import squareform

import pmdi_b200  # noqa: F401
from pmdi_b200 import capi
from pmdi_b200 import pmdi as host

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import hclust_ref  # noqa: E402


def _tie_free(n, seed):
    """Symmetric matrix of distinct random 31-bit similarities, U = 2^31."""
    rng = np.random.default_rng(seed)
    iu = np.triu_indices(n, 1)
    A = np.zeros((n, n), dtype=np.int64)
    A[iu] = rng.choice(2 ** 31, size=len(iu[0]), replace=False)
    return A + A.T, 2 ** 31


@pytest.mark.parametrize("linkage", hclust_ref.LINKAGES)
@pytest.mark.parametrize("n", [2, 3, 50, 200])
def test_reference_equals_scipy_without_ties(n, linkage):
    A, U = _tie_free(n, n)
    Z, _, _ = hclust_ref.linkage_counts(A, U, linkage)
    D = 1.0 - A / U
    np.fill_diagonal(D, 0.0)
    ref = hierarchy.linkage(squareform(D, checks=False), method=linkage)
    np.testing.assert_array_equal(Z[:, [0, 1, 3]], ref[:, [0, 1, 3]])
    np.testing.assert_allclose(Z[:, 2], ref[:, 2], rtol=0, atol=1e-12)
    assert hierarchy.is_valid_linkage(Z)
    for c in sorted({1, 2, 3, n // 2, n - 1, n} & set(range(1, n + 1))):
        got = host.cut_tree(Z, c)
        np.testing.assert_array_equal(got, hierarchy.cut_tree(ref, n_clusters=c).ravel() + 1)
        assert got.min() == 1 and got.max() == c


# Six observations, U = 4: {0, 3} and {1, 2, 4} are always together, 5 is alone.  Pairs of equal similarity
# everywhere: the rule picks the smallest (smaller rep, larger rep) at each step.
TIES = np.array([[0, 2, 2, 4, 2, 0],
                 [2, 0, 4, 2, 4, 1],
                 [2, 4, 0, 2, 4, 1],
                 [4, 2, 2, 0, 2, 0],
                 [2, 4, 4, 2, 0, 1],
                 [0, 1, 1, 0, 1, 0]])
TIES_Z = {
    # merges at 1.0: (0,3), (1,2), (1,4) -> ids 6, 7, 8; then {0,3}-{1,2,4} at 2 -> 9; then 5 at 1 (single) ...
    "single": [[0, 3, 0.0, 2], [1, 2, 0.0, 2], [4, 7, 0.0, 3], [6, 8, 0.5, 5], [5, 9, 0.75, 6]],
    "complete": [[0, 3, 0.0, 2], [1, 2, 0.0, 2], [4, 7, 0.0, 3], [6, 8, 0.5, 5], [5, 9, 1.0, 6]],
    "average": [[0, 3, 0.0, 2], [1, 2, 0.0, 2], [4, 7, 0.0, 3], [6, 8, 0.5, 5], [5, 9, 17 / 20, 6]],
}


@pytest.mark.parametrize("linkage", hclust_ref.LINKAGES)
def test_tie_rule_on_a_hand_built_matrix(linkage):
    Z, merges, _ = hclust_ref.linkage_counts(TIES, 4, linkage)
    np.testing.assert_array_equal(Z, np.array(TIES_Z[linkage]))
    assert [m[:2] for m in merges] == [(0, 3), (1, 2), (1, 4), (0, 1), (0, 5)]
    assert hierarchy.is_valid_linkage(Z)
    np.testing.assert_array_equal(host.cut_tree(Z, 3), [1, 2, 2, 1, 2, 3])


@pytest.mark.parametrize("linkage", hclust_ref.LINKAGES)
def test_reference_with_ties_is_valid_and_single_shortcut_is_generic(linkage):
    rng = np.random.default_rng(4)
    n, U = 120, 6
    z = rng.integers(0, 4, n)
    A = np.where(z[:, None] == z[None, :], U, rng.integers(0, 3, (n, n)))
    A = np.triu(A, 1)
    A = A + A.T
    Z, merges, _ = hclust_ref.linkage_counts(A, U, linkage)
    Zg, merges_g, _ = hclust_ref.linkage_counts(A, U, linkage, generic=True)
    np.testing.assert_array_equal(Z, Zg)
    assert merges == merges_g
    assert hierarchy.is_valid_linkage(Z) and (np.diff(Z[:, 2]) >= 0).all()
    _check_cut(Z)


def _check_cut(Z):
    """cut_tree gives c clusters numbered by first appearance, and equals scipy's wherever the cut falls between two
    different heights (scipy orders merges of equal height its own way, not by their row in Z)."""
    n = Z.shape[0] + 1
    for c in range(1, n + 1):
        got = host.cut_tree(Z, c)
        _, first = np.unique(got, return_index=True)
        assert got.max() == c and (np.diff(first) > 0).all()
        if c in (1, n) or Z[n - c - 1, 2] < Z[n - c, 2]:
            np.testing.assert_array_equal(got, hierarchy.cut_tree(Z, n_clusters=c).ravel() + 1)


def test_cut_tree_of_one_observation_and_refusals():
    np.testing.assert_array_equal(host.cut_tree(np.empty((0, 4)), 1), [1])
    Z, _, _ = hclust_ref.linkage_counts(*_tie_free(5, 1), "average")
    for bad in (0, 6):
        with pytest.raises(ValueError, match="n_clusters"):
            host.cut_tree(Z, bad)
    with pytest.raises(ValueError):
        host.cut_tree(Z[:, :3], 2)


def test_hclust_argument_errors_come_before_the_device(tmp_path):
    S = object.__new__(capi.PosteriorSummary)  # no device summary behind it
    S.K, S.n, S.h = 2, 10, None
    for kw in (dict(linkage="ward"), dict(linkage="centroid"), dict(k=2, linkage="single"),
               dict(k=-1, linkage="average")):
        with pytest.raises(ValueError):
            S.hclust(**kw)
    with pytest.raises(TypeError):
        S.hclust(0)  # linkage has no default
    Z = np.empty((9, 4))
    r = C.c_int64(0)
    L = capi.lib()
    assert L.pmdi_summary_hclust(None, 0, 0, Z.ctypes.data_as(C.c_void_p), C.byref(r)) == 1
    assert b"NULL summary" in L.pmdi_last_error()
    # the CSV path: refused before the summary is created
    p = str(tmp_path / "c.csv")
    with open(p, "w") as f:
        f.write(host.csv_header(2, 4, ["a", "b"]) + "\n")
        f.write(host.csv_row(np.ones(2), np.zeros(1), 0.0, np.ones((4, 2), dtype=np.int64)) + "\n")
    for kw in (dict(n_clusters=2, linkage="median"), dict(n_clusters=0, linkage="single"),
               dict(n_clusters=5, linkage="single"), dict(n_clusters=2, linkage="single", dataset=2)):
        with pytest.raises(ValueError):
            host.consensus_allocations(p, **kw)


def test_library_exports_hclust():
    capi.build()
    assert "pmdi_summary_hclust" in capi.EXPORTS and hasattr(capi.lib(), "pmdi_summary_hclust")
    assert capi.LINKAGES == {"single": 0, "complete": 1, "average": 2}

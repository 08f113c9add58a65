"""Exact CPU reference of the summary's hierarchical clustering (pmdi_summary_hclust, DESIGN.md §16): test
infrastructure, never on the product path.

The generic agglomerative algorithm on an integer similarity matrix A (A_ij = pooled pair count, dissimilarity
1 - A_ij / U).  A cluster pair's similarity is s / p: s = max (single), min (complete) or sum (average) of A_ij over
its pairs, p = 1 or |X| |Y| (average).  Each merge takes the largest s / p, compared exactly; equal values go to the
lexicographically smallest (smaller representative, larger representative), a cluster's representative being its
smallest observation index.  Every active row keeps a cache of its best partner (the smallest column among equals),
as the device does; rows are scanned vectorised.  Products are numpy int64 where they fit, Python ints otherwise.
"""
import numpy as np

LINKAGES = ("single", "complete", "average")


def _exact_best(s, p, tie, dt):
    """Index of the largest s / p (1-D, exact), the smallest `tie` among equals; -1 when s is empty."""
    if s.size == 0:
        return -1
    c = int(np.argmax(s.astype(np.float64) / p.astype(np.float64)))
    while True:  # the float argmax is a start; move to any entry that is exactly larger
        d = s * p[c] - s[c] * p
        up = np.flatnonzero(d > 0)
        if up.size == 0:
            break
        c = int(up[np.argmax((s[up].astype(np.float64) / p[up].astype(np.float64)))])
    eq = np.flatnonzero(d == 0)
    return int(eq[np.argmin(tie[eq])])


class _State:
    def __init__(self, A, U, linkage):
        self.n = n = A.shape[0]
        self.avg = linkage == "average"
        self.linkage = linkage
        q = (n // 2 + 1) ** 2  # bounds |X| |Y|
        self.dt = np.int64 if (q * U) * q < 2 ** 62 else object
        self.W = np.array(A, dtype=np.int64).astype(self.dt)
        self.size = np.ones(n, dtype=np.int64).astype(self.dt)
        self.active = np.ones(n, dtype=bool)
        self.cs = np.zeros(n, dtype=self.dt)
        self.cp = np.ones(n, dtype=self.dt)
        self.cj = np.full(n, -1, dtype=np.int64)

    def p_of(self, i, cols):
        return self.size[i] * self.size[cols] if self.avg else np.ones(len(cols), dtype=self.dt)

    def rescan(self, rows):
        cols = np.flatnonzero(self.active)
        for i in rows:
            c = cols[cols != i]
            j = _exact_best(self.W[i, c], self.p_of(i, c), c, self.dt)
            if j < 0:
                self.cj[i] = -1
            else:
                self.cs[i], self.cp[i], self.cj[i] = self.W[i, c[j]], self.p_of(i, c[j:j + 1])[0], c[j]

    def rescan_batch(self, rows):
        """rescan() for many rows at once (single / complete: p = 1 and argmax gives the smallest column)."""
        if self.avg or self.dt is object or len(rows) < 8:
            return self.rescan(rows)
        cols = np.flatnonzero(self.active)
        S = self.W[np.ix_(rows, cols)].copy()
        S[cols[None, :] == np.asarray(rows)[:, None]] = -1
        j = np.argmax(S, axis=1)
        v = S[np.arange(len(rows)), j]
        self.cs[rows] = np.where(v < 0, 0, v)
        self.cp[rows] = 1
        self.cj[rows] = np.where(v < 0, -1, cols[j])


def linkage_counts(A, U, linkage, generic=False):
    """(Z, merges, rescans) of the exact clustering of the symmetric integer matrix A (diagonal ignored) with
    dissimilarity 1 - A / U.  Z is scipy's linkage matrix; merges lists (a, b, s, p, size) by representative; rescans
    counts rows scanned again because their cached partner was a or b (the merged row itself not included).

    Single linkage skips those rescans unless `generic`, as the device does: the row's new entry in column a is then
    max(W[i, a], W[i, b]), its maximum, and a its smallest column holding it (the cache was the smallest such column,
    and a < b)."""
    if linkage not in LINKAGES:
        raise ValueError(linkage)
    A = np.asarray(A)
    n = A.shape[0]
    if n == 1:
        return np.empty((0, 4)), [], 0
    st = _State(A, U, linkage)
    st.rescan_batch(np.arange(n))
    ids = np.arange(n)
    Z = np.empty((n - 1, 4))
    merges, rescans = [], 0
    for m in range(n - 1):
        rows = np.flatnonzero(st.active & (st.cj >= 0))
        lo, hi = np.minimum(rows, st.cj[rows]), np.maximum(rows, st.cj[rows])
        r = _exact_best(st.cs[rows], st.cp[rows], lo * n + hi, st.dt)
        a, b = int(lo[r]), int(hi[r])
        s, p = int(st.cs[rows[r]]), int(st.cp[rows[r]])
        if linkage == "single":
            new = np.maximum(st.W[a], st.W[b])
        elif linkage == "complete":
            new = np.minimum(st.W[a], st.W[b])
        else:
            new = st.W[a] + st.W[b]
        st.W[a] = new
        st.W[:, a] = new
        st.size[a] = st.size[a] + st.size[b]
        st.active[b] = False
        others = np.flatnonzero(st.active)
        others = others[others != a]
        hit = (st.cj[others] == a) | (st.cj[others] == b)
        redo, keep = others[hit], others[~hit]
        if linkage == "single" and not generic:
            st.cs[redo], st.cj[redo] = st.W[redo, a], a
            redo = redo[:0]
        if keep.size:
            v, pv = st.W[keep, a], st.p_of(a, keep)
            d = v * st.cp[keep] - st.cs[keep] * pv
            up = keep[(d > 0) | ((d == 0) & (a < st.cj[keep]))]
            st.cs[up], st.cp[up], st.cj[up] = st.W[up, a], st.p_of(a, up), a
        rescans += len(redo)
        st.rescan_batch(np.concatenate([redo, [a]]).astype(np.int64))
        size = int(st.size[a])
        merges.append((a, b, s, p, size))
        pu = p * U
        u, v = int(ids[a]), int(ids[b])
        Z[m] = (min(u, v), max(u, v), float(pu - s) / float(pu), size)
        ids[a] = n + m
    return Z, merges, rescans


def counts_from_psm(psm, rows):
    """Integer numerators A = psm * rows (exact: every PSM entry is count / rows)."""
    A = np.rint(np.asarray(psm) * rows).astype(np.int64)
    np.fill_diagonal(A, 0)
    return A

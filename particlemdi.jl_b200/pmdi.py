"""Host side of ``pmdi()`` above the C-ABI: same entry point, asserts and CSV layout as the
reference (src/pmdi.jl:36-390); the allocation sweep (:188-350, :373) and feature selection
(:120-128, :354-370) run on the GPU through ``libpmdi_cuda.so``; the hyper-parameter updates
(src/update_hypers.jl), ``align_labels!`` (src/misc.jl:61-96) and the CSV writer stay on the host,
as the north-star prescribes.

The reference is Julia; Julia is not installed here, so this mirror is Python (DESIGN.md §0) and
none of it has been compared with a Julia run.  Deviations from the literal reference, all
switchable:

* ``stale_gamma_table`` (default False).  The reference builds its table of log gamma over the
  N^K label combinations once, before the loop (src/pmdi.jl:81-84), and never refreshes it, so
  ``update_gamma!``, ``update_Phi!`` and ``update_Z`` (:178-185) keep using the INITIAL gamma.
  Here the table follows gamma unless this flag is set.
* ``sstar_compat`` (default False).  ``pmdi()`` does not permute the stored trajectories on
  resampling (src/pmdi.jl:321-324, SURVEY F5); the tested twin ``__pmdi`` does (src/__pmdi.jl:285).
* Random numbers: numpy ``Generator(seed)`` on the host, Philox addressed by ``(seed, iteration)``
  on the device - not Julia's global RNG.

There is no CPU fallback: without the CUDA library or a device this raises.
"""
from __future__ import annotations

import math
import os
import time

import numpy as np
from scipy import special, stats

from . import capi

GAUSSIAN, CATEGORICAL, NEGBINOM = capi.GAUSSIAN, capi.CATEGORICAL, capi.NEGBINOM
EPS = float(np.finfo(np.float64).eps)
MAX_TABLE_ROWS = 50_000_000  # N^K rows of the hyper-parameter tables (SURVEY F6)


class GaussianCluster:      # names of the reference's cluster types (src/ParticleMDI.jl:31-36)
    tag = GAUSSIAN


class CategoricalCluster:
    tag = CATEGORICAL


class NegBinomCluster:
    tag = NEGBINOM


class UserCluster:
    """A user-defined cluster type (the reference's plugin contract, README.md:48-88): CUDA source of a struct with
    init / logprob / add / logmarginal (include/pmdi_cuda.h, pmdi_register_cluster_type).  ``integer_data``: the type
    is bound to Int64 data (counts, levels).

    Each dataset of a run may have a type of its own: ``pmdi([X_counts, X_expr], [MyPoisson, MyGaussian], ...)``.
    The run compiles its user types into one program when it starts (about 10-20 s of CPU; cached for the rest of
    the process, so a second run with the same types starts without compiling).  Each source lives in a namespace
    of its own, so two types may both name their struct ``Cluster``.  One GPU runs the pool engine unless
    ``PMDI_ENGINE=spec`` (``chains > 1`` runs the spec engine); ``distributed=True`` shards the particles as for the built-in types.  The type is
    registered in every process that reads ``tag`` (a rank started by torch.multiprocessing included), so the
    object can be handed to the ranks of a distributed run as it is."""

    def __init__(self, name, cuda_src, struct_name=None, integer_data=False):
        self.name, self.cuda_src = name, cuda_src
        self.struct_name = struct_name or name
        self.elem_kind = capi.I64 if integer_data else capi.F64
        _ = self.tag  # registers now: a bad elem_kind or a missing library is reported here

    @property
    def tag(self):
        """The type tag in this process (registering the same name and source again keeps it)."""
        return capi.register_cluster_type(self.name, self.cuda_src, self.struct_name, self.elem_kind)


def _tag(t):
    if isinstance(t, (int, np.integer)):
        return int(t)
    if hasattr(t, "tag"):
        return int(t.tag)
    raise TypeError(f"unknown cluster type {t!r}: only the three built-in types have device code")


def phi_lab(K):
    """calculate_Phi_lab (src/misc.jl:1-13): pairs (k1 < k2), row-major, 0-based here."""
    return [(k1, k2) for k1 in range(K - 1) for k2 in range(k1 + 1, K)]


# ------------------------------------------------------------------ hyper-parameter tables
class HyperTables:
    """c_combn, Gamma_c, Phi_index of src/pmdi.jl:69-92 (N^K rows)."""

    def __init__(self, N, K):
        rows = N ** K
        if rows > MAX_TABLE_ROWS:
            raise MemoryError(
                f"the reference's hyper-parameter updates enumerate N^K = {N}^{K} = {rows:.3g} label "
                "combinations (src/pmdi.jl:69-92); that is not feasible (SURVEY.md F6)")
        self.N, self.K = N, K
        idx = np.arange(rows)
        # c_combn[:, K-k+1] = div(0:N^K-1, N^(K-k)) % N + 1 for k = 1..K (src/pmdi.jl:70-72):
        # column j (0-based) cycles with period N^(j+1)
        self.combn = np.stack([(idx // N ** j) % N for j in range(K)], axis=1)  # 0-based labels
        pairs = phi_lab(K)
        self.phi_index = (np.stack([self.combn[:, a] == self.combn[:, b] for a, b in pairs], axis=1)
                          if K > 1 else np.ones((rows, 1), dtype=bool))
        self.log_gamma_sum = None
        # rows of every (dataset, label), ascending: what `col == n` selects (update_hypers.jl:75-78)
        self.rows_of = [[np.flatnonzero(self.combn[:, k] == n) for n in range(N)] for k in range(K)]
        self.rows_pair = [np.flatnonzero(self.phi_index[:, i]) for i in range(self.phi_index.shape[1])]

    def refresh(self, gamma):
        """sum(Gamma_c, dims=2): sum_k log gamma[c_k, k] per combination."""
        lg = np.log(gamma)
        self.log_gamma_sum = sum(lg[self.combn[:, k], k] for k in range(self.K))

    def norm_terms(self, phi):
        """exp(Phi_index * log(1+Phi) + sum Gamma) per combination (update_hypers.jl:32,75-78,101-104)."""
        if self.K > 1:
            t = self.phi_index @ np.log(np.asarray(phi) + 1.0) + self.log_gamma_sum
        else:
            # K == 1: Phi = zeros(1) (src/pmdi.jl:61) and Phi_index is all ones -> adds log(1) = 0
            t = self.log_gamma_sum.copy()
        return np.exp(t)


class FactorisedZ:
    """The sums the hyper-parameter updates take over the N^K label combinations
    (src/pmdi.jl:69-92, src/update_hypers.jl:29-39, 75-90, 101-125) WITHOUT the N^K tables.

    The summand is  prod_k gamma[c_k, k] * prod_{a<b} (1 + phi_ab)^[c_a == c_b].  Expanding
    prod (1 + phi_ab [c_a == c_b]) over subsets of pairs groups the datasets into the connected
    components of a graph; within a component all labels are equal, so

        Z = sum over set partitions {C_1..C_m} of the datasets of  prod_i conn(C_i) * s(C_i)

    with s(C) = sum_l prod_{k in C} gamma[l, k] and conn(C) = sum over CONNECTED graphs on C of
    prod phi_e, which follows from all(C) = prod_{e in C} (1 + phi_e) by the usual recursion.  All of
    it is a DP over the 2^K subsets of datasets: O(3^K + K 2^K N) instead of O(K N^K)
    (K = 6, N = 30: 7e8 table rows in the reference, a few thousand operations here)."""

    def __init__(self, N, K):
        self.N, self.K = N, K
        self.full = (1 << K) - 1
        self.pairs = phi_lab(K)
        self.members = [[k for k in range(K) if S >> k & 1] for S in range(1 << K)]
        # proper sub-subsets containing the lowest member, per subset
        self.subs = []
        for S in range(1 << K):
            if S == 0:
                self.subs.append([])
                continue
            low = S & -S
            rest = S ^ low
            out, T = [], rest
            while True:  # all subsets T of rest -> component low | T
                out.append(low | T)
                if T == 0:
                    break
                T = (T - 1) & rest
            self.subs.append(out)

    def _conn(self, phi):
        K = self.K
        allp = np.ones(1 << K)
        for S in range(1 << K):
            m = self.members[S]
            v = 1.0
            for i, (a, b) in enumerate(self.pairs):
                if (S >> a & 1) and (S >> b & 1):
                    v *= 1.0 + phi[i]
            allp[S] = v
        conn = np.zeros(1 << K)
        for S in range(1, 1 << K):
            acc = allp[S]
            for C in self.subs[S]:
                if C != S:
                    acc -= conn[C] * allp[S ^ C]
            conn[S] = acc
        return conn

    def _prods(self, gamma):
        """P_S[l] = prod_{k in S} gamma[l, k] for every subset S (P_0 = 1)."""
        K, N = self.K, self.N
        P = np.ones((1 << K, N))
        for S in range(1, 1 << K):
            low = (S & -S).bit_length() - 1
            P[S] = P[S & (S - 1)] * gamma[:, low]
        return P

    def _F(self, g):
        """F(S) = sum over set partitions of S of prod g(C)."""
        F = np.zeros(1 << self.K)
        F[0] = 1.0
        for S in range(1, 1 << self.K):
            F[S] = sum(g[C] * F[S ^ C] for C in self.subs[S])
        return F

    def Z(self, gamma, phi):
        P = self._prods(gamma)
        g = self._conn(phi) * P.sum(axis=1)
        return float(self._F(g)[self.full])

    def A(self, gamma, phi, k):
        """A_k[n] = sum over the combinations with c_k = n of the summand, divided by gamma[n, k]
        (what update_gamma! needs: beta_star = 1 + v * A_k[n], src/update_hypers.jl:75-81)."""
        P = self._prods(gamma)
        conn = self._conn(phi)
        F = self._F(conn * P.sum(axis=1))
        out = np.zeros(self.N)
        bit = 1 << k
        for C in range(1, 1 << self.K):
            if C & bit:
                out += conn[C] * P[C ^ bit] * F[self.full ^ C]
        return out

    def Q(self, gamma, phi, i):
        """Q_ab = sum over the combinations with c_a == c_b of the summand, divided by (1 + phi_ab)
        (update_Phi!: beta_star = 5 + v * Q_ab, src/update_hypers.jl:101-107).  Z is linear in phi_ab."""
        p1, p0 = np.array(phi, dtype=float), np.array(phi, dtype=float)
        p1[i], p0[i] = 1.0, 0.0
        return self.Z(gamma, p1) - self.Z(gamma, p0)


def update_Z(phi, tables, gamma=None):
    """update_Z (src/update_hypers.jl:29-39)."""
    if isinstance(tables, FactorisedZ):
        return tables.Z(gamma, phi)
    return float(tables.norm_terms(phi).sum())


def update_v(n_obs, Z, rng):
    """update_v (src/update_hypers.jl:1-3): Gamma(n_obs, 1/Z)."""
    return float(rng.gamma(n_obs, 1.0 / Z))


def _gamma_logpdf(x, a, scale):
    """scipy.stats.gamma.logpdf(x, a=a, scale=scale) for x > 0, spelled out (same operations in the same order,
    same bits; the generic rv_continuous wrapper costs ~100 us a call)."""
    y = x / scale
    return (special.xlogy(a - 1.0, y) - y - special.gammaln(a)) - math.log(scale)


def _binom_logpmf(j, n, p):
    """scipy.stats.binom.logpmf(j, n, p) for integer 0 <= j <= n, spelled out (same operations, same bits)."""
    combiln = special.gammaln(n + 1) - (special.gammaln(j + 1) + special.gammaln(n - j + 1))
    return combiln + special.xlogy(j, p) + special.xlog1py(n - j, -p)


def update_M(M, gamma, K, N, rng):
    """update_M! (src/update_hypers.jl:5-26): random-walk Metropolis on each mass parameter,
    prior Gamma(2, 0.25)."""
    for k in range(K):
        g, cur = gamma[:, k], M[k]
        ll = _gamma_logpdf(g, cur / N, 1.0).sum() + _gamma_logpdf(cur, 2.0, 0.25)
        prop = cur + rng.normal() / 10.0
        if prop <= 0.0:
            alpha = 0.0
        else:
            ll_new = _gamma_logpdf(g, prop / N, 1.0).sum() + _gamma_logpdf(prop, 2.0, 0.25)
            alpha = math.exp(min(ll_new - ll, 50.0))
        if rng.random() < alpha:
            M[k] = prop


def update_gamma(gamma, phi, v, M, s, tables, rng, counts_all=None):
    """update_gamma! (src/update_hypers.jl:64-92): Gibbs update of every component weight, with the
    normalising terms kept in step with the new value.  `counts_all` (N x K): the label counts the
    sweep reduced on the device (countn(s[:, k], n), :72); recounted from `s` when absent."""
    N, K = tables.N, tables.K
    if isinstance(tables, FactorisedZ):
        for k in range(K):
            counts = counts_all[:, k] if counts_all is not None else np.bincount(s[:, k] - 1, minlength=N)
            A = tables.A(gamma, phi, k)  # does not depend on column k: one evaluation serves all n
            for n in range(N):
                beta_star = 1.0 + v * A[n]
                gamma[n, k] = rng.gamma(M[k] / N + counts[n], 1.0 / beta_star) + EPS
        return
    norm = tables.norm_terms(phi)
    for k in range(K):
        counts = counts_all[:, k] if counts_all is not None else np.bincount(s[:, k] - 1, minlength=N)  # countn(s[:, k], n), :72
        for n in range(N):
            rows = tables.rows_of[k][n]  # ascending indices: the same elements in the same order as the mask `col == n`
            old = gamma[n, k]
            beta_star = 1.0 + v * norm[rows].sum() / old
            gamma[n, k] = rng.gamma(M[k] / N + counts[n], 1.0 / beta_star) + EPS
            norm[rows] *= gamma[n, k] / old


def update_phi(phi, v, s, tables, rng, agree_all=None, gamma=None):
    """update_Phi! (src/update_hypers.jl:95-128): each Phi is drawn from a mixture of Gammas indexed
    by 0..n_agree, prior shape 1 and rate 5.  The weight of component j is restated literally from
    :118-120, including ``- j * log(1 / beta_star)``.  `agree_all`: the per-pair agreement counts the
    sweep reduced on the device (:109-115)."""
    K = tables.K
    fact = isinstance(tables, FactorisedZ)
    norm = None if fact else tables.norm_terms(phi)
    for i, (a, b) in enumerate(phi_lab(K)):
        cur = phi[i]
        n_agree = int(agree_all[i]) if agree_all is not None else int((s[:, a] == s[:, b]).sum())
        if fact:
            beta_star = 5.0 + v * tables.Q(gamma, phi, i)
        else:
            rows = tables.rows_pair[i]
            beta_star = 5.0 + v * norm[rows].sum() / (1.0 + cur)
        j = np.arange(n_agree + 1)
        w = special.gammaln(j + 1.0) + _binom_logpmf(j, n_agree, 0.5) - j * math.log(1.0 / beta_star)
        w = np.exp(w - w.max())
        alpha_star = 1.0 + rng.choice(n_agree + 1, p=w / w.sum())
        phi[i] = rng.gamma(alpha_star, 1.0 / beta_star)
        if not fact:
            norm[rows] *= (1.0 + phi[i]) / (1.0 + cur)


def align_labels(s, phi, gamma, N, K, rng):
    """align_labels! (src/misc.jl:61-96): Metropolis label swaps within each dataset that favour
    agreement with the other datasets; gamma rows are swapped along with the labels."""
    if K == 1:
        return
    pairs = phi_lab(K)
    phi_log = np.log(np.asarray(phi) + 1.0)
    for k in range(K):
        others = [j for j in range(K) if j != k]
        rel = np.array([phi_log[i] for i, (a, b) in enumerate(pairs) if a == k or b == k])
        # pairs containing k, in pair order, line up with the other datasets in index order

        def agree(rows, lab):  # count_equals (:98-108) dotted with the relevant log(1+Phi)
            return float(((s[np.ix_(rows, others)] == lab).sum(axis=0) * rel).sum())

        for label in list(dict.fromkeys(s[:, k].tolist())):  # unique(), first-appearance order
            rows_l = np.flatnonzero(s[:, k] == label)
            if rows_l.size == 0:
                continue
            for new_label in range(1, N + 1):
                if new_label == label:
                    continue
                rows_n = np.flatnonzero(s[:, k] == new_label)
                keep = agree(rows_l, label) + agree(rows_n, new_label)
                swap = agree(rows_l, new_label) + agree(rows_n, label)
                if rng.random() < math.exp(min(swap - keep, 50.0)):
                    s[rows_l, k] = new_label
                    s[rows_n, k] = label
                    gamma[[new_label - 1, label - 1], k] = gamma[[label - 1, new_label - 1], k]
                    label = new_label
                    rows_l = np.flatnonzero(s[:, k] == label)


def align_labels_tables(s, cont, phi, gamma, N, K, rng):
    """align_labels! (src/misc.jl:61-108) from the contingency tables the sweep reduced on the
    device (`cont[pair][lb][la]` = observations with label la+1 in dataset a and lb+1 in dataset b):
    every count the Metropolis test needs is an entry of a table, a swap exchanges two rows (or
    columns) of the tables, and the allocations are relabelled once at the end - no pass over the
    n observations per proposal.  Same proposals, same random numbers, same result as
    :func:`align_labels`.  Returns (label counts N x K, per-pair agreement counts) after alignment."""
    pairs = phi_lab(K)
    phi_log = np.log(np.asarray(phi) + 1.0)
    # M[(a, b)][la, lb] for a < b
    M = {pr: np.array(cont[i], dtype=np.int64).T.copy() for i, pr in enumerate(pairs)}
    for k in range(K):
        others = [j for j in range(K) if j != k]
        rel = np.array([phi_log[i] for i, (a, b) in enumerate(pairs) if a == k or b == k])
        # T[j_index][l, lab] = observations with label l in dataset k and lab in dataset j
        T = np.stack([M[(k, j)] if k < j else M[(j, k)].T for j in others]).astype(np.float64)
        W = np.zeros((N, N))  # W[l, lab] = sum_j rel_j * T_j[l, lab], summed in dataset order like the reference
        for ji in range(len(others)):
            W = W + T[ji] * rel[ji]
        size = T[0].sum(axis=1)  # members of every label of dataset k
        perm = np.arange(N)      # perm[old label index] = current label index
        order = list(dict.fromkeys(s[:, k].tolist()))  # unique(), first-appearance order (1-based)
        for lab0 in order:
            # the reference tests `s[:, k] == label` with the label VALUE: after earlier swaps that value may
            # hold another group's members or nobody
            label = lab0 - 1
            if size[label] == 0:
                continue
            # one uniform per proposal, drawn as the reference does (N - 1 or N proposals per processed label; a block
            # draw is the same stream as scalar draws); the log-ratios of all proposals of the current
            # label come from W in one expression and are recomputed after an accepted swap
            u = rng.random(N - 1).tolist()
            ui = 0
            delta = ((W[label, :] + W[:, label]) - (W[label, label] + np.diagonal(W))).tolist()
            for new_label in range(N):
                if new_label == label:
                    continue
                if ui == len(u):  # a swap before the label's own index was reached: that index is proposed too
                    u.append(rng.random())
                accept = u[ui] < math.exp(min(delta[new_label], 50.0))
                ui += 1
                if accept:
                    W[[label, new_label]] = W[[new_label, label]]
                    T[:, [label, new_label]] = T[:, [new_label, label]]
                    size[[label, new_label]] = size[[new_label, label]]
                    gamma[[new_label, label], k] = gamma[[label, new_label], k]
                    # members that carried `label` now carry `new_label` and vice versa
                    a_, b_ = perm == label, perm == new_label
                    perm[a_], perm[b_] = new_label, label
                    label = new_label
                    delta = ((W[label, :] + W[:, label]) - (W[label, label] + np.diagonal(W))).tolist()
        s[:, k] = perm[s[:, k] - 1] + 1
        for ji, j in enumerate(others):  # the other datasets see dataset k's new labels
            if k < j:
                M[(k, j)] = T[ji].astype(np.int64)
            else:
                M[(j, k)] = T[ji].T.astype(np.int64)
    counts = np.zeros((N, K), dtype=np.int64)
    for k in range(K):
        j = 0 if k else 1
        counts[:, k] = M[(k, j)].sum(axis=1) if k < j else M[(j, k)].sum(axis=0)
    agree = np.array([int(np.trace(M[pr])) for pr in pairs], dtype=np.int64)
    return counts, agree


# ------------------------------------------------------------------ CSV (src/pmdi.jl:147-158,377-383)
def _jl(x):
    """A Float64 as Julia's writedlm prints it (shortest round-trip form; exponents as 1.0e-5)."""
    r = repr(float(x))
    if "e" in r:
        m, e = r.split("e")
        if "." not in m:
            m += ".0"
        r = f"{m}e{int(e)}"
    return r


def csv_header(K, n_obs, dataNames):
    pairs = phi_lab(K)
    cols = [f"MassParameter_{k + 1}" for k in range(K)]
    cols += [f"phi_{a + 1}_{b + 1}" for a, b in pairs] if K > 1 else ["phi_1_1"]
    cols += ["ll"]
    cols += [f"{dataNames[k]}_n{i + 1}" for k in range(K) for i in range(n_obs)]
    return ",".join(cols)


def csv_row(M, phi, ll, s):
    """[M; Phi; ll; vec(s)] promoted to Float64 (labels print as ``3.0``), dataset-major."""
    vals = [_jl(v) for v in M] + [_jl(v) for v in phi] + [_jl(ll)]
    vals += [f"{v}.0" for v in np.asarray(s).reshape(-1, order="F").tolist()]
    return ",".join(vals)


def n_hyper_columns(K):
    """Columns before the allocations: K + C(K,2) + (K == 1) + 1 (consensus_map.jl:38)."""
    return K + K * (K - 1) // 2 + (1 if K == 1 else 0) + 1


def read_allocations(outputFile, K, n_obs, burnin=0, thin=1):
    """Allocations of the retained rows, shape (rows, n_obs, K) - what ``generate_psm`` reads
    (src/output_analysis/consensus_map.jl:31-48)."""
    raw = np.loadtxt(outputFile, delimiter=",", skiprows=1, ndmin=2)
    raw = raw[burnin::thin, n_hyper_columns(K):]
    return raw.reshape(raw.shape[0], K, n_obs).transpose(0, 2, 1).astype(np.int64)


def _header_layout(header):
    """(K, n_obs, dataNames) from the header ``csv_header`` writes."""
    cols = header.strip().split(",")
    K = sum(c.startswith("MassParameter_") for c in cols)
    if K < 1 or "ll" not in cols:
        raise ValueError("not a pmdi() output header (no MassParameter_k / ll columns)")
    alloc = cols[n_hyper_columns(K):]
    names = list(dict.fromkeys(c.rsplit("_n", 1)[0] for c in alloc))
    if len(names) != K or len(alloc) % K:
        raise ValueError(f"header has {K} mass parameters but allocation columns of {len(names)} datasets")
    return K, len(alloc) // K, names


def read_chains(outputFiles, burnin=0, thin=1):
    """Allocations of one ``pmdi()`` CSV file or several (chains), with K, n_obs and the dataset names taken from the
    header.  Returns (list of (rows, n_obs, K) int64 arrays, one per file, each what ``read_allocations(file, K, n_obs,
    burnin, thin)`` returns; dataNames).  Every file must have the same layout.  Only the retained rows are parsed, and
    their label columns are read as integers in C (``pmdi_parse_allocations``, no device needed); DESIGN.md §14 gives
    its cost per row against ``np.loadtxt``."""
    files = [outputFiles] if isinstance(outputFiles, (str, os.PathLike)) else list(outputFiles)
    if not files:
        raise ValueError("no output files")
    if burnin < 0 or thin < 1:
        raise ValueError("need burnin >= 0 and thin >= 1")
    out, layout = [], None
    for f in files:
        with open(f, "rb") as fh:
            header = fh.readline().decode()
            body = fh.read()
        lay = _header_layout(header)
        if layout is not None and lay[:2] != layout[:2]:
            raise ValueError(f"{f}: K, n_obs = {lay[:2]} differ from {layout[:2]} of {files[0]}")
        layout = layout or lay
        K, n_obs, _ = lay
        total = body.count(b"\n") + (1 if body and not body.endswith(b"\n") else 0)
        if thin == 1:  # the rows after the burn-in are one stretch of the text: no split into lines
            at = 0
            for _ in range(min(burnin, total)):
                at = body.index(b"\n", at) + 1
            text, rows = body[at:], max(total - burnin, 0)
        else:
            kept = body.split(b"\n")[:total][burnin::thin]
            text, rows = b"\n".join(kept), len(kept)
        try:
            a = capi.parse_allocations(text, rows, n_hyper_columns(K), K * n_obs)
        except ValueError as e:
            raise ValueError(f"{f} (rows from {burnin + 1} every {thin}): {e}") from None
        out.append(a.reshape(rows, K, n_obs).transpose(0, 2, 1))
    return out, layout[2]


def _summary_of(outputFiles, burnin, thin, device):
    chains, _ = read_chains(outputFiles, burnin, thin)
    return _summary_of_chains(chains, device)


def _summary_of_chains(chains, device):
    rows, n_obs, K = chains[0].shape
    if any(c.shape[0] == 0 for c in chains):
        raise ValueError("a chain keeps no rows after burnin / thin")
    N = int(max(c.max() for c in chains))
    if N > 256:
        raise ValueError(f"labels up to {N}: the summaries take at most 256")
    S = capi.PosteriorSummary(K, n_obs, N, chains=len(chains), device=device)
    for c, a in enumerate(chains):
        S.add(c, a)
    return S


def generate_psm(outputFiles, burnin=0, thin=1, device=0):
    """The reference's ``generate_psm(outputFile, burnin, thin)`` (consensus_map.jl:31-65) on the GPU, over one
    CSV file or the files of several chains, pooled: shape (K + 1, n_obs, n_obs), the datasets in order, then Overall
    (their sum in k order divided by K).  Each dataset's PSM equals ``posterior_similarity`` of the rows of all files
    concatenated, bit for bit."""
    with _summary_of(outputFiles, burnin, thin, device) as S:
        return np.stack([S.psm(k) for k in range(S.K)] + [S.psm(None)])


def consensus_partition(outputFiles, burnin=0, thin=1, device=0):
    """Least-squares consensus (Dahl 2006) per dataset over the retained rows of one CSV file or several: the sample
    closest to the pooled PSM.  Returns (n_obs, K) labels."""
    with _summary_of(outputFiles, burnin, thin, device) as S:
        return np.stack([S.least_squares(k)[0] for k in range(S.K)], axis=1)


def chain_agreement(outputFiles, burnin=0, thin=1, device=0):
    """(max, mean) over i < j of |PSM_a - PSM_b| for every pair of chains (files) a < b, row-major, and dataset:
    two arrays of shape (C (C - 1) / 2, K)."""
    with _summary_of(outputFiles, burnin, thin, device) as S:
        return S.agreement()


def cut_tree(Z, n_clusters):
    """Labels 1..n_clusters of the n observations of scipy linkage matrix Z ((n - 1) x 4) cut into n_clusters: the
    last n_clusters - 1 merges (rows of Z) undone, the clusters numbered in order of their smallest observation
    index.  This is ``scipy.cluster.hierarchy.cut_tree(Z, n_clusters).ravel() + 1`` whenever the cut falls between
    two different heights; scipy takes merges of equal height in an order of its own, not by their row in Z."""
    Z = np.asarray(Z, dtype=np.float64)
    if Z.ndim != 2 or Z.shape[1] != 4:
        raise ValueError(f"Z must be (n - 1, 4), not {Z.shape}")
    n = Z.shape[0] + 1
    if not 1 <= int(n_clusters) <= n:
        raise ValueError(f"n_clusters {n_clusters} outside 1..{n}")
    rep = np.arange(2 * n - 1)  # smallest observation of every cluster id
    parent = np.arange(n)
    for m in range(n - int(n_clusters)):
        u, v = rep[int(Z[m, 0])], rep[int(Z[m, 1])]
        lo, hi = min(u, v), max(u, v)
        parent[hi] = lo
        rep[n + m] = lo
    while True:  # pointer jumping to the roots, each the smallest observation of its cluster
        up = parent[parent]
        if (up == parent).all():
            break
        parent = up
    return np.unique(parent, return_inverse=True)[1].astype(np.int64) + 1


def consensus_allocations(outputFiles, n_clusters, linkage, dataset=None, burnin=0, thin=1, device=0):
    """The reference's ``get_consensus_allocations(psm, k)`` (consensus_map.jl:92-105) over one CSV file or the files
    of several chains, pooled: the PSM of dataset ``dataset`` (0-based; None: Overall) clustered on the GPU with the
    named ``linkage`` ("single", "complete" or "average"; ``PosteriorSummary.hclust``), the tree cut into
    ``n_clusters``.  Returns n_obs labels in 1..n_clusters, numbered in order of their smallest observation."""
    if linkage not in capi.LINKAGES:
        raise ValueError(f"linkage is one of {sorted(capi.LINKAGES)}, not {linkage!r}")
    chains, _ = read_chains(outputFiles, burnin, thin)
    _, n_obs, K = chains[0].shape
    if not 1 <= int(n_clusters) <= n_obs:
        raise ValueError(f"n_clusters {n_clusters} outside 1..{n_obs}")
    if dataset is not None and not 0 <= int(dataset) < K:
        raise ValueError(f"dataset {dataset} outside 0..{K - 1}")
    with _summary_of_chains(chains, device) as S:
        return cut_tree(S.hclust(dataset, linkage=linkage), n_clusters)


def posterior_similarity(alloc):
    """PSM per dataset (consensus_map.jl:50-56): fraction of retained rows in which two
    observations share a label.  Returns (K, n, n)."""
    rows, n, K = alloc.shape
    out = np.zeros((K, n, n))
    for k in range(K):
        a = alloc[:, :, k]
        for r in range(rows):
            out[k] += a[r][:, None] == a[r][None, :]
    return out / rows


# ------------------------------------------------------------------ the entry point
class _Chain:
    """One chain of ``pmdi()``: its host RNG, hyper-parameters, allocations, context and output files, and the host
    steps of an iteration around the sweep (src/pmdi.jl:164-185 before it, :354-383 after it)."""

    def __init__(self, dataFiles, types, N, particles, rho, seed, factorised, stale_gamma_table, sstar_compat,
                 device_reductions, device, rank, world, engine=None):
        K, n_obs = len(dataFiles), int(dataFiles[0].shape[0])
        self.K, self.N, self.n_obs, self.n1, self.seed = K, N, n_obs, int(math.floor(rho * n_obs)), seed
        self.stale_gamma_table, self.factorised = stale_gamma_table, factorised
        self.sstar_compat, self.device_reductions = sstar_compat, device_reductions
        self.rng = rng = np.random.default_rng(seed)
        npairs = K * (K - 1) // 2
        self.M = np.full(K, 2.0)                                          # :59
        self.gamma = rng.gamma(1.0 / N, 1.0, (N, K)) + EPS                # :60
        self.phi = rng.gamma(1.0, 0.2, npairs) if K > 1 else np.zeros(1)  # :61
        self.s = np.stack([1 + rng.choice(N, size=n_obs, p=self.gamma[:, k] / self.gamma[:, k].sum())
                           for k in range(K)], axis=1).astype(np.int64)   # :63-66
        self.tables = FactorisedZ(N, K) if factorised else HyperTables(N, K)
        if not factorised:
            self.tables.refresh(self.gamma)
        Z = update_Z(self.phi, self.tables, self.gamma)                   # :95
        self.v = update_v(n_obs, Z, rng)                                  # :96
        self.counts = self.agree = None  # first iteration: counted from the initial allocation
        self.ctx = capi.Context(dataFiles, types, N, particles, device=device, rank=rank, n_ranks=world,
                                engine=engine)  # raises without a GPU
        self.stats = dict(sweep_device_ms=0.0, n_resamples=0, iterations=0)
        self.out = self.ffile = self.flags = self.feature_null = None
        self.offer = None  # pmdi(summary=S): every CSV row's allocations go to S as well

    def open(self, dataFiles, dataNames, outputFile, featureSelect_file):
        K, rng = self.K, self.rng
        if featureSelect_file is not None:                        # :106-128
            self.flags = [rng.random(d.shape[1]) < 0.5 for d in dataFiles]
            names = [f"{dataNames[k]}_d{d + 1}" for k in range(K) for d in range(dataFiles[k].shape[1])]
            self.ffile = open(featureSelect_file, "w")
            self.ffile.write(",".join(names) + "\n")
            self.ffile.write(",".join("true" if f else "false" for fl in self.flags for f in fl) + "\n")
            for k in range(K):
                self.ctx.set_flags(k, self.flags[k].astype(np.uint8))
            self.feature_null = [self.ctx.feature_null(k) for k in range(K)]
        self.out = open(outputFile, "w")
        self.out.write(csv_header(K, self.n_obs, dataNames) + "\n")  # :147-154

    def sweep_args(self, it):
        """The hyper-parameter updates of iteration `it` (:172-185); returns the sweep's arguments."""
        K, N, rng, tables = self.K, self.N, self.rng, self.tables
        order_obs = rng.permutation(self.n_obs) + 1                  # :172
        update_M(self.M, self.gamma, K, N, rng)                      # :176
        if not self.stale_gamma_table and not self.factorised:
            tables.refresh(self.gamma)
        update_gamma(self.gamma, self.phi, self.v, self.M, self.s, tables, rng, counts_all=self.counts)  # :177
        Pi = self.gamma / self.gamma.sum(axis=0, keepdims=True)     # :179
        if not self.stale_gamma_table and not self.factorised:
            tables.refresh(self.gamma)
        if K > 1:
            update_phi(self.phi, self.v, self.s, tables, rng, agree_all=self.agree, gamma=self.gamma)  # :181-183
        Z = update_Z(self.phi, tables, self.gamma)                   # :184
        self.v = update_v(self.n_obs, Z, rng)                        # :185
        return dict(s=self.s, order_obs=order_obs, n1=self.n1, Pi=Pi, phi=self.phi if K > 1 else None,
                    logweight_init=0.0 if it == 1 else 1.0,          # :99, :372
                    seed=self.seed, it=it, sstar_compat=self.sstar_compat)

    def record(self, r, it, thin, t0):
        """What iteration `it` does after its sweep `r`: feature selection, align_labels!, the CSV rows."""
        K, N, rng = self.K, self.N, self.rng
        self.s = s = np.array(r["s"], dtype=np.int64, order="C")
        self.stats["sweep_device_ms"] += r["device_ms"]
        self.stats["n_resamples"] += r["n_resamples"]
        if self.ffile is not None:                                # :354-370
            for k in range(K):
                _, fl = self.ctx.feature_select(k, s[:, k], self.feature_null[k], seed=self.seed, it=it)
                self.flags[k] = fl.astype(bool)
                self.ctx.set_flags(k, fl)
        # :375 - and the counts the next update_gamma! / update_Phi! read (update_hypers.jl:72,109-115),
        # from the tables the sweep reduced on the device
        if not self.device_reductions:
            align_labels(s, self.phi, self.gamma, N, K, rng)
            self.counts = self.agree = None
        elif K > 1:
            self.counts, self.agree = align_labels_tables(s, r["contingency"], self.phi, self.gamma, N, K, rng)
        else:
            self.counts, self.agree = np.array(r["label_counts"]), None
        ll = time.perf_counter() - t0                             # :377 (cumulative seconds)
        if it % thin == 0:                                        # :378-383
            self.out.write(csv_row(self.M, self.phi, ll, s) + "\n")
            if self.offer is not None:
                self.offer(s)
            if self.ffile is not None:
                self.ffile.write(",".join("true" if f else "false" for fl in self.flags for f in fl) + "\n")
        self.stats["iterations"] = it
        self.stats["loop_s"] = ll

    def close(self):
        for f in (self.out, self.ffile):
            if f is not None:
                f.close()
        if getattr(self, "ctx", None) is not None:
            self.ctx.close()


def pmdi(dataFiles, dataTypes, N, particles, rho, iter, outputFile, *, thin=1, featureSelect=None,
         dataNames=None, seed=0, device=0, stale_gamma_table=False, sstar_compat=False, factorised=None,
         device_reductions=True, reference_literal=False, distributed=False, chains=1, summary=None):
    """``pmdi(dataFiles, dataTypes, N, particles, rho, iter, outputFile; thin, featureSelect,
    dataNames)`` of src/pmdi.jl:36-40.  Side effect: the CSV file(s); returns a small dict of
    timings and counters (the reference returns nothing).

    ``chains=C > 1`` runs C independent chains side by side on one GPU: chain c is the run ``pmdi(..., seed=seed + c)``
    would make alone (same CSV rows but the elapsed-seconds column), and ``outputFile`` (and ``featureSelect`` when
    given) are sequences of C paths.  The chains' host steps run in lockstep, and each iteration sweeps all C chains in
    ONE launch of the spec engine (``capi.Group``), each chain on a share of the SMs.  Returns a list of C dicts.
    Needs K <= 4 and one GPU (not ``distributed``).  User-defined cluster types (``UserCluster`` or tags) work too: their
    chains run on the spec engine, so chain c writes what ``pmdi(..., seed=seed + c)`` writes alone with
    ``PMDI_ENGINE=spec`` (a single chain with user types still runs the pool engine by default).  Whether it pays
    depends on the problem: see DESIGN.md §13 for the measured aggregate rates against sweeping the chains one after
    another, with built-in and with user types (cfg2 with two user types: 1.6x at C = 2, 3.7x at C = 8 over sequential
    spec; a one-chain group measured 0.997x, and ``chains=1`` runs no group).

    ``summary=S`` (a ``capi.PosteriorSummary`` with K datasets, n_obs observations, at least C chains and labels up to
    at least N): chain c also offers every row it writes to its CSV file, the initial row included, to S as chain c, so
    that PSMs, the least-squares consensus and the chains' agreement are at hand without reading the files back (S
    applies its own burnin / thin to the rows offered).  Not with ``distributed``."""
    if reference_literal:  # the literal reference in one switch: never-refreshed gamma table, trajectories not permuted
        stale_gamma_table, sstar_compat, factorised = True, True, False
    t_entry = time.perf_counter()
    K = len(dataFiles)
    n_obs = int(dataFiles[0].shape[0])
    if dataNames is None:
        dataNames = [f"K{i + 1}" for i in range(K)]
    # the reference's asserts (src/pmdi.jl:50-55)
    assert len(dataTypes) == K, "Number of datatypes not equal to number of datasets"
    assert len(dataNames) == K, "Number of data names not equal to number of datasets"
    assert all(d.shape[0] == n_obs for d in dataFiles), \
        "Datasets don't have same number of observations. Each row must correspond to the same " \
        "underlying observational unit across datasets."
    assert 0 < rho < 1, "ρ must be between 0 and 1"
    assert 1 < N <= n_obs, \
        f"Number of clusters must be greater than 1 and not greater than the number of observations, " \
        f"suggest using floor(log(n)) = {int(math.floor(math.log(n_obs)))}"
    assert particles > 1, "Conditional particle filter requires 2 or more particles"
    n1 = int(math.floor(rho * n_obs))
    assert n1 >= 1, "floor(ρ * n_obs) must be at least 1 (order_obs[n1:n_obs], src/pmdi.jl:209)"

    types = [_tag(t) for t in dataTypes]
    C = int(chains)
    if C < 1:
        raise ValueError("chains must be >= 1")
    outputs, fsel = [outputFile], [featureSelect]
    if C > 1:
        if distributed:
            raise ValueError("chains > 1 runs several chains on one GPU; distributed=True shards one chain's particles "
                             "over the GPUs of a node: choose one")
        if K > 4:
            raise ValueError("chains > 1 sweeps the chains in one launch of the spec engine, which runs K <= 4 "
                             "datasets (K > 4 runs the pool engine, which has no group launch)")
        outputs = list(outputFile)
        fsel = list(featureSelect) if featureSelect is not None else [None] * C
        if len(outputs) != C or len(fsel) != C:
            raise ValueError(f"chains={C}: outputFile (and featureSelect when given) need {C} paths")
    if summary is not None:
        if distributed:
            raise ValueError("summary= takes the allocations of one GPU's chains; with distributed=True read the CSV "
                             "file back (generate_psm)")
        if (summary.K, summary.n) != (K, n_obs) or summary.chains < C or summary.N < N:
            raise ValueError(f"summary has K={summary.K}, n_obs={summary.n}, {summary.chains} chains, N={summary.N}; "
                             f"this run needs K={K}, n_obs={n_obs}, >= {C} chains, N >= {N}")
    # the N^K-row tables of :69-92 where they are small, the factorised sums (FactorisedZ) otherwise
    if factorised is None:
        factorised = N ** K > 200_000
    if factorised and stale_gamma_table:
        raise ValueError("stale_gamma_table needs the literal N^K tables")

    # distributed: one process per GPU of a node (torch.distributed initialised by the caller), the particles sharded
    # over the ranks; every rank runs this same loop with the same seed (identical hyper-parameters everywhere),
    # rank 0 writes the files
    rank, world = 0, 1
    if distributed:
        import torch.distributed as dist
        rank, world = dist.get_rank(), dist.get_world_size()
    # a group runs the spec engine; user types default to pool on one GPU, so their chains ask for spec themselves
    engine = "spec" if C > 1 and any(t >= 16 for t in types) else None
    chain_list, group = [], None
    try:
        for c in range(C):
            chain_list.append(_Chain(dataFiles, types, N, particles, rho, seed + c, factorised, stale_gamma_table,
                                     sstar_compat, device_reductions, device, rank, world, engine))
        if world > 1:
            chain_list[0].ctx.connect()
        if rank != 0:
            outputs, fsel = ["/dev/null"], ["/dev/null" if featureSelect is not None else None]
        for ch, o, f in zip(chain_list, outputs, fsel):
            ch.open(dataFiles, dataNames, o, f)
        if C > 1:
            group = capi.Group([ch.ctx for ch in chain_list])
        t0 = time.perf_counter()
        for c, ch in enumerate(chain_list):
            ch.stats["setup_s"] = t0 - t_entry  # data to the device, pool allocation (and a user type's compilation)
            ch.out.write(csv_row(ch.M, ch.phi, 0, ch.s) + "\n")  # :158
            if summary is not None:
                ch.offer = (lambda a, c=c: summary.add(c, a))
                ch.offer(ch.s)
        for it in range(1, iter + 1):                             # :164
            args = [ch.sweep_args(it) for ch in chain_list]
            if group is not None:
                for ch, a in zip(chain_list, args):
                    ch.ctx.upload(**a)
                group.run()
                res = [ch.ctx.download(cluster_sizes=False) for ch in chain_list]
            else:
                ctx = chain_list[0].ctx
                do_sweep = ctx.sweep_sharded if world > 1 else ctx.sweep
                res = [do_sweep(**args[0], cluster_sizes=False)]  # :188-350, :373
            for ch, r in zip(chain_list, res):
                ch.record(r, it, thin, t0)
    finally:
        if group is not None:
            group.close()
        for ch in chain_list:
            ch.close()
    stats = [ch.stats for ch in chain_list]
    return stats if C > 1 else stats[0]

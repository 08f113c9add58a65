"""Device memory of the host library comes back: summary read-outs free their temporaries, and contexts, groups and
summaries return what they hold when they are destroyed.

Free memory is read with torch.cuda.mem_get_info, which is device-wide and moves with anything else on the GPU.  So
each check allows 8 MB of drift, and each loop would leak several times that if the library kept what it allocates.
"""
import numpy as np
import pytest

from helpers import C, G, NB, problem

pytestmark = pytest.mark.gpu

MB = 1 << 20
SLACK = 8 * MB


def _free():
    import torch
    torch.cuda.synchronize()
    return torch.cuda.mem_get_info(0)[0]


def test_summary_least_squares_frees_its_buffers():
    """n = 64, K = 1, one chain of 100,000 rows: every least_squares call takes (R + 2) x 8 bytes = 0.8 MB for the
    per-sample sums.  Kept, 100 calls would leak 80 MB; free memory may drop by less than 8 MB."""
    from pmdi_b200 import capi
    n, rows = 64, 100_000
    a = np.random.default_rng(0).integers(1, 4, size=(rows, n, 1))
    with capi.PosteriorSummary(1, n, 3) as S:
        S.add(0, a)
        S.least_squares(0)  # warm-up: the first call loads the summary kernels
        before = _free()
        for _ in range(100):
            S.least_squares(0)
        assert before - _free() < SLACK


def test_summary_agreement_frees_its_buffers():
    """n = 3,072 (300 tiles, so 2 x 148 = 296 CTAs on a B200), K = 1, 8 chains (28 pairs): every agreement call
    takes 2 x 296 x 28 doubles = 0.13 MB of partials.  Kept, 600 calls would leak 80 MB; free memory may drop by less
    than 8 MB.  The chains' pair counts take about 160 MB."""
    from pmdi_b200 import capi
    n, chains = 3072, 8
    rng = np.random.default_rng(1)
    with capi.PosteriorSummary(1, n, 3, chains=chains) as S:
        for c in range(chains):
            S.add(c, rng.integers(1, 4, size=(4, n, 1)))
        S.agreement()  # warm-up
        before = _free()
        for _ in range(600):
            S.agreement()
        assert before - _free() < SLACK


def _round(pr, args):
    """Create, use and destroy a context on each engine, a two-member group and a summary."""
    from pmdi_b200 import capi
    for engine in ("spec", "pool", None):  # None: PMDI_ENGINE=dense
        with capi.Context(pr["data"], pr["types"], pr["N"], pr["P"], engine=engine) as ctx:
            got = ctx.sweep(**args)
            assert got["engine"] == (engine or "dense")
            ctx.psm(got["s"][None])
            ctx.feature_select(0, got["s"][:, 0], ctx.feature_null(0), seed=1, it=1)
            ctx.cluster_eval(0, np.arange(1, 11), obs_1based=11, logmarginal=True)
    ctxs = [capi.Context(pr["data"], pr["types"], pr["N"], pr["P"], engine="spec") for _ in range(2)]
    with capi.Group(ctxs) as grp:
        grp.sweep([args, args])
        ctxs[0].close()  # a member destroyed before its group
    ctxs[1].close()
    with capi.PosteriorSummary(pr["K"], pr["n"], pr["N"]) as S:
        S.add(0, got["s"][None])
        S.psm(0)


def test_create_use_destroy_returns_memory(monkeypatch):
    """Five rounds of _round: free memory after rounds 2..5 is within 8 MB of what it was after round 1 (which loads
    the modules and sizes the driver's per-context reservations)."""
    monkeypatch.setenv("PMDI_ENGINE", "dense")  # for the context that asks for no engine of its own
    pr = problem(sets=[(G, 130, 0), (C, 65, 3), (NB, 100, 0)], n=120, N=12, P=64, seed=3)
    args = dict(s=pr["s"], order_obs=pr["order"], n1=pr["n1"], Pi=pr["Pi"], phi=pr["phi"], seed=11, it=3)
    _round(pr, args)
    base = _free()
    for _ in range(4):
        _round(pr, args)
        assert abs(_free() - base) < SLACK

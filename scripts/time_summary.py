#!/usr/bin/env python
"""Posterior summaries (capi.PosteriorSummary, pmdi_summary_*) on one GPU.  First line: the card's name, power limit and
SM clock.  Then, for n in {500, 5,000, 20,000}, K = 2, R in {1,000, 4,000} rows in all, spread over chains in {1, 4, 8}
(labels 1..20 drawn around a planted partition), one line per arm:

  count      the tile pass over all R rows: kernel time of k_summary_count (torch.profiler, a run of its own),
             pair-sample comparisons per second (R * K * n (n + 1) / 2 over the kernel time), and end to end: wall time
             of the adds, the pass and one f32 read-out (host staging and the device -> host copy included), per row
  readout    psm(k) of the pooled chains as f64 and f32 (wall, device -> host copy included), psm() Overall
  ls         least_squares(0) (wall)
  agreement  agreement() (wall; chains >= 2)
  context    the existing per-row loop, Context.psm, on the same rows: per-row time from the difference of two row counts
             (its read-out cancels; the faster of 3 repeats of each), against the tile pass per row, kernel only and end
             to end (a difference that is not positive is reported as not measured)
  numpy      pmdi.posterior_similarity per row where n <= 2,000

Then pmdi(chains=4) on cfg2 for 20 iterations, without and with summary= (alternated, 3 rounds each): aggregate
iterations/s.
  python scripts/time_summary.py [out.jsonl]"""
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]
import pmdi_b200  # noqa: E402,F401
from pmdi_b200 import capi, synth  # noqa: E402
from pmdi_b200 import pmdi as host  # noqa: E402

SHAPES = [500, 5000, 20000]
ROWS = [1000, 4000]
CHAINS = [1, 4, 8]
K, N = 2, 20


def samples(n, R, seed=0):
    rng = np.random.default_rng(seed)
    base = rng.integers(1, N + 1, (n, K))
    a = np.repeat(base[None], R, axis=0)
    flip = rng.random(a.shape) < 0.2
    a[flip] = rng.integers(1, N + 1, int(flip.sum()))
    return a


def fill(S, a, C):
    per = len(a) // C
    for c in range(C):
        S.add(c, a[c * per:(c + 1) * per])


def wall(f):
    t = time.perf_counter()
    r = f()
    return time.perf_counter() - t, r


def count_kernel_ms(n, a, C):
    """Sum of k_summary_count durations over one fill + flush, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    with capi.PosteriorSummary(K, n, N, chains=C) as S:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fill(S, a, C)
            S.psm(0, dtype=np.float32)
        return sum(e.device_time_total for e in prof.key_averages() if "k_summary_count" in e.key) / 1e3


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    if capi.device_count() < 1:
        raise SystemExit("time_summary.py needs a CUDA device")
    import torch
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    lines = []

    def emit(d):
        lines.append(d)
        print(json.dumps(d), flush=True)
        if out_path:
            with open(out_path, "w") as f:
                for ln in lines:
                    f.write(json.dumps(ln) + "\n")

    emit(dict(device=torch.cuda.get_device_name(0), nvidia_smi=smi[:1]))
    # warm-up: module load, first launches of every kernel
    with capi.PosteriorSummary(K, 300, N, chains=2) as S:
        fill(S, samples(300, 300), 2)
        S.psm(0), S.psm(0, dtype=np.float32), S.least_squares(0), S.agreement()
    for n in SHAPES:
        for R in ROWS:
            a = samples(n, R, seed=n + R)
            comps = R * K * n * (n + 1) / 2
            for C in CHAINS:
                base = dict(n=n, K=K, rows=R, chains=C)
                kern = count_kernel_ms(n, a, C)
                with capi.PosteriorSummary(K, n, N, chains=C) as S:
                    t_e2e, _ = wall(lambda: (fill(S, a, C), S.psm(0, dtype=np.float32)))
                    t_ro32, _ = wall(lambda: S.psm(0, dtype=np.float32))
                    t_ro64, _ = wall(lambda: S.psm(0))
                    t_all, _ = wall(lambda: S.psm(None))
                    emit(dict(base, arm="count", kernel_ms=round(kern, 3),
                              comparisons_per_s=float(f"{comps / (kern / 1e3):.4g}"),
                              kernel_us_per_row=round(kern * 1e3 / R, 3),
                              add_pass_readout_ms=round(t_e2e * 1e3, 2),
                              e2e_us_per_row=round(t_e2e * 1e6 / R, 2)))
                    emit(dict(base, arm="readout", f64_ms=round(t_ro64 * 1e3, 2), f32_ms=round(t_ro32 * 1e3, 2),
                              overall_f64_ms=round(t_all * 1e3, 2)))
                    t_ls, (_, loss, best) = wall(lambda: S.least_squares(0))
                    t_ls2, _ = wall(lambda: S.least_squares(0))
                    emit(dict(base, arm="ls", ms=[round(t_ls * 1e3, 2), round(t_ls2 * 1e3, 2)], best=list(best)))
                    if C > 1:
                        t_ag, _ = wall(lambda: S.agreement())
                        emit(dict(base, arm="agreement", ms=round(t_ag * 1e3, 2)))
                if C == 1:
                    # the existing per-row loop on the same rows
                    m0, m1 = 5, 45 if n >= 20000 else 405
                    with capi.Context([np.zeros((n, 1))] * K, [capi.GAUSSIAN] * K, N, 4) as ctx:
                        ctx.psm(a[:m0])
                        t0 = min(wall(lambda: ctx.psm(a[:m0]))[0] for _ in range(3))
                        t1 = min(wall(lambda: ctx.psm(a[:m1]))[0] for _ in range(3))
                    per_row = (t1 - t0) / (m1 - m0)
                    if per_row <= 0:
                        emit(dict(base, arm="context", measured=False, reason="the difference of the two wall times is "
                                  f"not positive ({per_row * 1e3:.4f} ms per row)"))
                    else:
                        emit(dict(base, arm="context", ms_per_row=round(per_row * 1e3, 4),
                                  tile_pass_kernel_ms_per_row=round(kern / R, 5),
                                  speedup_kernel_only=round(per_row * 1e3 / (kern / R), 1),
                                  tile_pass_e2e_ms_per_row=round(t_e2e * 1e3 / R, 5),
                                  speedup_end_to_end=round(per_row / (t_e2e / R), 1)))
                    if n <= 2000:
                        t_np, _ = wall(lambda: host.posterior_similarity(a[:50]))
                        emit(dict(base, arm="numpy", ms_per_row=round(t_np * 1e3 / 50, 3)))
    # pmdi(chains=4) on cfg2 with and without summary=
    cfg = synth.make_config("cfg2_multiomics")
    iters, C = 20, 4
    with tempfile.TemporaryDirectory() as td:
        outs = [os.path.join(td, f"c{c}.csv") for c in range(C)]
        rates = {"without": [], "with": []}
        for rnd in range(3):
            for arm in ("without", "with"):
                S = capi.PosteriorSummary(len(cfg["data"]), cfg["n"], cfg["N"], chains=C) if arm == "with" else None
                st = host.pmdi(cfg["data"], cfg["types"], cfg["N"], cfg["P"], cfg["rho"], iters, outs, seed=5,
                               chains=C, summary=S)
                rates[arm].append(round(C * iters / max(s["loop_s"] for s in st), 2))
                if S is not None:
                    assert S.rows(0) == iters + 1
                    S.close()
        emit(dict(config="cfg2_multiomics", pmdi_chains=C, iterations=iters,
                  aggregate_iters_per_s_without=rates["without"], aggregate_iters_per_s_with=rates["with"]))


if __name__ == "__main__":
    main()

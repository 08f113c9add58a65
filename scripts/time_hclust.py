#!/usr/bin/env python
"""Hierarchical consensus clustering of the pooled PSM on one GPU (PosteriorSummary.hclust, pmdi_summary_hclust)
against the host path a user has without it: the PSM read out, squareform(1 - PSM), scipy's linkage.

K = 2, 1,000 rows (labels 1..20 drawn around a planted partition, as scripts/time_summary.py), dataset 0,
n in {500, 5,000, 20,000}, linkage single / complete / average.  One line per (n, linkage), each with the card's name
and power limit read in the same call:

  gpu_wall_ms      wall time of hclust() (warmed up, median of repeats; set-up, merge kernel and copy included)
  gpu_kernel_ms    device time of the k_hclust_* kernels (torch.profiler, a call of its own)
  rescans_per_merge   rows rescanned per merge (the statistic the library returns)
  scipy_readout_ms psm(0) read-out plus squareform(1 - psm) (what scipy's path needs first)
  scipy_linkage_ms scipy.cluster.hierarchy.linkage on that condensed matrix (one call)
  ari_2_30         adjusted Rand index of the GPU's cut against scipy's (pmdi.cut_tree on both Z), c = 2..30;
                   ties make a difference legitimate, so this is reported, not asserted

  python scripts/time_hclust.py [out.jsonl]"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]
import pmdi_b200  # noqa: E402,F401
from pmdi_b200 import capi  # noqa: E402
from pmdi_b200 import pmdi as host  # noqa: E402

SHAPES = [500, 5000, 20000]
LINKAGES = ["single", "complete", "average"]
K, N, ROWS = 2, 20, 1000


def samples(n, R, seed=0):
    rng = np.random.default_rng(seed)
    base = rng.integers(1, N + 1, (n, K))
    a = np.repeat(base[None], R, axis=0)
    flip = rng.random(a.shape) < 0.2
    a[flip] = rng.integers(1, N + 1, int(flip.sum()))
    return a


def ari(a, b):
    from scipy.special import comb
    ct = np.zeros((a.max() + 1, b.max() + 1))
    np.add.at(ct, (a, b), 1)
    s = comb(ct, 2).sum()
    sa, sb = comb(ct.sum(1), 2).sum(), comb(ct.sum(0), 2).sum()
    e = sa * sb / comb(len(a), 2)
    return float((s - e) / (0.5 * (sa + sb) - e))


def kernel_ms(S, linkage):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        S.hclust(0, linkage=linkage)
    return sum(e.device_time_total for e in prof.key_averages() if "k_hclust" in e.key) / 1e3


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    if capi.device_count() < 1:
        raise SystemExit("time_hclust.py needs a CUDA device")
    from scipy.cluster import hierarchy
    from scipy.spatial.distance import squareform
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in smi.split(",")]
    lines = []
    for n in SHAPES:
        a = samples(n, ROWS, seed=n)
        with capi.PosteriorSummary(K, n, N) as S:
            S.add(0, a)
            t = time.perf_counter()
            psm = S.psm(0)
            d = squareform(1.0 - psm, checks=False)
            readout = time.perf_counter() - t
            del psm
            for linkage in LINKAGES:
                Z = S.hclust(0, linkage=linkage)  # warm-up
                reps = 3 if n >= 20000 else 7
                walls = []
                for _ in range(reps):
                    t = time.perf_counter()
                    Z2 = S.hclust(0, linkage=linkage)
                    walls.append(time.perf_counter() - t)
                assert (Z2 == Z).all()
                rescans = S.last_rescans
                kms = kernel_ms(S, linkage)
                t = time.perf_counter()
                Zs = hierarchy.linkage(d, method=linkage)
                t_scipy = time.perf_counter() - t
                aris = [ari(host.cut_tree(Z, c), host.cut_tree(Zs, c)) for c in range(2, 31)]
                rec = dict(arm="hclust", gpu=name, power_limit=power, n=n, K=K, rows=ROWS, linkage=linkage,
                           gpu_wall_ms=round(1e3 * float(np.median(walls)), 3), gpu_kernel_ms=round(kms, 3),
                           rescans_per_merge=round(rescans / (n - 1), 4),
                           scipy_readout_ms=round(1e3 * readout, 1), scipy_linkage_ms=round(1e3 * t_scipy, 1),
                           speedup_vs_scipy=round((readout + t_scipy) / float(np.median(walls)), 1),
                           ari_2_30_min=round(min(aris), 6), ari_2_30_mean=round(float(np.mean(aris)), 6),
                           same_z_as_scipy=bool(np.array_equal(Z[:, [0, 1, 3]], Zs[:, [0, 1, 3]])))
                print(json.dumps(rec), flush=True)
                lines.append(rec)
            del d
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()

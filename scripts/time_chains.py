#!/usr/bin/env python
"""Several chains on one GPU: C contexts swept one after another, each with the whole GPU ("sequential"), against the
same C chains swept as ONE group (capi.Group, pmdi_group_run: one cooperative launch, each chain on a share of the
SMs).  Timed alternately in one process on settled chains (8 untimed burn-in sweeps per chain, as
scripts/time_user_types.py), round by round: a round sweeps every chain once (upload, run, download).
Configurations: cfg1 and cfg2 at C = 1, 2, 4, 8; cfg4 at C = 2 (reported as not measured when it does not fit).
Per arm: aggregate sweeps/s (C / host wall time of a round, which ends in the downloads' synchronisations), the same
from device time (C / the sum of the sweeps' kernel times for sequential, C / the group kernel's time for the group),
microseconds per observation step of one chain, CTAs per chain.  Then pmdi() end to end at chains = 1 and 4 for cfg1
and cfg2 (host loop included): aggregate MCMC iterations/s.  First line: the card's name and power limit.
  python scripts/time_chains.py [rounds=10] [out.jsonl]"""
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
from pmdi_b200.pmdi import pmdi  # noqa: E402

BURN_IN = 8
PLAN = [("cfg1_iris", (1, 2, 4, 8)), ("cfg2_multiomics", (1, 2, 4, 8)), ("cfg4_singlecell", (2,))]
PMDI_PLAN = [("cfg1_iris", 60), ("cfg2_multiomics", 20)]


class Chain:
    """One context and its chain of sweeps (split form, so that a group can run it)."""

    def __init__(self, cfg, hy, n1, seed):
        self.cfg, self.hy, self.n1, self.seed = cfg, hy, n1, seed
        self.ctx = capi.Context(cfg["data"], cfg["types"], cfg["N"], cfg["P"])
        self.rng = np.random.default_rng(seed)
        self.s, self.it = hy["s"], 0

    def upload(self):
        self.ctx.upload(self.s, self.rng.permutation(self.cfg["n"]) + 1, self.n1, self.hy["Pi"], self.hy["phi"],
                        seed=self.seed, it=self.it, logweight_init=float(self.it > 0))

    def download(self):
        r = self.ctx.download(cluster_sizes=False)
        self.s, self.it = r["s"], self.it + 1
        return r


def seq_round(chains):
    t = time.perf_counter()
    rs = []
    for ch in chains:
        ch.upload()
        ch.ctx.run()
        rs.append(ch.download())
    return time.perf_counter() - t, sum(r["sweep_kernel_ms"] for r in rs), rs


def group_round(chains, grp):
    t = time.perf_counter()
    for ch in chains:
        ch.upload()
    grp.run()
    rs = [ch.download() for ch in chains]
    return time.perf_counter() - t, rs[0]["sweep_kernel_ms"], rs


def measure(name, C, rounds):
    cfg = synth.make_config(name)
    K = len(cfg["sets"])
    hy = synth.make_hypers(K, cfg["N"], cfg["n"], cfg["seed"])
    n1 = int(np.floor(cfg["rho"] * cfg["n"]))
    steps = cfg["n"] - n1 + 1
    seq = [Chain(cfg, hy, n1, 100 + c) for c in range(C)]
    grouped = [Chain(cfg, hy, n1, 100 + c) for c in range(C)]
    grp = capi.Group([ch.ctx for ch in grouped])
    try:
        for _ in range(BURN_IN):
            seq_round(seq)
            group_round(grouped, grp)
        res = {"sequential": [], "group": []}
        for _ in range(rounds):  # alternate the arms round by round
            res["sequential"].append(seq_round(seq)[:2])
            res["group"].append(group_round(grouped, grp)[:2])
        # same seeds, same chains: the two arms must have computed the same allocations
        same = all(np.array_equal(a.s, b.s) for a, b in zip(seq, grouped))
        out = dict(config=name, chains=C, steps=steps, burn_in=BURN_IN, rounds=rounds, same_allocations=same)
        for arm, v in res.items():
            wall, ker = np.array([x[0] for x in v]), np.array([x[1] for x in v])
            out[arm] = dict(
                sweeps_per_s_wall=round(C / float(np.median(wall)), 2),
                sweeps_per_s_kernel=round(C / (1e-3 * float(np.median(ker))), 2),
                round_ms_median=round(1e3 * float(np.median(wall)), 3),
                kernel_ms_median=round(float(np.median(ker)), 3),
                us_per_step_per_chain=round(1e3 * float(np.median(ker)) / (steps * (C if arm == "sequential" else 1)), 2))
        out["group_over_sequential_wall"] = round(out["group"]["sweeps_per_s_wall"] /
                                                  out["sequential"]["sweeps_per_s_wall"], 3)
        return out
    finally:
        grp.close()
        for ch in seq + grouped:
            ch.ctx.close()


def grid_of(name, C, n_sm):
    """CTAs per chain alone and in a group of C (the library's split, restated for the report)."""
    cfg = synth.CONFIGS[name]

    def split(budget):
        Ps, K = cfg["P"], len(cfg["sets"])
        gp = max(1, min(min(Ps, (Ps * K + 14) // 15), budget - max(8, budget // 8)))
        ge = max(1, min(budget - gp - 1, 64))
        return dict(G=gp + ge + 1, GP=gp, GE=ge)
    solo = split(n_sm)
    budget = solo["G"] if C * solo["G"] <= n_sm else n_sm * solo["G"] // (C * solo["G"])
    return dict(alone=solo, in_group=split(budget))


def pmdi_rate(name, iters, C, td):
    cfg = synth.make_config(name)
    outs = [os.path.join(td, f"{name}_{C}_{c}.csv") for c in range(C)]
    st = pmdi(cfg["data"], cfg["types"], cfg["N"], cfg["P"], cfg["rho"], iters, outs if C > 1 else outs[0],
              seed=5, chains=C)
    st = st if C > 1 else [st]
    loop = max(s["loop_s"] for s in st)
    return dict(config=name, pmdi_chains=C, iterations=iters, loop_s=round(loop, 3),
                aggregate_iters_per_s=round(C * iters / loop, 2),
                sweep_device_ms_per_iteration=round(float(np.mean([s["sweep_device_ms"] / iters for s in st])), 3))


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 10
    out_path = sys.argv[2] if len(sys.argv) > 2 else None
    if capi.device_count() < 1:
        raise SystemExit("time_chains.py needs a CUDA device")
    import torch
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    lines = [dict(device=torch.cuda.get_device_name(0), nvidia_smi=smi[:1], sms=n_sm, burn_in=BURN_IN, rounds=rounds)]
    print(json.dumps(lines[-1]), flush=True)

    def emit(d):
        lines.append(d)
        print(json.dumps(d), flush=True)
        if out_path:
            with open(out_path, "w") as f:
                for ln in lines:
                    f.write(json.dumps(ln) + "\n")

    for name, cs in PLAN:
        for C in cs:
            try:
                d = measure(name, C, rounds if name != "cfg4_singlecell" else max(3, rounds // 2))
                d["ctas_per_chain"] = grid_of(name, C, n_sm)
            except capi.PmdiError as e:  # e.g. cfg4's pools of 2 x 2 chains do not fit the GPU's memory
                d = dict(config=name, chains=C, measured=False, reason=str(e)[:300])
            emit(d)
    with tempfile.TemporaryDirectory() as td:
        for name, iters in PMDI_PLAN:
            for C in (1, 4):
                emit(pmdi_rate(name, iters, C, td))


if __name__ == "__main__":
    main()

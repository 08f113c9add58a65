#!/usr/bin/env python
"""Cost of the wide kernels (sweep_wide.cu), which read each observation from global memory, against the staged ones.
One GPU; every line is JSON on stdout and in profiles/r08_wide.jsonl (or the path given as the first argument).

Workloads (settled chains: 8 burn-in sweeps, then timed sweeps; CUDA events of the library):
  boundary   two Gaussian datasets of 6,000 features (staged) and of 6,750 (wide; 1.125x the work), n = 1,000, N = 20,
             P = 256, spec engine, alternated in one process; then one Gaussian dataset of 12,000 and of 13,500 features
             (both wide: a row of more than 8,192 features), with phase timers on the last sweep
  omics      cfg2's structure widened: Gaussian 20,000, Categorical 5,000 (3 levels), NegBinom 10,000; n = 500, N = 20,
             P = 256, rho = 0.25, on spec and on pool; one settled sweep of the oracle (the reference arm); pmdi() end to
             end with featureSelect, in iterations/s
The bytes model per step counts, for each row task (the evaluation of one row, and for spec of its child), the
statistics read and written and the two observations read, per feature: Gaussian 4 x 8 B read + 4 x 8 B written + 2 x 8 B
of x; NegBinom and packed Categorical 8 + 8 + 2 x 4 B.  Over the kernel time per step it gives the rate the step
implies; a rate far below HBM bandwidth means the step is bound by latency."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pmdi_b200  # noqa: E402,F401
from pmdi_b200 import capi, synth  # noqa: E402

OUT = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r08_wide.jsonl")
BURN, TIMED = 8, int(os.environ.get("TIME_WIDE_SWEEPS", "6"))
BYTES = {synth.GAUSSIAN: 32 + 32 + 16, synth.CATEGORICAL: 8 + 8 + 8, synth.NEGBINOM: 8 + 8 + 8}
G, C, NB = synth.GAUSSIAN, synth.CATEGORICAL, synth.NEGBINOM
lines = []


def emit(d):
    print(json.dumps(d), flush=True)
    lines.append(d)


class Chain:
    def __init__(self, name, sets, n, N, P, engine=None, seed=5):
        self.name, self.sets, self.n, self.N, self.P = name, sets, n, N, P
        self.data, self.types, _ = synth.make_data(sets, n, 5, seed)
        self.K = len(sets)
        self.hy = synth.make_hypers(self.K, N, n, seed)
        self.n1 = n // 4
        self.steps = n - self.n1 + 1
        self.ctx = capi.Context(self.data, self.types, N, P, engine=engine)
        self.s, self.it = self.hy["s"], 0
        self.rng = np.random.default_rng(seed)

    def sweep(self, phases=False):
        r = self.ctx.sweep(self.s, self.rng.permutation(self.n) + 1, self.n1, self.hy["Pi"], self.hy["phi"], seed=9,
                           it=self.it, logweight_init=float(self.it > 0), time_phases=phases, cluster_sizes=False)
        self.s, self.it = r["s"], self.it + 1
        return r

    def line(self, rs):
        kern = np.array([r["sweep_kernel_ms"] for r in rs])
        dev = np.array([r["device_ms"] for r in rs])
        st = self.steps
        tasks = np.zeros(self.K)  # row tasks per step and dataset
        for r in rs:
            comp = np.array(r["rows_computed"][:self.K], dtype=float)
            tasks += (comp / 2 if r["engine"] == "spec" else comp) / st
        tasks /= len(rs)
        bytes_step = float(sum(tasks[k] * self.sets[k][1] * BYTES[self.sets[k][0]] for k in range(self.K)))
        us = 1e3 * float(np.median(kern)) / st
        return dict(workload=self.name, engine=rs[-1]["engine"], wide=self.ctx.wide,
                    D=[d for _, d, _ in self.sets], n=self.n, N=self.N, P=self.P, sweeps=len(rs),
                    ms_per_sweep=round(float(np.median(dev)), 3), kernel_ms=round(float(np.median(kern)), 3),
                    kernel_ms_min=round(float(kern.min()), 3), kernel_ms_max=round(float(kern.max()), 3),
                    us_per_step=round(us, 2),
                    rows_evaluated_per_step=round(float(np.mean([sum(r["rows_evaluated"][:self.K]) for r in rs])) / st, 1),
                    row_tasks_per_step=round(float(tasks.sum()), 1),
                    model_MB_per_step=round(bytes_step / 1e6, 3), model_TB_per_s=round(bytes_step / (us * 1e-6) / 1e12, 3),
                    resamples=int(np.mean([r["n_resamples"] for r in rs])))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def alternated(chains, phases_last=False):
    for c in chains:
        for _ in range(BURN):
            c.sweep()
    res = {c.name: [] for c in chains}
    for i in range(TIMED):
        for c in chains:
            res[c.name].append(c.sweep())
    for c in chains:
        emit(c.line(res[c.name]))
        if phases_last:
            r = c.sweep(phases=True)
            emit(dict(workload=c.name, phases_ms=[round(v, 3) for v in r["phase_ms"]],
                      phases_ms_max=[round(v, 3) for v in r["phase_ms_max"]], kernel_ms=round(r["sweep_kernel_ms"], 3)))
        c.ctx.close()


def main():
    if capi.device_count() < 1:
        raise SystemExit("time_wide.py needs a CUDA device")
    emit(dict(gpu=gpu_info(), burn_in=BURN, timed=TIMED))
    which = os.environ.get("TIME_WIDE", "boundary,omics").split(",")
    if "boundary" in which:
        alternated([Chain("boundary_2x6000", [(G, 6000, 0), (G, 6000, 0)], 1000, 20, 256),
                    Chain("boundary_2x6750", [(G, 6750, 0), (G, 6750, 0)], 1000, 20, 256)], phases_last=True)
        alternated([Chain("single_12000", [(G, 12000, 0)], 1000, 20, 256),
                    Chain("single_13500", [(G, 13500, 0)], 1000, 20, 256)], phases_last=True)
    if "omics" in which:
        sets = [(G, 20000, 0), (C, 5000, 3), (NB, 10000, 0)]
        alternated([Chain("omics_spec", sets, 500, 20, 256, engine="spec"),
                    Chain("omics_pool", sets, 500, 20, 256, engine="pool")], phases_last=True)
        from oracle import oracle as orc
        data, types, _ = synth.make_data(sets, 500, 5, 5)
        hy = synth.make_hypers(3, 20, 500, 5)
        o = orc.Oracle(data, types, 20, 256)
        rng = np.random.default_rng(5)
        s = o.sweep(hy["s"], rng.permutation(500) + 1, 125, hy["Pi"], hy["phi"], mode=orc.MODE_DEDUP, seed=9, it=0)["s"]
        t0 = time.perf_counter()
        o.sweep(s, rng.permutation(500) + 1, 125, hy["Pi"], hy["phi"], mode=orc.MODE_DEDUP | orc.MODE_LITERAL_NEWID,
                seed=9, it=1, logweight_init=1.0)
        emit(dict(workload="omics_reference", impl="oracle C++ de-duplicated literal mode, 1 thread, host CPU",
                  s_per_sweep=round(time.perf_counter() - t0, 2)))
        from pmdi_b200 import pmdi as host
        import tempfile
        with tempfile.TemporaryDirectory() as d:
            iters = int(os.environ.get("TIME_WIDE_ITERS", "20"))
            host.pmdi(data, types, 20, 256, 0.25, 2, os.path.join(d, "w.csv"), featureSelect=os.path.join(d, "f.csv"),
                      seed=1)
            t0 = time.perf_counter()
            host.pmdi(data, types, 20, 256, 0.25, iters, os.path.join(d, "o.csv"), featureSelect=os.path.join(d, "g.csv"),
                      seed=2)
            dt = time.perf_counter() - t0
        emit(dict(workload="omics_pmdi_featureSelect", iterations=iters, seconds=round(dt, 2),
                  iterations_per_s=round(iters / dt, 3)))
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    with open(OUT, "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()

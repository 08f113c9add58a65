#!/usr/bin/env python
"""Cost of a resampling event on the spec engine, one GPU: chained settled sweeps of a BASELINE configuration.
  python scripts/time_resample.py cfg2_multiomics [sweeps] [out.jsonl]
Two measurements, alternated sweep by sweep after a warm-up:
  - the production kernel: kernel ms and resamplings per sweep; a least-squares line kernel_ms = a + b * resamplings
    gives b, the time one event adds to a sweep, and a, a sweep without one;
  - the instrumented kernel (time_phases=True): per event, the sub-phase timers of the resampling
    (phase_ms[4] plan + first barrier, [5] row maps + recount, [7] list rebuild; [6] the whole event as the CTAs
    see it, the P-CTAs' wait for the decision and the undo included), mean over CTAs; each instrumented sweep's line
    also carries all eight timer slots, mean and maximum over CTAs (an instrumented build may time other sub-phases
    in them).
One JSON line per sweep and a summary line; with out.jsonl they are appended there too."""
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pmdi_b200  # noqa: E402,F401
from pmdi_b200 import capi, synth  # noqa: E402

name = sys.argv[1]
sweeps = int(sys.argv[2]) if len(sys.argv) > 2 else 40
out = open(sys.argv[3], "a") if len(sys.argv) > 3 else None
warm = 6


def emit(d):
    line = json.dumps(d)
    print(line, flush=True)
    if out:
        out.write(line + "\n")


cfg = synth.make_config(name)
K = len(cfg["sets"])
hy = synth.make_hypers(K, cfg["N"], cfg["n"], cfg["seed"])
n1 = int(np.floor(cfg["rho"] * cfg["n"]))
steps = cfg["n"] - n1 + 1
rng = np.random.default_rng(1)
prod, inst = [], []
with capi.Context(cfg["data"], cfg["types"], cfg["N"], cfg["P"]) as ctx:
    s = hy["s"]
    for it in range(sweeps):
        timed = it >= warm and (it - warm) % 2 == 1
        r = ctx.sweep(s, rng.permutation(cfg["n"]) + 1, n1, hy["Pi"], hy["phi"], seed=9, it=it,
                      logweight_init=float(it > 0), time_phases=timed)
        s = r["s"]
        row = dict(config=name, sweep=it, instrumented=timed, kernel_ms=round(r["sweep_kernel_ms"], 4),
                   resamples=r["n_resamples"])
        if timed:
            row["phase_ms"] = [round(v, 4) for v in r["phase_ms"]]
            row["phase_ms_max"] = [round(v, 4) for v in r["phase_ms_max"]]
            inst.append(row)
        elif it >= warm:
            prod.append(row)
        emit(row)
x = np.array([p["resamples"] for p in prod], float)
y = np.array([p["kernel_ms"] for p in prod], float)
summ = dict(config=name, P=cfg["P"], N=cfg["N"], steps=steps, sweeps_production=len(prod), resamples_per_sweep=round(float(x.mean()), 2) if len(x) else None)
if len(x) > 2 and x.std() > 0:
    b, a = np.polyfit(x, y, 1)
    summ.update(us_per_event_fit=round(1e3 * b, 1), ms_per_sweep_without_event_fit=round(a, 4))
no_ev = y[x == 0]
if len(no_ev):
    summ["ms_per_sweep_no_resample"] = [round(float(no_ev.mean()), 4), round(float(no_ev.min()), 4), int(len(no_ev))]
summ["ms_per_sweep_mean"] = round(float(y.mean()), 4) if len(y) else None
ev = sum(i["resamples"] for i in inst)
if ev:
    ph = np.sum([i["phase_ms"] for i in inst], axis=0)
    summ["instrumented_events"] = ev
    summ["us_per_event_timers"] = {"plan+barrier": round(1e3 * ph[4] / ev, 1), "rowmaps+recount": round(1e3 * ph[5] / ev, 1),
                                   "list_rebuild": round(1e3 * ph[7] / ev, 1), "event_as_seen_by_ctas": round(1e3 * ph[6] / ev, 1)}
emit(summ)

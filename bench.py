#!/usr/bin/env python
"""Benchmark of the conditional-SMC allocation sweep (BASELINE.json metric) on B200.

One "step" = one full sweep (one MCMC iteration's pass over the n - n1 + 1 remaining observations,
reference src/pmdi.jl:188-350 + :373) of the workload BASELINE.json quotes the metric on
(configs[1]: K=3 synthetic multi-omics, n=500, Gaussian 2000 + Categorical 500 (3 levels) +
NegBinom 1000 features, N=20, 256 particles, rho=0.25).

  python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
  python bench.py --impl reference ...                   # the restated reference on the host CPU
  python bench.py ... --dump-outputs DIR                 # also write the last timed sweep's results as DIR/*.npy

Prints ONE JSON line (contract in the task statement).  Besides the headline workload the line
carries: `parity` (one sweep checked against the oracle before anything is timed - the oracle is
used as the checker only), at N = 1 a `cfg4` block (the 20,000-cell configuration the north-star
puts its targets on: default engine and the dense engine's HBM roofline) and `pmdi_end_to_end`
(MCMC iterations per second through pmdi() with the host-side hyper-parameter updates), at N > 1 a
`cfg4_strong` block (1,024 particles sharded over the N GPUs).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

# Both arms time sweeps of a chain that has left its start-up transient: the reference's cost per
# sweep falls ~40x once the particles coalesce (scripts/diag_cpu_baseline.py: 3-5.6 s for the first
# sweeps from the random initial allocation, ~0.15 s afterwards), and a 1000-iteration run spends
# >99 % of its time in that settled regime.  Burn-in sweeps are set-up, not warm-up steps.
BURN_IN = 8

METRIC = "particle*cluster*feature evals/sec (dense count P*N*sum_k D_k per observation step)"
UNIT = "evals/s"
PHASES = {
    "spec": ["wait_at_barrier", "evaluate(E-CTAs)", "propose+commit(P-CTAs)", "outcome_bookkeeping(E-CTAs)", "-", "-", "resample"],
    "pool": ["wait_at_barrier_B1", "evaluate", "propose", "resolve", "wait_at_barrier_B2", "-", "resample"],
    "dense": ["warp_idle_or_waiting", "items(predictive+fused add)", "proposal+fold+arrive", "-", "-", "-", "resample"],
}
LAUNCHES = {"spec": 7, "pool": 7, "dense": 8}  # kernels per sweep: init, prefix lists/build/aux, (pool init | broadcast+empty), sweep, finish

# algorithmic bytes per predictive term / per feature of an added cluster at the reference's widths
# (SURVEY.md 8(d)) and as stored on the device
READ_B = {0: 16, 1: 8, 2: 8}
ADD_B = {0: 64, 1: 16, 2: 16}
READ_B_STORED = {0: 16, 1: 8, 2: 8}
ADD_B_STORED = {0: 64, 1: 16, 2: 16}


def make_workload(name, seed_shift=0, particles=None, **over):
    import pmdi_b200  # noqa: F401
    from pmdi_b200 import synth
    if particles:
        over["P"] = particles
    cfg = synth.make_config(name, **over)
    K = len(cfg["sets"])
    hy = synth.make_hypers(K, cfg["N"], cfg["n"], cfg["seed"])
    rng = np.random.default_rng(cfg["seed"] + 31 + seed_shift)
    cfg.update(K=K, hy=hy, n1=int(np.floor(cfg["rho"] * cfg["n"])), rng=rng)
    return cfg


def dense_evals_per_sweep(cfg):
    steps = cfg["n"] - cfg["n1"] + 1
    return steps * cfg["P"] * cfg["N"] * sum(d.shape[1] for d in cfg["data"])


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, res):
    """Writes what a caller of the sweep receives (one download) as `out_dir/<name>.npy` in float64, so that two
    builds run with the same arguments can be compared output for output.  An array larger than its share of
    DUMP_BYTES is replaced by a fixed, seeded sample of its flattened elements."""
    arrays = {k: np.asarray(v) for k, v in res.items() if isinstance(v, np.ndarray)}
    arrays["p_star"] = np.array([res["p_star"]])
    arrays["n_resamples"] = np.array([res["n_resamples"]])
    share = DUMP_BYTES // len(arrays) // 8
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.astype(np.float64)
        if a.size > share:
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def common_config(cfg, burn):
    """The keys BOTH arms print under `config` (the driver compares them)."""
    return {"workload": cfg["name"], "n_obs": cfg["n"], "K": cfg["K"], "N": cfg["N"], "particles": cfg["P"],
            "rho": cfg["rho"], "features": [int(d.shape[1]) for d in cfg["data"]],
            "observation_steps_per_sweep": cfg["n"] - cfg["n1"] + 1,
            "chain_state": f"settled: {burn} untimed burn-in sweeps from the random initial allocation",
            "l2": "GPU arm: 160 MiB buffer written between timed sweeps (L2 flush); CPU arm: not applicable"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.index, self.rows, self.proc, self.first = index, [], None, 0

    def mark(self):
        """Samples taken before this call (warm-up) are not reported."""
        self.first = len(self.rows)

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows[self.first:]:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for nm, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle port on the host cores (the one place it is the thing timed)
# --------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's own algorithm on the host CPU: the C++ restatement in its literal,
    de-duplicated form (copy-on-write cluster pool + fprob cache, src/pmdi.jl:131-146,223-310),
    single thread like the Julia code.  Julia itself is not installed (SURVEY.md F2)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    # the same job as the GPU arm at this N: the configuration's particle count per GPU x GPUs
    base = make_workload(args.workload, particles=args.particles)
    cfg = make_workload(args.workload, particles=base["P"] * max(1, args.gpus))
    o = orc.Oracle(cfg["data"], cfg["types"], cfg["N"], cfg["P"])
    hy, n, rng = cfg["hy"], cfg["n"], cfg["rng"]
    mode = orc.MODE_DEDUP | orc.MODE_LITERAL_NEWID
    s = hy["s"]
    times, burn = [], []
    n_burn = BURN_IN
    for it in range(BURN_IN + args.warmup + args.steps):
        if it < n_burn and sum(burn) > 150.0:   # bound the whole run: stop burning in, say so below
            n_burn = it
        if it >= n_burn + args.warmup + args.steps:
            break
        order = rng.permutation(n) + 1
        t0 = time.perf_counter()
        r = o.sweep(s, order, cfg["n1"], hy["Pi"], hy["phi"], mode=mode, seed=cfg["seed"], it=it,
                    logweight_init=0.0 if it == 0 else 1.0)
        dt = time.perf_counter() - t0
        s = r["s"]
        if it < n_burn:
            burn.append(dt)
        elif it >= n_burn + args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, r)
    total = float(np.sum(times))
    dense = dense_evals_per_sweep(cfg)
    val = dense * args.steps / total
    sample = (f"{args.steps} full sweeps of {args.workload} (n={n}, {n - cfg['n1'] + 1} observation steps "
              f"each) after {n_burn} burn-in sweeps, de-duplicated literal mode, g++ -O3, 1 thread")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": common_config(cfg, BURN_IN),
        "detail": {"burn_in_sweeps_run": n_burn, "burn_in_sweep_ms": [round(1e3 * v, 1) for v in burn],
                   "note": "restated reference (C++), not Julia: julia is not installed in this image; "
                           "value counts the DENSE evals the sweep stands for, the reference evaluates "
                           "only unique clusters (calc_logprob calls in last sweep: %d)" % r["n_ops"]},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "mcmc_sweeps_per_s": args.steps / total,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_leg(cfg, budget_s=6.0):
    """Bounded sample of the same workload on the host (rank 0, N=1 only): the same chain state as
    the GPU arm (BURN_IN untimed sweeps), then sweeps until the budget is spent."""
    from oracle import oracle as orc
    o = orc.Oracle(cfg["data"], cfg["types"], cfg["N"], cfg["P"])
    hy, n = cfg["hy"], cfg["n"]
    rng = np.random.default_rng(5)
    mode = orc.MODE_DEDUP | orc.MODE_LITERAL_NEWID
    s, t_tot, k, burn = hy["s"], 0.0, 0, []
    for it in range(BURN_IN):
        t0 = time.perf_counter()
        r = o.sweep(s, rng.permutation(n) + 1, cfg["n1"], hy["Pi"], hy["phi"], mode=mode, seed=3, it=it,
                    logweight_init=0.0 if it == 0 else 1.0)
        burn.append(time.perf_counter() - t0)
        s = r["s"]
    while k < 3 or (t_tot < budget_s and k < 40):
        order = rng.permutation(n) + 1
        t0 = time.perf_counter()
        r = o.sweep(s, order, cfg["n1"], hy["Pi"], hy["phi"], mode=mode, seed=3, it=BURN_IN + k,
                    logweight_init=1.0)
        t_tot += time.perf_counter() - t0
        s = r["s"]
        k += 1
    val = dense_evals_per_sweep(cfg) * k / t_tot
    return {"value": val, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"{k} full sweeps of the same workload ({t_tot:.1f} s) after {BURN_IN} burn-in sweeps "
                      f"({sum(burn):.1f} s), restated reference (C++, de-duplicated literal mode, 1 thread); "
                      f"dense-equivalent evals/s",
            "ms_per_sweep": 1e3 * t_tot / k, "burn_in_sweep_ms": [round(1e3 * v, 1) for v in burn],
            "calc_logprob_calls_last_sweep": r["n_ops"]}


# --------------------------------------------------------------------------------------------------
# this repo's arm
# --------------------------------------------------------------------------------------------------
class Runner:
    """One workload on this rank's GPU (all ranks together when the particles are sharded)."""

    def __init__(self, cfg, world, rank, local, stream, flush, engine=None):
        import torch.distributed as dist
        from pmdi_b200 import capi
        self.cfg, self.world, self.rank, self.flush, self.dist = cfg, world, rank, flush, dist
        old = os.environ.get("PMDI_ENGINE")
        if engine:
            os.environ["PMDI_ENGINE"] = engine
        try:
            self.ctx = capi.Context(cfg["data"], cfg["types"], cfg["N"], cfg["P"], device=local, rank=rank, n_ranks=world)
            if world > 1:
                self.ctx.connect()
            capi._check(capi.lib().pmdi_ctx_set_stream(self.ctx.h, stream.cuda_stream))
            # the engine is fixed when the arena is laid out: force that now, while the variable is set
            self.ctx.upload(cfg["hy"]["s"], np.arange(cfg["n"]) + 1, cfg["n1"], cfg["hy"]["Pi"], cfg["hy"]["phi"])
        finally:
            if engine:
                if old is None:
                    os.environ.pop("PMDI_ENGINE", None)
                else:
                    os.environ["PMDI_ENGINE"] = old
        self.stream = stream
        self.s = cfg["hy"]["s"]
        self.it = 0
        self.engine = None

    def _sync_ranks(self):
        """With several ranks every rank's grid counter must be reset (upload) before any rank's
        kernel starts to arrive on it (include/pmdi_cuda.h)."""
        if self.world > 1 and os.environ.get("PMDI_ENGINE") == "dense":
            self.dist.barrier()

    def chain(self, sweeps, orders, record=None):
        """Untimed sweeps through the same upload -> L2 flush -> run -> download sequence as the timed ones."""
        cfg, hy = self.cfg, self.cfg["hy"]
        for _ in range(sweeps):
            self.ctx.upload(self.s, orders[self.it], cfg["n1"], hy["Pi"], hy["phi"], seed=cfg["seed"], it=self.it,
                            logweight_init=0.0 if self.it == 0 else 1.0)
            self._sync_ranks()
            self.flush.zero_()
            self.ctx.run()
            r = self.ctx.download()
            self.s = r["s"]
            self.engine = r["engine"]
            if record is not None:
                record.append(r["sweep_kernel_ms"])
            self.it += 1

    def timed(self, steps, orders):
        """K sweeps back to back on the device, CUDA events on the launching stream.  Each sweep's inputs
        (allocations, the shuffled order, Pi, Phi: a few KB) are handed to the context right before its run;
        the allocations are those of the chain so far, so there is no device->host read in the region."""
        import torch
        cfg, hy = self.cfg, self.cfg["hy"]
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        ev[0].record(self.stream)
        for t in range(steps):
            self.ctx.upload(self.s, orders[self.it + t], cfg["n1"], hy["Pi"], hy["phi"], seed=cfg["seed"], it=self.it + t,
                            logweight_init=1.0)
            self._sync_ranks()
            self.flush.zero_()
            self.ctx.run()
            ev[t + 1].record(self.stream)
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()
        last = self.ctx.download()
        return ev[0].elapsed_time(ev[steps]), [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)], last

    def per_launch(self, steps, orders):
        """The same sweeps once more, one at a time: kernel time per launch (CUDA events inside the library,
        on the same stream) and the work counters."""
        cfg, hy, K = self.cfg, self.cfg["hy"], self.cfg["K"]
        do = self.ctx.sweep_sharded if self.world > 1 else self.ctx.sweep
        out = dict(kms=[], rows=np.zeros(K), rows_computed=np.zeros(K), resamples=0, copies=0, evals=0, remote=0,
                   rows_ref=np.zeros(K), rows_added=np.zeros(K))
        r = None
        for t in range(steps):
            self.flush.zero_()
            r = do(self.s, orders[self.it + t], cfg["n1"], hy["Pi"], hy["phi"], seed=cfg["seed"], it=self.it + t,
                   logweight_init=1.0, time_phases=(t == steps - 1))
            if t < steps - 1:  # the last launch runs the instrumented kernel (phase timers): not a kernel time
                out["kms"].append(r["sweep_kernel_ms"])
            out["rows"] += np.array(r["rows_evaluated"][:K], dtype=float)
            out["rows_computed"] += np.array(r["rows_computed"][:K], dtype=float)
            out["rows_ref"] += np.array(r["rows_referenced"][:K], dtype=float)
            out["rows_added"] += np.array(r["rows_added"][:K], dtype=float)
            out["resamples"] += r["n_resamples"]
            out["copies"] += r["n_copies"]
            out["evals"] += r["n_evals"]
            out["remote"] += r["n_remote_rows"]
        out["phase_ms"], out["phase_ms_max"], out["engine"] = r["phase_ms"], r["phase_ms_max"], r["engine"]
        return out

    def e2e(self, steps, orders):
        """End to end through pmdi_sweep() with host buffers, allocations chained sweep to sweep."""
        import torch
        cfg, hy = self.cfg, self.cfg["hy"]
        do = self.ctx.sweep_sharded if self.world > 1 else self.ctx.sweep
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        s2 = self.s
        for t in range(steps):
            r2 = do(s2, orders[self.it + t], cfg["n1"], hy["Pi"], hy["phi"], seed=cfg["seed"], it=self.it + t,
                    logweight_init=1.0)
            s2 = r2["s"]
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    def close(self):
        self.ctx.close()


def roofline(cfg, pl, steps, k_ms, world, peak, peak_src, traffic, engine):
    """HBM roofline of the sweep kernel by ALGORITHMIC bytes: what the reference's own algorithm has to
    move - every distinct cluster's predictive once per observation (16|8|8 B per feature at the
    reference's widths) and the add of every chosen cluster (64|16|16 B per feature, read + write)."""
    K, types = cfg["K"], cfg["types"]
    D = [int(d.shape[1]) for d in cfg["data"]]
    steps_obs = cfg["n"] - cfg["n1"] + 1
    # adds: dense - one per (particle, dataset) and step; copy-on-write - one per DISTINCT chosen cluster and step.
    # A row that is added and evaluated in one pass is charged the add only (64 B per feature, not 64 + 16).
    rows, adds = pl["rows"] / steps, pl["rows_added"] / steps
    alg = sum((rows[k] - min(rows[k], adds[k])) * D[k] * READ_B[types[k]] + adds[k] * D[k] * ADD_B[types[k]] for k in range(K))
    alg_unfused = sum(rows[k] * D[k] * READ_B[types[k]] + adds[k] * D[k] * ADD_B[types[k]] for k in range(K))
    moved = None
    if engine == "spec":  # what this engine really reads and writes: every live row and its child, every step
        moved = sum(pl["rows_computed"][k] / steps / 2.0 * D[k] * ADD_B_STORED[types[k]] for k in range(K))
    achieved = alg / (k_ms * 1e-3) / 1e9
    out = {
        "bound": "hbm", "kernel": {"spec": "k_sweep_spec", "pool": "k_sweep_pool", "dense": "k_sweep"}[engine] +
                                  " (persistent, one launch per sweep)" + ("" if world == 1 else "; rank 0's launch and particles"),
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
        "traffic": traffic, "algorithmic_bytes_per_launch": alg, "kernel_ms": k_ms,
        "achieved_if_add_and_eval_counted_separately": alg_unfused / (k_ms * 1e-3) / 1e9,
        "us_per_observation_step": 1e3 * k_ms / steps_obs,
    }
    if moved is not None:
        out["device_bytes_model_per_launch"] = moved
    if engine != "dense":
        out["note"] = ("the copy-on-write engines evaluate each DISTINCT cluster once per observation, as the reference does: "
                       "the bytes are ~1e2-1e3 x fewer than the dense form's and the sweep is a chain of dependent per-"
                       "observation phases bound by latency (us_per_observation_step), not by HBM; `frac` is reported because "
                       "the contract asks for it - the dense engine's figure, where the HBM roofline is the binding one, is "
                       "under cfg4.dense_engine")
    return out


def parity_block(cfg_name, world, rank, local, stream, flush, particles=None, **over):
    """One sweep of the workload checked against the oracle (the checker, never the thing measured):
    allocations, selected particle, resampling count bit-exact, log-weights to 1e-5."""
    import fullsize
    cfg = make_workload(cfg_name, particles=particles, **over)
    cfg.update(chain=0, debug=False)
    run = Runner(cfg, world, rank, local, stream, flush)
    hy = cfg["hy"]

    def sweep_fn(s, order, it, lw0, debug):
        do = run.ctx.sweep_sharded if world > 1 else run.ctx.sweep
        return do(s, order, cfg["n1"], hy["Pi"], hy["phi"], seed=77, it=it, logweight_init=lw0)
    if rank == 0:
        out = fullsize.compare(cfg, sweep_fn)
        ok = (out["s_mismatch"] == 0 and out["p_star_equal"] and out["n_resamples"][0] == out["n_resamples"][1]
              and out["logweight_max_rel"] <= 1e-5)
        res = {"checked": f"one sweep of {cfg_name} (P={cfg['P']}, n={cfg['n']}) from the random initial allocation vs the "
                          "oracle's de-duplicated corrected mode", "ok": bool(ok),
               "allocation_mismatches": out["s_mismatch"], "draws": out["draws"], "p_star_equal": out["p_star_equal"],
               "n_resamples_gpu_vs_oracle": out["n_resamples"], "logweight_max_rel": out["logweight_max_rel"],
               "cluster_size_mismatches": out.get("cluster_n_mismatch"), "oracle_s": out["oracle_s"]}
    else:  # the other ranks run the same sweep (same arguments), rank 0 checks
        rng = np.random.default_rng(77)
        order = rng.permutation(cfg["n"]) + 1
        sweep_fn(hy["s"], order, 0, 0.0, False)
        res = None
    run.close()
    return res


def run_ours(args):
    import torch
    import torch.distributed as dist
    import pmdi_b200  # noqa: F401
    from pmdi_b200 import capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available() or capi.device_count() < 1:
        raise RuntimeError("bench.py needs a CUDA device: the sweep has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    stream = torch.cuda.current_stream()
    flush = torch.empty(160 << 20, dtype=torch.uint8, device="cuda")  # 168 MB > 126 MB L2
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    traffic_db = []
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic_db = tj if isinstance(tj, list) else [tj]

    def traffic_for(workload, P, engine):
        for e in traffic_db:
            if e.get("workload") == workload and e.get("particles") == P and e.get("engine", "dense") == engine and world == 1:
                return e.get("dram_bytes_per_launch")
        return None

    # ---------------------------------------------------------------- parity first (checker only)
    parity = None if args.no_parity else parity_block(
        args.workload, world, rank, local, stream, flush,
        particles=(args.particles or make_workload(args.workload)["P"]) * world)

    # ---------------------------------------------------------------- the headline workload
    # Particles are sharded over the GPUs (SURVEY 8e): weak scaling = the configuration's particle
    # count PER GPU, so the job has P * world particles; every rank passes identical arguments.
    base = make_workload(args.workload, particles=args.particles)
    cfg = make_workload(args.workload, particles=base["P"] * world)
    n, K, N, P = cfg["n"], cfg["K"], cfg["N"], cfg["P"]
    rng = cfg["rng"]
    orders = [rng.permutation(n) + 1 for _ in range(BURN_IN + args.warmup + 3 * args.steps + 2)]
    run = Runner(cfg, world, rank, local, stream, flush)
    # the clock sampler starts BEFORE the warm-up: nvidia-smi's NVML start-up stalls launches on the
    # device for a while and must not land inside the timed region; it keeps sampling through it
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(1.5)
    burn_ms = []
    run.chain(BURN_IN, orders, burn_ms)
    run.chain(args.warmup, orders)   # warm-up = the SAME step as the timed one
    if rank == 0:
        sampler.mark()
    dev_ms, step_ms, last = run.timed(args.steps, orders)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    pl = run.per_launch(args.steps, orders)
    e2e_s = run.e2e(args.steps, orders)
    run.close()

    dense = dense_evals_per_sweep(cfg)
    t_dev = torch.tensor([dev_ms, e2e_s * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = float(t_dev[0]), float(t_dev[1])
    value = dense * args.steps / (dev_ms * 1e-3)       # `dense` already counts the whole job
    e2e_val = dense * args.steps / (e2e_ms * 1e-3)
    evals_t = torch.tensor([float(pl["evals"]), float(pl["remote"])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(evals_t, op=dist.ReduceOp.SUM)
    evals, remote_rows = float(evals_t[0]), float(evals_t[1])

    # ---------------------------------------------------------------- the other blocks
    cfg4 = cfg4_block(world, rank, local, stream, flush, peak, peak_src, traffic_for) if not args.no_cfg4 else None
    pmdi_e2e = pmdi_block(local) if (world == 1 and rank == 0 and not args.no_pmdi) else None

    if rank == 0:
        engine = pl["engine"]
        k_ms = float(np.mean(pl["kms"]))
        h2d = n * K * 8 + n * 8 + N * K * 8 + max(1, K * (K - 1) // 2) * 8
        d2h = n * K * 8 + P * 8 + K * P * N * 8 + N * K * 8 + max(1, K * (K - 1) // 2) * 8 + 8 + 4 + 64 * 6
        roof = roofline(cfg, pl, args.steps, k_ms, world, peak, peak_src, traffic_for(args.workload, P, engine), engine)
        roof["kernel_share_of_step"] = k_ms / (dev_ms / args.steps)
        roof["warp_ms_mean_over_ctas"] = dict(zip(PHASES[engine], [round(v, 3) for v in pl["phase_ms"][:7]]))
        roof["warp_ms_max_over_ctas"] = dict(zip(PHASES[engine], [round(v, 3) for v in pl["phase_ms_max"][:7]]))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": common_config(cfg, BURN_IN),
            "detail": {
                "engine": engine,
                "step": "one full conditional-SMC sweep (prefix build, per-observation loop, selection)",
                "burn_in_kernel_ms": [round(v, 2) for v in burn_ms],
                "parallelism": "single GPU" if world == 1 else
                               f"one chain, {P} particles sharded over {world} GPUs ({P // world} per GPU): every rank keeps its own "
                               "copy-on-write pool; per observation one ESS partial per rank is pushed to the peers (NVLink stores, "
                               "off the dependent chain), allocations go to every rank's log; resampled ancestors held by another "
                               "rank have their rows pulled through peer memory (each remote row once); no NCCL call and no host "
                               "barrier in the data path",
                "particles_per_gpu": P // world,
                "rows_pulled_from_peers_per_sweep": remote_rows / args.steps,
                "distinct_clusters_evaluated_per_sweep": float(pl["rows"].sum()) / args.steps,
                "row_evaluations_computed_per_sweep": float(pl["rows_computed"].sum()) / args.steps,
                "occupied_particle_clusters_referenced_per_sweep": float(pl["rows_ref"].sum()) / args.steps,
                "evals_performed_frac": evals / (dense * args.steps),
                "resamples_per_sweep": pl["resamples"] / args.steps,
            },
            "mcmc_sweeps_per_s": args.steps / (dev_ms * 1e-3),
            "ms_per_timed_step": [round(v, 3) for v in step_ms],
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / args.steps,
                    "path": "pmdi_sweep() C-ABI call with host buffers, allocations chained sweep to sweep"},
            "gpu_launches": LAUNCHES[engine] * args.steps,
            "roofline": roof,
            "parity": parity,
        }
        if cfg4 is not None:
            line["cfg4" if world == 1 else "cfg4_strong"] = cfg4
        if pmdi_e2e is not None:
            line["pmdi_end_to_end"] = pmdi_e2e
        line["cpu_baseline"] = cpu_baseline_leg(cfg) if (world == 1 and not args.no_cpu) else None
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def cfg4_block(world, rank, local, stream, flush, peak, peak_src, traffic_for, steps=3, burn=3):
    """configs[3]: 20,000 cells x 2,000 genes x 2, N=50, 1,024 particles - the configuration the north-star puts
    its 60 %-of-HBM target on.  N = 1: the default engine, and the dense engine whose regime the HBM roofline
    describes.  N > 1: the 1,024 particles sharded over the N GPUs (strong scaling)."""
    cfg = make_workload("cfg4_singlecell")
    rng = np.random.default_rng(4)
    orders = [rng.permutation(cfg["n"]) + 1 for _ in range(burn + 2 * steps + 4)]
    out = {"config": common_config(cfg, burn), "scaling": "strong" if world > 1 else None}
    run = Runner(cfg, world, rank, local, stream, flush)
    burn_ms = []
    run.chain(burn, orders, burn_ms)
    dev_ms, step_ms, _ = run.timed(steps, orders)
    pl = run.per_launch(steps, orders)
    run.close()
    k_ms = float(np.mean(pl["kms"]))
    engine = pl["engine"]
    out.update({"engine": engine, "ms_per_sweep": dev_ms / steps, "ms_per_timed_sweep": [round(v, 2) for v in step_ms],
                "value": dense_evals_per_sweep(cfg) * steps / (dev_ms * 1e-3), "unit": UNIT,
                "burn_in_kernel_ms": [round(v, 1) for v in burn_ms],
                "distinct_clusters_evaluated_per_sweep": float(pl["rows"].sum()) / steps,
                "particles_per_gpu": cfg["P"] // world,
                "roofline": roofline(cfg, pl, steps, k_ms, world, peak, peak_src,
                                     traffic_for("cfg4_singlecell", cfg["P"], engine), engine)})
    if world == 1:
        d = Runner(cfg, 1, 0, local, stream, flush, engine="dense")
        d.s, d.it = run.s, run.it   # the same chain state
        dsteps = 2
        d.chain(1, orders)
        ddev, dstep, _ = d.timed(dsteps, orders)
        dpl = d.per_launch(dsteps + 1, orders)
        d.close()
        dk = float(np.mean(dpl["kms"]))
        roof = roofline(cfg, dpl, dsteps + 1, dk, 1, peak, peak_src, traffic_for("cfg4_singlecell", cfg["P"], "dense"), "dense")
        if roof["traffic"]:
            roof["frac_by_measured_dram_traffic"] = roof["traffic"] / (dk * 1e-3) / 1e9 / peak
        out["dense_engine"] = {"ms_per_sweep": ddev / dsteps, "ms_per_timed_sweep": [round(v, 1) for v in dstep],
                               "rows_evaluated_per_sweep": float(dpl["rows"].sum()) / (dsteps + 1), "roofline": roof,
                               "note": "PMDI_ENGINE=dense: every particle owns its N clusters per dataset (the form the HBM "
                                       "roofline describes); the default engine does the same sweep, same results, in "
                                       f"{dev_ms / steps:.0f} ms"}
    if world > 1:
        import torch
        import torch.distributed as dist
        t = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out["ms_per_sweep"] = float(t[0]) / steps
        out["value"] = dense_evals_per_sweep(cfg) * steps / (float(t[0]) * 1e-3)
    return out if rank == 0 else None


def pmdi_block(local):
    """MCMC iterations per second through pmdi() - the sweep on the GPU plus the host-side hyper-parameter
    updates, align_labels! and the CSV writer (src/pmdi.jl:164-384).  cfg3 runs with featureSelect on
    (calc_logmarginal!, src/pmdi.jl:354-370) and needs the factorised normalising sums (N^K = 7.3e8)."""
    from pmdi_b200 import pmdi as host
    out = {}
    for name, iters, fs in (("cfg1_iris", 12, False), ("cfg2_multiomics", 12, False), ("cfg3_tcga", 5, True),
                            ("cfg4_singlecell", 3, False)):
        cfg = make_workload(name)
        with tempfile.TemporaryDirectory() as td:
            t0 = time.perf_counter()
            st = host.pmdi(cfg["data"], cfg["types"], cfg["N"], cfg["P"], cfg["rho"], iters, os.path.join(td, "out.csv"),
                           featureSelect=os.path.join(td, "fs.csv") if fs else None, seed=1, device=local)
            dt = time.perf_counter() - t0
        out[name] = {"iterations": iters, "mcmc_iters_per_s": iters / st["loop_s"], "ms_per_iteration": 1e3 * st["loop_s"] / iters,
                     "sweep_device_ms_per_iteration": st["sweep_device_ms"] / iters, "feature_select": fs,
                     "setup_s": st["setup_s"], "total_s": dt,
                     "note": "the first iterations of a fresh chain (the expensive regime); setup_s = data to the device and "
                             "allocation of the row pool, once per run"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2_multiomics")
    ap.add_argument("--particles", type=int, default=None)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-cfg4", action="store_true", help="skip the cfg4 block")
    ap.add_argument("--no-pmdi", action="store_true", help="skip the pmdi() end-to-end block")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity check against the oracle")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed sweep as DIR/<name>.npy")
    args = ap.parse_args()
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

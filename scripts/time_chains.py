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

--user-types: the same on cfg2 with its Gaussian and NegBinom datasets as user-defined cluster types
(tests/multi_user_types.py, the plan of scripts/time_user_types.py), Categorical built-in, at C = 1, 2, 4, 8 with three
arms alternated round by round: sequential on the pool engine (the one-GPU default for user types), sequential on the
spec engine, and the group (spec).  Then pmdi() with those types at chains = 1 (pool) and 4, and the NVRTC seconds of
the group program.
  python scripts/time_chains.py [--user-types] [rounds=10] [out.jsonl]"""
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import pmdi_b200  # noqa: E402,F401
from pmdi_b200 import capi, synth  # noqa: E402
from pmdi_b200.pmdi import pmdi  # noqa: E402

BURN_IN = 8
PLAN = [("cfg1_iris", (1, 2, 4, 8)), ("cfg2_multiomics", (1, 2, 4, 8)), ("cfg4_singlecell", (2,))]
PMDI_PLAN = [("cfg1_iris", 60), ("cfg2_multiomics", 20)]
USER_PLAN = [("cfg2_multiomics", (1, 2, 4, 8))]
USER_PMDI_PLAN = [("cfg2_multiomics", 20)]


def user_types(cfg):
    """cfg2's types with the Gaussian and the NegBinom dataset as user types (registered in this process)."""
    import multi_user_types as mu
    tg, tn = mu.register(capi)
    return [tg if t == capi.GAUSSIAN else tn if t == capi.NEGBINOM else t for t in cfg["types"]]


class Chain:
    """One context and its chain of sweeps (split form, so that a group can run it)."""

    def __init__(self, cfg, hy, n1, seed, types=None, engine=None):
        self.cfg, self.hy, self.n1, self.seed = cfg, hy, n1, seed
        self.ctx = capi.Context(cfg["data"], types or cfg["types"], cfg["N"], cfg["P"], engine=engine)
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


def measure(name, C, rounds, user=False):
    """Built-in types: the arms "sequential" and "group".  user=True: user types, the arms "sequential_pool",
    "sequential_spec" and "group"."""
    cfg = synth.make_config(name)
    K = len(cfg["sets"])
    hy = synth.make_hypers(K, cfg["N"], cfg["n"], cfg["seed"])
    n1 = int(np.floor(cfg["rho"] * cfg["n"]))
    steps = cfg["n"] - n1 + 1
    types = user_types(cfg) if user else None
    seq_arms = {"sequential_pool": None, "sequential_spec": "spec"} if user else {"sequential": None}
    seqs = {arm: [Chain(cfg, hy, n1, 100 + c, types, eng) for c in range(C)] for arm, eng in seq_arms.items()}
    grouped = [Chain(cfg, hy, n1, 100 + c, types, "spec" if user else None) for c in range(C)]
    grp = capi.Group([ch.ctx for ch in grouped])
    try:
        engines = {}
        for _ in range(BURN_IN):
            for arm, seq in seqs.items():
                engines[arm] = seq_round(seq)[2][0]["engine"]
            engines["group"] = group_round(grouped, grp)[2][0]["engine"]
        res = {**{arm: [] for arm in seqs}, "group": []}
        for _ in range(rounds):  # alternate the arms round by round
            for arm, seq in seqs.items():
                res[arm].append(seq_round(seq)[:2])
            res["group"].append(group_round(grouped, grp)[:2])
        # same seeds, same chains: the group and the sequential arm of its engine must have computed the same allocations
        seq = seqs["sequential_spec" if user else "sequential"]
        same = all(np.array_equal(a.s, b.s) for a, b in zip(seq, grouped))
        out = dict(config=name, chains=C, steps=steps, burn_in=BURN_IN, rounds=rounds, same_allocations=same)
        if user:
            out["user_types"] = True
            out["engines"] = engines
            out["pool_same_allocations_as_spec"] = all(
                np.array_equal(a.s, b.s) for a, b in zip(seqs["sequential_pool"], seq))
        for arm, v in res.items():
            wall, ker = np.array([x[0] for x in v]), np.array([x[1] for x in v])
            out[arm] = dict(
                sweeps_per_s_wall=round(C / float(np.median(wall)), 2),
                sweeps_per_s_kernel=round(C / (1e-3 * float(np.median(ker))), 2),
                round_ms_median=round(1e3 * float(np.median(wall)), 3),
                kernel_ms_median=round(float(np.median(ker)), 3),
                us_per_step_per_chain=round(1e3 * float(np.median(ker)) / (steps * (C if arm != "group" else 1)), 2))
        for arm in seqs:
            out[f"group_over_{arm}_wall"] = round(out["group"]["sweeps_per_s_wall"] / out[arm]["sweeps_per_s_wall"], 3)
        return out
    finally:
        grp.close()
        for ch in [ch for seq in seqs.values() for ch in seq] + grouped:
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


def pmdi_rate(name, iters, C, td, user=False):
    cfg = synth.make_config(name)
    outs = [os.path.join(td, f"{name}_{C}_{c}.csv") for c in range(C)]
    st = pmdi(cfg["data"], user_types(cfg) if user else cfg["types"], cfg["N"], cfg["P"], cfg["rho"], iters,
              outs if C > 1 else outs[0], seed=5, chains=C)
    st = st if C > 1 else [st]
    loop = max(s["loop_s"] for s in st)
    return dict(config=name, **(dict(user_types=True) if user else {}), pmdi_chains=C, iterations=iters,
                loop_s=round(loop, 3),
                aggregate_iters_per_s=round(C * iters / loop, 2),
                sweep_device_ms_per_iteration=round(float(np.mean([s["sweep_device_ms"] / iters for s in st])), 3))


def group_compile_seconds(name):
    """NVRTC seconds of the group program of the user types (a fresh compile: nothing of it is cached yet)."""
    from time_user_types import nvrtc_log
    cfg = synth.make_config(name)
    _, log = nvrtc_log(lambda: capi.group_type_check([t for t in user_types(cfg) if t >= 16]))
    return [dict(types=t, program=e, seconds=s) for t, e, s in log]


def main():
    argv = sys.argv[1:]
    user = "--user-types" in argv
    argv = [a for a in argv if a != "--user-types"]
    rounds = int(argv[0]) if len(argv) > 0 else 10
    out_path = argv[1] if len(argv) > 1 else None
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

    if user:
        for name, _ in USER_PLAN:
            emit(dict(config=name, user_types=True, nvrtc=group_compile_seconds(name)))
    for name, cs in (USER_PLAN if user else PLAN):
        for C in cs:
            try:
                d = measure(name, C, rounds if name != "cfg4_singlecell" else max(3, rounds // 2), user)
                d["ctas_per_chain"] = grid_of(name, C, n_sm)
            except capi.PmdiError as e:  # e.g. cfg4's pools of 2 x 2 chains do not fit the GPU's memory
                d = dict(config=name, chains=C, measured=False, reason=str(e)[:300])
            emit(d)
    with tempfile.TemporaryDirectory() as td:
        for name, iters in (USER_PMDI_PLAN if user else PMDI_PLAN):
            for C in (1, 4):
                emit(pmdi_rate(name, iters, C, td, user))


if __name__ == "__main__":
    main()

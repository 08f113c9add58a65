#!/usr/bin/env python
"""Cost of user-defined cluster types against the built-in ones, on the cfg2 shape (Gaussian 2000 + Categorical 500 +
NegBinom 1000 features, n=500, N=20, P=256).  Arms, timed alternately in one process on settled chains (8 untimed
burn-in sweeps each, as bench.py):
  builtin        the built-in types, default engine (spec for K = 3)
  builtin_pool   the built-in types, PMDI_ENGINE=pool
  user_pool      Gaussian and NegBinom as user types (tests/multi_user_types.py), Categorical built-in, pool engine
  user_spec      the same, spec engine
  user_sharded   the same, particles sharded over every GPU of the node (default engine), when there are >= 2
Prints one JSON line per arm (ms per sweep: device events around the sweep's kernels, and host wall time of
ctx.sweep), the NVRTC seconds of each user-type program, and the device name and power limit.
  python scripts/time_user_types.py [sweeps=20] [out.json]"""
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import pmdi_b200  # noqa: E402,F401
from pmdi_b200 import capi, synth  # noqa: E402

import multi_user_types as mu  # noqa: E402

BURN_IN = 8
CFG = "cfg2_multiomics"


def problem():
    cfg = synth.make_config(CFG)
    K = len(cfg["sets"])
    hy = synth.make_hypers(K, cfg["N"], cfg["n"], cfg["seed"])
    return cfg, hy, int(np.floor(cfg["rho"] * cfg["n"]))


class Chain:
    """One context and its chain of sweeps."""

    def __init__(self, cfg, hy, n1, types, engine, device=0, rank=0, world=1):
        self.cfg, self.hy, self.n1 = cfg, hy, n1
        if engine:
            os.environ["PMDI_ENGINE"] = engine
        else:
            os.environ.pop("PMDI_ENGINE", None)
        self.ctx = capi.Context(cfg["data"], types, cfg["N"], cfg["P"], device=device, rank=rank, n_ranks=world)
        if world > 1:
            self.ctx.connect()
        self.rng = np.random.default_rng(1)
        self.s, self.it = hy["s"], 0
        self.setup_s = self.step()[2]  # the engine is fixed when the context is first prepared
        os.environ.pop("PMDI_ENGINE", None)
        self.engine = self.last["engine"]

    def step(self):
        t = time.perf_counter()
        r = self.ctx.sweep(self.s, self.rng.permutation(self.cfg["n"]) + 1, self.n1, self.hy["Pi"], self.hy["phi"],
                           seed=9, it=self.it, logweight_init=float(self.it > 0), cluster_sizes=False)
        wall = time.perf_counter() - t
        self.s, self.it, self.last = r["s"], self.it + 1, r
        return r["device_ms"], r["sweep_kernel_ms"], wall


def nvrtc_log(fn):
    """Runs fn() with the library's compile log (stderr) captured: (fn's result, [(types, engine, seconds)])."""
    os.environ["PMDI_JIT_LOG"] = "1"
    with tempfile.TemporaryFile(mode="w+") as f:
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            out = fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            os.environ.pop("PMDI_JIT_LOG", None)
        f.seek(0)
        text = f.read()
    sys.stderr.write(text)
    return out, [(m.group(1), m.group(2), float(m.group(3)))
                 for m in re.finditer(r"nvrtc compiled (.*) for the ([\w-]+) engine in ([0-9.]+) s", text)]


def summary(name, chain, dev, ker, wall, extra=None):
    d = dict(arm=name, engine=chain.engine, sweeps=len(dev), device_ms_median=round(float(np.median(dev)), 3),
             device_ms_min=round(float(np.min(dev)), 3), kernel_ms_median=round(float(np.median(ker)), 3),
             wall_ms_median=round(1e3 * float(np.median(wall)), 3), setup_s=round(chain.setup_s, 2),
             resamples_last=chain.last["n_resamples"])
    d.update(extra or {})
    return d


def sharded_rank(rank, world, port, sweeps, out_dir):
    """One rank of the user_sharded arm."""
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        cfg, hy, n1 = problem()
        tg, tn = mu.register(capi)
        ch = Chain(cfg, hy, n1, [tg, cfg["types"][1], tn], None, device=rank, rank=rank, world=world)
        for _ in range(BURN_IN - 1):
            ch.step()
        dev, ker, wall = zip(*[ch.step() for _ in range(sweeps)])
        if rank == 0:
            with open(os.path.join(out_dir, "sharded.json"), "w") as f:
                json.dump(summary("user_sharded", ch, dev, ker, wall, dict(ranks=world)), f)
        dist.barrier()
        ch.ctx.close()
    finally:
        dist.destroy_process_group()


def main():
    sweeps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    out_path = sys.argv[2] if len(sys.argv) > 2 else None
    if capi.device_count() < 1:
        raise SystemExit("time_user_types.py needs a CUDA device")
    import torch
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    head = dict(config=CFG, device=torch.cuda.get_device_name(0), nvidia_smi=smi[:1], gpus=capi.device_count(),
                burn_in=BURN_IN, timed_sweeps_per_arm=sweeps)
    cfg, hy, n1 = problem()
    tg, tn = mu.register(capi)
    user = [tg, cfg["types"][1], tn]
    arms, compiles = {}, []
    arms["builtin"] = Chain(cfg, hy, n1, cfg["types"], None)
    arms["builtin_pool"] = Chain(cfg, hy, n1, cfg["types"], "pool")
    for eng in ("pool", "spec"):
        arms[f"user_{eng}"], log = nvrtc_log(lambda: Chain(cfg, hy, n1, user, eng))
        compiles += log
    head["nvrtc"] = [dict(types=t, engine=e, seconds=s) for t, e, s in compiles]
    print(json.dumps(head), flush=True)
    for ch in arms.values():
        for _ in range(BURN_IN - 1):
            ch.step()
    res = {k: [] for k in arms}
    for _ in range(sweeps):  # alternate the arms sweep by sweep
        for k, ch in arms.items():
            res[k].append(ch.step())
    lines = [head]
    for k, ch in arms.items():
        dev, ker, wall = zip(*res[k])
        lines.append(summary(k, ch, dev, ker, wall))
        print(json.dumps(lines[-1]), flush=True)
        ch.ctx.close()
    world = capi.device_count()
    if world >= 2:
        import socket
        import torch.multiprocessing as mp
        with socket.socket() as so:
            so.bind(("127.0.0.1", 0))
            port = so.getsockname()[1]
        with tempfile.TemporaryDirectory() as td:
            mp.spawn(sharded_rank, args=(world, port, sweeps, td), nprocs=world, join=True)
            lines.append(json.load(open(os.path.join(td, "sharded.json"))))
    else:
        lines.append(dict(arm="user_sharded", measured=False, reason="one GPU"))
    print(json.dumps(lines[-1]), flush=True)
    if out_path:
        with open(out_path, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()

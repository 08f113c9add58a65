"""Several user-defined cluster types in one context: the sources the tests register, and the spawn target of the
sharded tests (a module-level function, so that torch.multiprocessing can pickle it).

USER_NEGBINOM restates the reference's NegBinomCluster (src/datatypes/negbinom_cluster.jl:9-60, the oracle's
calc_logprob / calc_logmarginal) feature by feature: one word of state, the sum of the counts.  GAUSSIAN_CLUSTER and
NEGBINOM_CLUSTER are the user Gaussian of user_types.py and USER_NEGBINOM with their structs both named `Cluster`:
they can only share a program if every source lives in a namespace of its own."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import user_types as ut  # noqa: E402

USER_NEGBINOM = r"""
struct MyNegBinom {
  static constexpr int WORDS = 1;  // sum of the counts
  __device__ static void init(double* st) { st[0] = 0.0; }
  __device__ static double logprob(const double* st, int n, double x) {
    const double nn = (double)n, S = st[0];
    return lgamma(1 + nn + 1) + lgamma(1 + x + S) + lgamma(1 + nn + 1 + S) - lgamma(1 + nn + 1 + 1 + x + S)
         - lgamma(1 + nn) - lgamma(1 + S);
  }
  __device__ static void add(double* st, int n, double x) { st[0] += x; }
  __device__ static double logmarginal(const double* st, int n) {
    const double nn = (double)n, S = st[0];
    return lgamma(S + 1) - lgamma(S + (nn + 1 + 1)) + lgamma(1 + nn);
  }
};
"""

GAUSSIAN_CLUSTER = ut.USER_GAUSSIAN.replace("MyGaussian", "Cluster")
NEGBINOM_CLUSTER = USER_NEGBINOM.replace("MyNegBinom", "Cluster")

# the first "WORDS =" of the text (a comment) says 1; the struct keeps 2 doubles per feature
WORDS_MISMATCH = r"""
struct TwoWords {   // WORDS = 1 was enough for the first draft
  static constexpr int WORDS = 2;
  __device__ static void init(double* st) { st[0] = 0.0; st[1] = 0.0; }
  __device__ static double logprob(const double* st, int n, double x) { return -0.5 * (x - st[1]) * (x - st[1]); }
  __device__ static void add(double* st, int n, double x) { st[0] += x; st[1] = st[0] / n; }
  __device__ static double logmarginal(const double* st, int n) { return 0.0; }
};
"""


# a problem on which resampling duplicates particles across ranks (tests/test_gpu_sharded.py, "gauss_manyP")
MANY_P = dict(sets=[(0, 64, 0), (2, 33, 0)], n=64, N=5, P=600)
MANY_P_SEED = 4


def register(capi, named_cluster=False):
    """(Gaussian tag, NegBinom tag) of the user restatements of the built-in types."""
    if named_cluster:
        return (capi.register_cluster_type("GaussianCluster_u", GAUSSIAN_CLUSTER, "Cluster", capi.F64),
                capi.register_cluster_type("NegBinomCluster_u", NEGBINOM_CLUSTER, "Cluster", capi.I64))
    return (capi.register_cluster_type("MyGaussian", ut.USER_GAUSSIAN, "MyGaussian", capi.F64),
            capi.register_cluster_type("MyNegBinom", USER_NEGBINOM, "MyNegBinom", capi.I64))


def sharded_user_sweep(rank, world, port, engine, out_dir):
    """One rank of a [user Gaussian, user NegBinom] context with the particles sharded over `world` GPUs; writes its
    sweep's debug outputs to out_dir/rank<r>.npz."""
    import torch
    import torch.distributed as dist
    os.environ["PMDI_ENGINE"] = engine
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import pmdi_b200  # noqa: F401
        from pmdi_b200 import capi
        from helpers import problem
        pr = problem(**MANY_P, seed=MANY_P_SEED)
        tags = register(capi)
        ctx = capi.Context(pr["data"], list(tags), pr["N"], pr["P"], device=rank, rank=rank, n_ranks=world)
        ctx.connect()
        r = ctx.sweep_sharded(pr["s"], pr["order"], pr["n1"], pr["Pi"], pr["phi"], seed=11, it=3, debug=True)
        ctx.close()
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), alloc=r["alloc"], anc=r["anc"], lw=r["lw"], s=r["s"],
                 p_star=r["p_star"], n_remote_rows=r["n_remote_rows"], n_resamples=r["n_resamples"],
                 engine=r["engine"])
    finally:
        dist.destroy_process_group()


def planted(n=90, seed=0):
    """Counts and continuous data with the same three planted clusters: (counts, expr, z)."""
    rng = np.random.default_rng(seed)
    z = np.arange(n) % 3
    counts = rng.poisson(np.array([0.5, 8.0, 60.0])[z][:, None] * np.ones((n, 30))).astype(np.int64)
    expr = rng.normal(size=(n, 20)) + 4.0 * np.array([-1.0, 0.0, 1.0])[z][:, None]
    return counts, expr, z


def pmdi_types():
    """UserCluster objects of a counts type and a continuous type (registered in this process)."""
    from pmdi_b200 import pmdi as host
    return (host.UserCluster("MyPoisson", ut.USER_POISSON, integer_data=True),
            host.UserCluster("MyGaussian", ut.USER_GAUSSIAN))


def pmdi_rank(rank, world, port, out_dir, iters, types):
    """pmdi() with two user types and the particles sharded over `world` GPUs; rank 0 writes out_dir/sharded.csv.
    `types` are UserCluster objects made by the parent process (pickled into this one)."""
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        import pmdi_b200  # noqa: F401
        from pmdi_b200 import pmdi as host
        counts, expr, _ = planted()
        host.pmdi([counts, expr], list(types), 6, 24, 0.25, iters, os.path.join(out_dir, "sharded.csv"), seed=3,
                  device=rank, distributed=True)
        dist.barrier()
    finally:
        dist.destroy_process_group()

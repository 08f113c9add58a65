"""User-defined cluster types with the particles sharded over the GPUs of one node.  A [user Gaussian, user NegBinom]
context must reproduce the oracle's run of the global particle set with the built-in types: allocations of every
step, ancestors, selected particle and final allocations bit-exact on every rank, log-weights to 1e-5, on a problem
whose resamplings pull rows between ranks (the user-type branch of the row pull).  Needs >= 2 GPUs; skipped below."""
import os
import socket

import numpy as np
import pytest

import multi_user_types as mu
from helpers import problem

pytestmark = pytest.mark.gpu
RTOL = 1e-5


def _n_gpus():
    try:
        import pmdi_b200.capi as capi
        return capi.device_count()
    except Exception:
        return 0


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("engine", ["spec", "pool"])
def test_sharded_user_types_match_the_oracle(engine, world, tmp_path):
    if _n_gpus() < world:
        pytest.skip(f"needs {world} GPUs")
    import torch.multiprocessing as mp
    from oracle import oracle as orc
    mp.spawn(mu.sharded_user_sweep, args=(world, _free_port(), engine, str(tmp_path)), nprocs=world, join=True)
    got = [np.load(os.path.join(tmp_path, f"rank{r}.npz")) for r in range(world)]
    pr = problem(**mu.MANY_P, seed=mu.MANY_P_SEED)
    ref = orc.Oracle(pr["data"], pr["types"], pr["N"], pr["P"]).sweep(
        pr["s"], pr["order"], pr["n1"], pr["Pi"], pr["phi"], mode=orc.MODE_DENSE, seed=11, it=3, debug=True)
    for r in range(world):
        assert str(got[r]["engine"]) == engine
        np.testing.assert_array_equal(got[r]["s"], ref["s"], err_msg=f"rank {r}")
        assert int(got[r]["p_star"]) == ref["p_star"]
        np.testing.assert_array_equal(got[r]["anc"], ref["anc"])
        assert int(got[r]["n_resamples"]) == ref["n_resamples"]
    # per-step captures are written by the rank that holds the particle: add the ranks up
    np.testing.assert_array_equal(sum(g["alloc"] for g in got), ref["alloc"])
    np.testing.assert_allclose(sum(g["lw"] for g in got), ref["lw"], rtol=RTOL, atol=1e-9)
    assert sum(int(g["n_remote_rows"]) for g in got) > 0   # rows of user types were pulled from another GPU


def test_pmdi_sharded_with_user_types_equals_one_gpu(tmp_path):
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from pmdi_b200 import pmdi as host
    iters = 8
    types = mu.pmdi_types()
    mp.spawn(mu.pmdi_rank, args=(2, _free_port(), str(tmp_path), iters, types), nprocs=2, join=True)
    counts, expr, _ = mu.planted()
    one = tmp_path / "one.csv"
    host.pmdi([counts, expr], list(types), 6, 24, 0.25, iters, str(one), seed=3)
    a = host.read_allocations(str(tmp_path / "sharded.csv"), 2, len(expr))
    b = host.read_allocations(str(one), 2, len(expr))
    np.testing.assert_array_equal(a, b)

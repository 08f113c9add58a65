"""bench.py --dump-outputs: the results of the last timed sweep, written so that two builds run with the same
arguments can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def _bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         check=True).stdout
    return json.loads(out.strip().split("\n")[-1])


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_is_float64_and_a_large_output_is_a_fixed_sample(tmp_path):
    big = np.arange(bench.DUMP_BYTES // 8, dtype=np.int64).reshape(-1, 4)
    res = {"s": np.array([[1, 2], [3, 1]], dtype=np.int64, order="F"), "logweight": np.array([0.5, -1.0]),
           "big": big, "p_star": 2, "n_resamples": 7, "sweep_kernel_ms": 1.0}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), res)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sorted(a) == ["big", "logweight", "n_resamples", "p_star", "s"]
    assert all(v.dtype == np.float64 for v in a.values())
    np.testing.assert_array_equal(a["s"], res["s"])
    assert a["p_star"].tolist() == [2.0] and a["n_resamples"].tolist() == [7.0]
    assert sum(v.nbytes for v in a.values()) <= bench.DUMP_BYTES
    assert a["big"].size < big.size and np.isin(a["big"], big).all()
    for k in a:
        np.testing.assert_array_equal(a[k], b[k])


def test_reference_arm_dump_is_reproducible(tmp_path):
    args = ["--impl", "reference", "--workload", "cfg1_iris", "--steps", "2", "--warmup", "1"]
    for d in ("a", "b"):
        line = _bench(*args, "--dump-outputs", str(tmp_path / d))
        assert line["steps"] == 2
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert {"s", "p_star", "logweight", "cluster_n", "n_resamples"} <= set(a)
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)


@pytest.mark.gpu
def test_gpu_dump_is_reproducible_and_steps_are_the_timed_steps(tmp_path):
    args = ["--workload", "cfg1_iris", "--steps", "4", "--warmup", "3", "--no-cpu", "--no-cfg4", "--no-pmdi",
            "--no-parity"]
    for d in ("a", "b"):
        line = _bench(*args, "--dump-outputs", str(tmp_path / d))
        assert line["steps"] == 4 and len(line["ms_per_timed_step"]) == 4
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert {"s", "p_star", "logweight", "cluster_n", "label_counts", "n_resamples"} <= set(a)
    assert a["s"].shape == (150, 1) and ((a["s"] >= 1) & (a["s"] <= 10)).all()
    assert (a["cluster_n"].sum(axis=2) == 150).all()
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)

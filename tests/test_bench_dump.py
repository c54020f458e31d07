"""bench.py --dump-outputs: what the last timed step computed, written as .npy files that two builds can be compared
by."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_writes_float_arrays_and_samples_rows_over_the_budget(tmp_path, monkeypatch):
    monkeypatch.setattr(sys, "dont_write_bytecode", sys.dont_write_bytecode)  # importing bench sets it
    import bench
    rng = np.random.default_rng(0)
    arrays = {"points": rng.normal(size=(20000, 4)).astype(np.float32),
              "indices": rng.integers(0, 20000, (20000, 10), dtype=np.int32),
              "T": np.eye(4, dtype=np.float32), "converged": np.asarray(True), "iterations": np.asarray(7)}
    arrays["points"][:, 0] = np.arange(20000)  # row ids
    monkeypatch.setattr(bench, "DUMP_BYTES", 1_000_000)
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert sorted(got) == sorted(arrays)
    assert got["points"].dtype == np.float32 and got["indices"].dtype == np.float64 and got["converged"].dtype == np.float64
    assert sum(a.nbytes for a in got.values()) <= 1_000_000
    assert 0 < len(got["points"]) == len(got["indices"]) < 20000
    # one seeded sample of rows, shared by the arrays of the same length and the same in every run
    rows = got["points"][:, 0].astype(np.int64)
    assert (np.diff(rows) > 0).all()
    assert np.array_equal(got["points"], arrays["points"][rows])
    assert np.array_equal(got["indices"], arrays["indices"][rows].astype(np.float64))
    assert np.array_equal(got["T"], np.eye(4)) and got["iterations"] == 7
    for k, a in got.items():
        assert np.array_equal(a, np.load(tmp_path / "b" / f"{k}.npy"))


@pytest.mark.gpu
def test_bench_dumps_the_same_last_step_twice(tmp_path):
    """Two runs dump the same arrays, and they are those of the last timed step: the voxelised clouds of pair
    (steps - 1) % 4 with their own k-NN lists, covariances and pose, each checked against the oracle."""
    import oracle
    import synthetic
    steps = 3
    env = dict(os.environ, SPX_BENCH_TINY="1")
    dirs = [tmp_path / "run0", tmp_path / "run1"]
    for d in dirs:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                            "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(d)], capture_output=True, text=True,
                           env=env, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
    a = {f[:-4]: np.load(dirs[0] / f) for f in os.listdir(dirs[0])}
    b = {f[:-4]: np.load(dirs[1] / f) for f in os.listdir(dirs[1])}
    assert sorted(a) == sorted(b)
    # identical seeded inputs, and every stage is run-to-run deterministic (the align folds its block sums in a fixed
    # order: DESIGN.md), so the two dumps agree bit for bit
    for k in a:
        assert np.array_equal(a[k], b[k]), k

    # the tiny pairs of bench.py (SPX_BENCH_TINY): the last timed step processed pair (steps - 1) % 4
    tgt_raw, src_raw, _ = synthetic.kitti_pair(42 + (steps - 1) % 4, sweeps=1, azimuth_steps=256)
    for name, raw in (("source", src_raw), ("target", tgt_raw)):
        pts = a[f"{name}_points"]
        assert np.array_equal(pts, oracle.voxel_downsample(raw, 0.25)), name
        oi, od = oracle.knn_bruteforce(pts, pts, 10)
        assert np.array_equal(a[f"{name}_knn_indices"], oi) and np.array_equal(a[f"{name}_knn_sq_distances"], od), name
        oc = oracle.covariance(pts, oi)
        assert np.allclose(a[f"{name}_covs"], oc, rtol=0, atol=1e-6), name
    # bench.py's align: GICP, Gauss-Newton, Huber scale 10, reference defaults otherwise
    P = oracle.default_params(reg_type=3, loss=1, robust_default_scale=10.0)
    o = oracle.align(P, a["source_points"], a["source_covs"], a["target_points"], a["target_covs"], None,
                     oracle.KDTree(a["target_points"]))
    dT = np.linalg.inv(o["T"].astype(np.float64)) @ a["result_T"].astype(np.float64)
    ang = np.linalg.norm(0.5 * np.array([dT[2, 1] - dT[1, 2], dT[0, 2] - dT[2, 0], dT[1, 0] - dT[0, 1]]))
    assert np.linalg.norm(dT[:3, 3]) < 1e-4 and ang < 1e-4, dT

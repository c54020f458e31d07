"""Outlier removal on a ~2 M-point raw cloud (synthetic.kitti_pair target: 16 sweeps x 64 beams x 2048 azimuth steps):
index build, statistical (k = 50 and k = 10; the k+1 self-search and the statistics + compaction timed apart) and
radius (r = 0.3 and 1.0 m, min_neighbors = 5).

    python tools/bench_outlier.py [--reps 7] [--out FILE]

CUDA-event times; the L2 is overwritten (a 512 MB memset) before every timed call; warm-up first; median, min and
max over the repetitions.  Algorithmic bytes per call count what the algorithm must move in HBM at least (points
read, neighbour lists written and read back, per-point outputs), not the candidates a search reads from L2.  The card
name and power limit are read with nvidia-smi in the same run.  Prints one JSON line per step."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import synthetic
    import sycl_points_b200 as spx

    L = spx.lib()
    pts, _, _ = synthetic.kitti_pair()
    n = len(pts)
    q = spx.DeviceQueue(0)
    cloud = spx.PointCloudShared(q, pts)
    flush = spx.DeviceArray(q, (512 << 20,), np.uint8)
    ev0, ev1 = spx.Event(), spx.Event()
    gpu = card()
    lines = []

    def timed(fn, reps=a.reps):
        fn()  # warm-up: modules loaded, scratch grown
        ts = []
        for _ in range(reps):
            spx._lib.check(L.spx_memset(q.handle, flush.ptr, 0, flush.nbytes))
            ev0.record(q)
            fn()
            ev1.record(q)
            q.wait()
            ts.append(ev0.elapsed_ms(ev1))
        return float(np.median(ts)), float(min(ts)), float(max(ts))

    def emit(step, t, nbytes, **kw):
        med, lo, hi = t
        rec = dict(step=step, n=n, ms_median=round(med, 4), ms_min=None if lo is None else round(lo, 4),
                   ms_max=None if hi is None else round(hi, 4), reps=a.reps,
                   algorithmic_bytes=int(nbytes), GBps_at_median=round(nbytes / med / 1e6, 1), gpu=gpu, **kw)
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    trees = []

    def build():
        t = spx.KDTree.build(q, cloud)
        trees.append(t)

    emit("index_build", timed(build), 16 * n + 2 * 16 * n)  # points read, sorted copy written + read by the scatter
    for t in trees:
        t.close()
    tree = spx.KDTree.build(q, cloud)
    q.wait()

    idx = spx.DeviceArray(q, (n,), np.int32)
    mean = spx.DeviceArray(q, (n,), np.float32)
    m = C.c_size_t()
    for k in (50, 10):
        kk = k + 1
        chunk = min(n, 1 << 20, max(256, (1 << 25) // kk // 256 * 256))
        nn_i = spx.DeviceArray(q, (chunk, kk), np.int32)
        nn_d = spx.DeviceArray(q, (chunk, kk), np.float32)

        def knn_only():  # the same chunked self-search the filter runs
            for base in range(0, n, chunk):
                nq = min(chunk, n - base)
                spx._lib.check(L.spx_index_knn(tree.handle, C.c_void_p(cloud.points.ptr.value + 16 * base), nq, kk, None,
                                               nn_i.ptr, nn_d.ptr))

        def full():
            spx._lib.check(L.spx_statistical_outlier_indices(tree.handle, cloud.points.ptr, n, k, 1.0, mean.ptr, idx.ptr,
                                                             C.byref(m)))

        t_knn = timed(knn_only)
        t_all = timed(full)
        lists = 2 * 8 * kk * n  # neighbour lists written by the k-NN and read back
        emit(f"statistical_k{k}_knn", t_knn, 16 * n + 8 * kk * n)
        emit(f"statistical_k{k}_total", t_all, 16 * n + lists + 4 * n * 3 + 4 * int(m.value), kept=int(m.value))
        emit(f"statistical_k{k}_stats_and_compaction", (t_all[0] - t_knn[0], None, None),
             8 * kk * n + 4 * n * 3 + 4 * int(m.value), note="median of the total minus median of the k-NN alone")
        del nn_i, nn_d
    for r in (0.3, 1.0):
        def rad():
            spx._lib.check(L.spx_radius_outlier_indices(tree.handle, cloud.points.ptr, n, r, 5, idx.ptr, C.byref(m)))

        t = timed(rad)
        emit(f"radius_r{r}_m5", t, 16 * n + 4 * n * 2 + 4 * int(m.value), kept=int(m.value))
    if a.out:
        with open(a.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()

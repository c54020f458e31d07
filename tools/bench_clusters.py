"""Euclidean cluster extraction (spx_euclidean_clusters) on the config-2 cloud after the 0.25 m voxel grid (~120 k
points; t = 0.3, 0.5, 1.0 m) and on the ~2 M-point raw cloud (synthetic.kitti_pair target; t = 0.1, 0.2 m).

    python tools/bench_clusters.py [--reps 9] [--out FILE]

Whole calls are timed with CUDA events; the L2 is overwritten (a 512 MB memset) before every timed call; warm-up
first; median, min and max over the repetitions.  The phases are timed apart from the kernel durations of a separate
torch.profiler run over the same calls (mean per call): link (cl_link_kernel), flatten / select (init, flatten, select,
root compaction and the flag scan, up to the call's synchronisation), the cluster sort (radix passes over the C roots),
labels (rank, offsets scan, labels, member scan and compaction) and the member sort (radix passes over the kept
points).  The link's cost scales with the number of neighbours within t, so the mean per point is printed (fp64
cKDTree count).  Algorithmic bytes count the points read once and the per-point outputs written, not the candidates
the search reads from L2.  The card name and power limit are read with nvidia-smi in the same run.  Prints one JSON
line per workload."""
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


def mean_neighbours(pts: np.ndarray, t: float) -> float:
    from scipy.spatial import cKDTree
    p = pts[np.isfinite(pts[:, :3]).all(1), :3].astype(np.float64)
    tree = cKDTree(p)
    return float(tree.count_neighbors(tree, t) - len(p)) / max(len(p), 1)


# kernel name -> phase; the radix passes belong to the cluster sort before cl_rank_kernel, to the member sort after
# cl_member_compact_kernel; scans belong to the phase they run in
PHASE_START = (("cl_init_kernel", "flatten_select"), ("cl_link_kernel", "link"), ("cl_flatten_kernel", "flatten_select"),
               ("cl_rank_kernel", "labels"), ("cl_member_compact_kernel", "member_sort"))


def phase_times(kernels, calls: int) -> dict:
    """kernels: (start_us, name, duration_us) of every kernel of `calls` calls, in launch order"""
    out = {"link": 0.0, "flatten_select": 0.0, "cluster_sort": 0.0, "labels": 0.0, "member_sort": 0.0}
    phase = "flatten_select"
    for _, name, dur in kernels:
        for key, ph in PHASE_START:
            if key in name:
                phase = ph
        if phase == "flatten_select" and "radix_" in name:  # first radix pass after the synchronisation
            phase = "cluster_sort"
        if phase == "member_sort" and "cl_member_compact_kernel" in name:
            out["labels"] += dur
            continue
        out[phase] += dur
    return {k: round(v / calls / 1e3, 4) for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    import synthetic
    import sycl_points_b200 as spx

    L = spx.lib()
    raw, _, _ = synthetic.kitti_pair()
    q = spx.DeviceQueue(0)
    voxel = spx.VoxelGrid(q, 0.25).downsampling(spx.PointCloudShared(q, raw)).points_host()
    flush = spx.DeviceArray(q, (512 << 20,), np.uint8)
    ev0, ev1 = spx.Event(), spx.Event()
    gpu = card()
    lines = []

    for name, pts, tols in (("voxel_0.25", voxel, (0.3, 0.5, 1.0)), ("raw", raw, (0.1, 0.2))):
        n = len(pts)
        cloud = spx.PointCloudShared(q, pts)
        tree = spx.KDTree.build(q, cloud)
        labels = spx.DeviceArray(q, (n,), np.int32)
        idx = spx.DeviceArray(q, (n,), np.int32)
        offs = spx.DeviceArray(q, (n + 1,), np.uint32)
        nc, nm = C.c_size_t(), C.c_size_t()
        for t in tols:
            def call():
                spx._lib.check(L.spx_euclidean_clusters(tree.handle, cloud.points.ptr, n, t, 1, 2 ** 31 - 1, labels.ptr,
                                                        idx.ptr, offs.ptr, C.byref(nc), C.byref(nm)))

            call()  # warm-up: modules loaded, scratch grown
            ts = []
            for _ in range(a.reps):
                spx._lib.check(L.spx_memset(q.handle, flush.ptr, 0, flush.nbytes))
                ev0.record(q)
                call()
                ev1.record(q)
                q.wait()
                ts.append(ev0.elapsed_ms(ev1))
            prof_calls = 3
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for _ in range(prof_calls):
                    call()
                q.wait()
            kern = sorted((e.time_range.start, e.name, e.time_range.elapsed_us()) for e in prof.events()
                          if e.device_type == torch.autograd.DeviceType.CUDA and "kernel" in e.name.lower())
            med = float(np.median(ts))
            nbytes = 16 * n + 4 * n + 4 * int(nm.value) + 4 * (int(nc.value) + 1)
            rec = dict(workload=name, n=n, tolerance=t, ms_median=round(med, 4), ms_min=round(min(ts), 4),
                       ms_max=round(max(ts), 4), reps=a.reps, phases_ms=phase_times(kern, prof_calls),
                       clusters=int(nc.value), members=int(nm.value), mean_neighbours_within_t=round(
                           mean_neighbours(pts, t), 2), algorithmic_bytes=int(nbytes),
                       GBps_at_median=round(nbytes / med / 1e6, 1), gpu=gpu)
            lines.append(rec)
            print(json.dumps(rec), flush=True)
        tree.close()
    if a.out:
        with open(a.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()

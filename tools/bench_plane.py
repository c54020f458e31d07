"""RANSAC plane segmentation (spx_plane_segment) on the ~2 M-point raw cloud (synthetic.kitti_pair target) and on the
config-2 cloud after the 0.25 m voxel grid (~120 k points), for 100, 1000 and 10 000 hypotheses at t = 0.1 m, with
refinement (the library's default).

    python tools/bench_plane.py [--reps 9] [--out FILE]

Whole calls are timed with CUDA events; the L2 is overwritten (a 512 MB memset) before every timed call; warm-up
first; median, min and max over the repetitions.  The kernels are timed apart, from a separate torch.profiler run over
the same calls (mean per call): the scoring kernel (pl_score_kernel, the hypotheses x points hot path) and everything
else.  The scoring kernel's floor is its FP32 issue: about 3.5 lane-instructions per point-hypothesis test (1.5 packed
FFMA2, one FADD and one LEA.HI per test, one broadcast LDS.128 per point for four tests) at 148 SMs x 128 lanes x
1.965 GHz = 37.2 T lane-instructions/s; score_floor_fraction = that floor over the measured kernel time.  The card name
and power limit are read with nvidia-smi in the same run.  Prints one JSON line per workload."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LANE_INSTR_PER_TEST = 3.5
LANE_INSTR_PER_S = 148 * 128 * 1.965e9


def card() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    import synthetic
    import sycl_points_b200 as spx

    raw, _, _ = synthetic.kitti_pair()
    q = spx.DeviceQueue(0)
    voxel = spx.VoxelGrid(q, 0.25).downsampling(spx.PointCloudShared(q, raw)).points_host()
    flush = spx.DeviceArray(q, (512 << 20,), np.uint8)
    ev0, ev1 = spx.Event(), spx.Event()
    gpu = card()
    t = 0.1
    lines = []

    for name, pts in (("raw", raw), ("voxel_0.25", voxel)):
        n = len(pts)
        cloud = spx.PointCloudShared(q, pts)
        seg = spx.PlaneSegmentation(q)
        for H in (100, 1000, 10000):
            def call():
                return seg.segment(cloud, t, H)

            r = call()  # warm-up: modules loaded, scratch grown
            ts = []
            for _ in range(a.reps):
                spx._lib.check(spx.lib().spx_memset(q.handle, flush.ptr, 0, flush.nbytes))
                ev0.record(q)
                r = call()
                ev1.record(q)
                q.wait()
                ts.append(ev0.elapsed_ms(ev1))
            prof_calls = 3
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for _ in range(prof_calls):
                    call()
                q.wait()
            kern = [(e.name, e.time_range.elapsed_us()) for e in prof.events()
                    if e.device_type == torch.autograd.DeviceType.CUDA and "kernel" in e.name.lower()]
            score_ms = sum(d for nm, d in kern if "pl_score_kernel" in nm) / prof_calls / 1e3
            other_ms = sum(d for nm, d in kern if "pl_score_kernel" not in nm) / prof_calls / 1e3
            floor_ms = LANE_INSTR_PER_TEST * n * H / LANE_INSTR_PER_S * 1e3
            med = float(np.median(ts))
            rec = dict(workload=name, n=n, hypotheses=H, threshold=t, ms_median=round(med, 4), ms_min=round(min(ts), 4),
                       ms_max=round(max(ts), 4), reps=a.reps, score_kernel_ms=round(score_ms, 4),
                       other_kernels_ms=round(other_ms, 4), score_floor_ms=round(floor_ms, 4),
                       score_floor_fraction=round(floor_ms / score_ms, 3) if score_ms else None,
                       tests_per_s=round(n * H / (score_ms * 1e-3), 1) if score_ms else None,
                       inliers=len(r.inliers), hypothesis=r.hypothesis, gpu=gpu)
            lines.append(rec)
            print(json.dumps(rec), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()

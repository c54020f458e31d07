"""Global registration stages on the GPU: normals, radius search, FPFH (spx_fpfh), feature correspondences plain and
mutual (spx_feature_correspondences) and RANSAC (spx_ransac_registration) at 10^4 / 10^5 / 10^6 hypotheses, on the
1.0 m voxel clouds of synthetic.kitti_pair(42) with T_gt = trans(4, -2, 0.05) Rz(60 deg) (the end-to-end test's
pair), plus the correspondence search on the 0.25 m voxel clouds (~120 k x 120 k rows), where it is clearly
FP32-bound.

    python tools/bench_global.py [--reps 9] [--out FILE]

Whole calls are timed with CUDA events; the L2 is overwritten (a 512 MB memset) before every timed call; warm-up
first; median, min and max over the repetitions.  The hot kernels are timed apart, from a separate torch.profiler run
over the same calls (mean per call).  Floors are FP32 issue at 148 SMs x 128 lanes x 1.965 GHz = 37.2 T
lane-instructions/s:
- matching (fc_nn_kernel): N_s N_t pairs at 33 lane-instructions each (per target row and two source rows the loop
  issues 33 FADD2, 32 FFMA2 and 1 FMUL2), the nine broadcast LDS.128 per row left out;
- scoring (rs_score_kernel): H M tests at 9 lane-instructions each (per two hypotheses and one correspondence 9 FFMA2
  for R p + t, 3 FADD2 for y - q, 1 FMUL2 + 2 FFMA2 for d^2, 1 FADD2 for d^2 - eps^2, and one LEA.HI per test).
floor_fraction = floor / measured kernel time.  The card name and power limit are read with nvidia-smi in the same
run.  Prints one JSON line per measurement."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LANE_INSTR_PER_S = 148 * 128 * 1.965e9
MATCH_INSTR_PER_PAIR = 33.0
SCORE_INSTR_PER_TEST = 9.0


def card() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def pose(deg, t):
    a = np.deg2rad(deg)
    T = np.eye(4)
    T[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
    T[:3, 3] = t
    return T


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    import synthetic
    import sycl_points_b200 as spx

    tgt_raw, src_raw, _ = synthetic.kitti_pair(42, T_gt=pose(60.0, (4.0, -2.0, 0.05)))
    q = spx.DeviceQueue(0)
    flush = spx.DeviceArray(q, (512 << 20,), np.uint8)
    ev0, ev1 = spx.Event(), spx.Event()
    gpu = card()
    lines = []

    def timed(call, kernels=()):
        call()  # warm-up: modules loaded, scratch grown
        ts = []
        for _ in range(a.reps):
            spx._lib.check(spx.lib().spx_memset(q.handle, flush.ptr, 0, flush.nbytes))
            ev0.record(q)
            call()
            ev1.record(q)
            q.wait()
            ts.append(ev0.elapsed_ms(ev1))
        kms = {}
        if kernels:
            calls = 3
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for _ in range(calls):
                    call()
                q.wait()
            ev = [(e.name, e.time_range.elapsed_us()) for e in prof.events()
                  if e.device_type == torch.autograd.DeviceType.CUDA]
            for k in kernels:
                kms[k] = sum(d for nm, d in ev if k in nm) / calls / 1e3
        return dict(ms_median=round(float(np.median(ts)), 4), ms_min=round(min(ts), 4), ms_max=round(max(ts), 4),
                    reps=a.reps), kms

    def emit(rec):
        rec["gpu"] = gpu
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    def prepare(raw, voxel):
        pts = spx.VoxelGrid(q, voxel).downsampling(spx.PointCloudShared(q, raw)).points_host()
        cloud = spx.PointCloudShared(q, pts)
        tree = spx.KDTree.build(q, cloud)
        return cloud, tree

    feats = {}
    for name, raw in (("source", src_raw), ("target", tgt_raw)):
        cloud, tree = prepare(raw, 1.0)
        n = cloud.size()

        def normals():
            spx.covariance.estimate_normals(tree.knn_search(cloud, 15), cloud)
        t, _ = timed(normals)
        emit(dict(stage="normals_k15", cloud=name, voxel=1.0, n=n, **t))
        nn = spx.KNNResult()

        def radius():
            tree.radius_search_async(cloud, 100, 5.0, nn)
        t, _ = timed(radius)
        emit(dict(stage="radius_search_r5_k100", cloud=name, voxel=1.0, n=n, **t))
        f = spx.DeviceArray(q, (n, 33), np.float32)

        def fpfh():
            spx._lib.check(spx.lib().spx_fpfh(q.handle, cloud.points.ptr, cloud.normals.ptr, n, nn.indices.ptr,
                                              nn.distances.ptr, 100, f.ptr))
        t, k = timed(fpfh, ("fp_spfh_kernel", "fp_fpfh_kernel"))
        listed = int((nn.indices_host() >= 0).sum())
        emit(dict(stage="fpfh_r5_k100", cloud=name, voxel=1.0, n=n, listed_neighbours=listed, **t,
                  spfh_kernel_ms=round(k["fp_spfh_kernel"], 4), fpfh_kernel_ms=round(k["fp_fpfh_kernel"], 4)))
        feats[name] = (cloud, f)

    (sc, sf), (tc, tf) = feats["source"], feats["target"]
    ns, nt = sc.size(), tc.size()
    corr = None
    for mutual in (False, True):
        out = {}

        def match():
            out["c"] = spx.match_features(q, sf, tf, mutual=mutual)
        t, k = timed(match, ("fc_nn_kernel",))
        floor = MATCH_INSTR_PER_PAIR * ns * nt * (2 if mutual else 1) / LANE_INSTR_PER_S * 1e3
        emit(dict(stage="correspondences_mutual" if mutual else "correspondences", n_source=ns, n_target=nt,
                  m=len(out["c"][0]), **t, match_kernel_ms=round(k["fc_nn_kernel"], 4), match_floor_ms=round(floor, 4),
                  floor_fraction=round(floor / k["fc_nn_kernel"], 3)))
        if not mutual:
            corr = out["c"]
    M = len(corr[0])
    reg = spx.RANSACRegistration(q)
    for H in (10_000, 100_000, 1_000_000):
        out = {}

        def ransac():
            out["r"] = reg.align(sc, tc, corr, 1.0, H)
        t, k = timed(ransac, ("rs_score_kernel",))
        floor = SCORE_INSTR_PER_TEST * H * M / LANE_INSTR_PER_S * 1e3
        emit(dict(stage="ransac", hypotheses=H, m=M, **t, score_kernel_ms=round(k["rs_score_kernel"], 4),
                  score_floor_ms=round(floor, 4), floor_fraction=round(floor / k["rs_score_kernel"], 3),
                  inliers=len(out["r"].inliers), hypothesis=out["r"].hypothesis))

    # the correspondence search at ~120 k x 120 k: descriptors of the 0.25 m clouds (r = 1.25 m, 100 neighbours)
    big = []
    for raw in (src_raw, tgt_raw):
        cloud, tree = prepare(raw, 0.25)
        spx.covariance.estimate_normals(tree.knn_search(cloud, 15), cloud)
        big.append(spx.FPFHEstimation(q).compute(cloud, 1.25, 100, tree=tree))
    ns, nt = big[0].shape[0], big[1].shape[0]
    t, k = timed(lambda: spx.match_features(q, big[0], big[1]), ("fc_nn_kernel",))
    floor = MATCH_INSTR_PER_PAIR * ns * nt / LANE_INSTR_PER_S * 1e3
    emit(dict(stage="correspondences", voxel=0.25, n_source=ns, n_target=nt, **t,
              match_kernel_ms=round(k["fc_nn_kernel"], 4), match_floor_ms=round(floor, 4),
              floor_fraction=round(floor / k["fc_nn_kernel"], 3)))
    if a.out:
        with open(a.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()

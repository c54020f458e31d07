#!/usr/bin/env python
"""bench.py — the registration hot path on BASELINE.json's configurations.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl spx|reference]
                    [--workload pair|batch|knn_index|knn_bf|align_sharded] [--no-extras] [--no-cpu-baseline]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   (N > 1)

--workload pair (DEFAULT, BASELINE config 2 — the configuration the metric is quoted on):
    a "step" is one pass of the whole per-pair hot path over one synthetic LiDAR-shaped scan pair
    (2.0 M raw points per cloud -> ~120 k points after the 0.25 m voxel grid):
        voxel-grid downsample (both clouds) -> exact KNN index build (both) -> KNN k=10 (both)
        -> covariance from 10 neighbours (both) -> GICP align (Gauss-Newton, Huber scale 10,
        max_correspondence_distance 2.0, <= 20 iterations, criteria 1e-3 / 1e-3, initial guess I)
    FOUR distinct pairs (scene seeds 42.. per rank) rotate through the timed loop, so no step re-processes the
    cloud its predecessor left in the caches and the voxel grid's guessed key box is a real guess.
    `value`      = scan pairs per second, whole job (all ranks), raw clouds resident in HBM;
    `e2e`        = the same through the public API from pinned HOST buffers: every step copies its own two raw
                   clouds (65 MB) host->device and reads its registration result back inside the timed region
                   (the copy of pair s+1 is double-buffered on a copy queue: a streaming front end);
    `ms_per_iter`= GICP align milliseconds per executed ICP iteration (the other half of the metric);
    `roofline`   = the persistent align kernel (nearest neighbour + linearise + reduce + solve, every iteration of
                   an align in one launch): algorithmic bytes 192 N_s + 16 N_t per iteration (SURVEY.md §8(d));
    `cpu_baseline` = the oracle port of the reference's CPU path (-O3 -march=native build) on the same pairs;
    `extras`     = quick runs of the other configurations in the same job: config 3 (KNN Mqueries/s, index and
                   brute force, queries sharded over the ranks), config 4 (dense pair, source sharded, ms/iter with
                   the in-kernel NVLink exchange), config 5 (batched pairs inside one GPU, pairs/s), and the odometry
                   loop that calls the path in production (LiDAROdometryPipeline on a synthetic drive, frames/s).
    N > 1: every rank aligns its own independent pairs on its own GPU (no data-path collective: weak scaling of
    batched pairs, SURVEY.md §8(e)); max over ranks of the device time.

--dump-outputs DIR (--workload pair): after the timed steps, what the last of them computed -- both voxelised clouds,
    their covariances and k-NN lists, and the registration result -- as DIR/<name>.npy (float32, or float64 for
    integer data; at most DUMP_BYTES in all).  The inputs are seeded, so two builds run with the same arguments can be
    compared output for output.

--workload batch (config 5): a step = 64 raw scan pairs (~1 M points per cloud -> ~64 k) per rank through
    spx_align_batch: per cloud voxel grid -> index -> KNN -> covariances on concurrent lanes, then ONE batched align.
--workload knn_index / knn_bf (config 3): 1 M x 1 M, k = 20, queries sharded over the ranks (strong scaling).
--workload align_sharded (config 4): GICP on the dense pair, source sharded over the ranks, 20 forced iterations.
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)

import synthetic  # noqa: E402

VOXEL = 0.25
K_COV = 10
N_ROTATE = 4
STREAM_SLOTS = 3
DUMP_BYTES = 64_000_000  # --dump-outputs writes at most this much in all
TINY = bool(os.environ.get("SPX_BENCH_TINY"))  # CPU tests of the launch logic only
WORKLOADS = {
    "pair": ("config 2: synthetic KITTI-shaped pair (16 accumulated 64-beam sweeps, ~2.0M raw pts/cloud), 0.25 m voxel "
             "-> ~120k pts, KNN k=10 covariances, GICP GN Huber(10) max_corr 2.0 <=20 iters; 4 distinct pairs rotate"),
    "batch": ("config 5: batched odometry, 64 independent raw scan pairs per GPU per step (~1.0M raw pts/cloud -> ~64k "
              "after the 0.25 m voxel grid), voxel + KNN k=10 covariances (both clouds) + GICP GN Huber(10) <=20 iters, "
              "one spx_align_batch call"),
    "knn_index": "config 3: exact KNN through the grid index, k=20, 1M queries x 1M targets (mt19937 1234/4321), queries sharded",
    "knn_bf": "config 3: brute-force KNN, k=20, 1M queries x 1M targets (mt19937 1234/4321), queries sharded",
    "align_sharded": ("config 4: GICP on the dense pair (8.2M raw pts/cloud -> ~1.6M after the 0.05 m voxel grid), source "
                      "sharded over the ranks, target + index replicated, 20 forced GN iterations, in-kernel NVLink exchange"),
}
METRICS = {"pair": ("gicp_scan_pairs_per_s", "pairs/s", True, "weak"), "batch": ("gicp_scan_pairs_per_s", "pairs/s", True, "weak"),
           "knn_index": ("knn_mqueries_per_s", "Mqueries/s", True, "strong"), "knn_bf": ("knn_mqueries_per_s", "Mqueries/s", True, "strong"),
           "align_sharded": ("gicp_align_ms_per_iter", "ms", False, "strong")}


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


# ------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i",
                 str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------ job context
class Ctx:
    def __init__(self, args):
        self.args = args
        self.rank, self.world, self.local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
        self.dist = None
        self.torch = None
        self.peaks = load_peaks()
        self.peak_hbm = float(self.peaks.get("hbm_gbs", 6650.0))

    def init_gpu(self):
        if self.world > 1:
            import torch
            import torch.distributed as dist
            torch.cuda.set_device(self.local)
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist, self.torch = dist, torch
        import sycl_points_b200 as spx  # fails loudly if libspx.so is missing / cannot be built
        self.spx = spx
        self.q = spx.DeviceQueue(self.local)
        self.info = self.q.device_info()
        self.flush = spx.DeviceArray(self.q, (256 << 20,), np.uint8)  # > 126 MB L2

    def l2_flush(self):
        spx = self.spx
        spx._lib.check(spx.lib().spx_memset(self.q.handle, self.flush.ptr, 0, self.flush.nbytes))

    def barrier(self, *queues):
        self.q.wait()
        for qq in queues:
            qq.wait()
        if self.dist is not None:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        if self.dist is None:
            return list(vals)
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def sum_over_ranks(self, *vals):
        if self.dist is None:
            return list(vals)
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return t.tolist()


# ------------------------------------------------------------------ config 2: one pair per step
class PairPipeline:
    """One scan pair through the hot path.  The two clouds' chains (voxel grid -> index -> KNN k=10 ->
    covariances) are independent until the align, so they run on two queues (two CUDA streams, the
    source chain driven by a worker thread): the kernels of this stage are latency-bound at 120 k
    points and overlap almost perfectly.  Distinct DeviceQueues running concurrently is the
    documented contract of the C-ABI (include/spx.h); the align then runs on the target's queue."""

    def __init__(self, spx, q, n_src_raw, n_tgt_raw):
        from concurrent.futures import ThreadPoolExecutor
        self.spx, self.q = spx, q
        # the source chain starts later (worker thread) and its k-NN is the longer one: it gets the more urgent
        # stream so that both chains are done at the same time (SPX_BENCH_Q2_PRIORITY=0 to compare)
        self.q2 = spx.DeviceQueue(q.device, priority=int(os.environ.get("SPX_BENCH_Q2_PRIORITY", "1")))
        self.vg, self.vg2 = spx.VoxelGrid(q, VOXEL), spx.VoxelGrid(self.q2, VOXEL)
        params = spx.RegistrationParams()  # GICP, GN, max_corr 2.0, max_iter 20, criteria 1e-3 (reference defaults)
        params.robust.type = spx.RobustLossType.HUBER
        params.robust.default_scale = 10.0
        self.reg = spx.Registration(q, params)
        self.nn_s, self.nn_t = spx.KNNResult(), spx.KNNResult()
        # ONE worker thread per queue: a queue (its scratch arena, its pinned staging block, its voxel-grid state) is
        # single-threaded by contract (include/spx.h), and in the pipelined mode the chains of pair s+1 are submitted
        # while those of pair s may still be running — a shared two-worker pool could hand the second chain of a
        # queue to the idle worker while the first is still inside the library on the same queue.
        self.pool = ThreadPoolExecutor(max_workers=1)   # drives q2 (source chains)
        self.pool_t = ThreadPoolExecutor(max_workers=1)  # drives q (target chains) in the pipelined mode
        self.src_done = spx.Event()
        self.last = None
        # pipelined mode (two pairs in flight): the align of pair s runs on its own queue while both feeder chains
        # of pair s+1 run on q / q2
        self.q3 = spx.DeviceQueue(q.device)
        # the pipelined align leaves SM resources to the next pair's feeder kernels: its persistent grid is capped at
        # two CTAs per SM (a full-occupancy cooperative grid can neither start while feeders hold SMs nor share them)
        import copy
        params3 = copy.deepcopy(params)
        params3.max_blocks = int(os.environ.get("SPX_BENCH_ALIGN_BLOCKS", 2 * q.device_info()["sm_count"]))
        self.reg3 = spx.Registration(self.q3, params3)
        self.nn_pipe = [(spx.KNNResult(), spx.KNNResult()) for _ in range(2)]
        self.done_pipe = [(spx.Event(), spx.Event()) for _ in range(2)]
        # resident raw clouds: one (source, target) per rotating pair, sized for the largest
        self.n_src_raw, self.n_tgt_raw = n_src_raw, n_tgt_raw
        self.resident = []
        # end-to-end (streaming) mode: a copy queue and three sets of raw buffers, so that the copy engine
        # works two pairs ahead of the align (what a LiDAR front end does with its frames): upload of pair s+2 ||
        # feeder chains of pair s+1 || align of pair s
        self.qc = spx.DeviceQueue(q.device)
        self.stream_raw = []
        self.stream_xyz = []
        for _ in range(STREAM_SLOTS):
            rs, rt = spx.PointCloudShared(self.qc), spx.PointCloudShared(self.qc)
            rs.adopt_points(spx.DeviceArray(self.qc, (max(n_src_raw), 4), np.float32), 0)
            rt.adopt_points(spx.DeviceArray(self.qc, (max(n_tgt_raw), 4), np.float32), 0)
            self.stream_raw.append((rs, rt, spx.Event()))
            # the host sends packed xyz (12 B per point); the device expands it to xyz1
            self.stream_xyz.append((spx.DeviceArray(self.qc, (max(n_src_raw), 3), np.float32),
                                    spx.DeviceArray(self.qc, (max(n_tgt_raw), 3), np.float32)))

    def add_resident(self, src_host, tgt_host):
        spx = self.spx
        rs, rt = spx.PointCloudShared(self.q2), spx.PointCloudShared(self.q)
        rs.adopt_points(spx.DeviceArray(self.q2, src_host.shape, np.float32), len(src_host))
        rt.adopt_points(spx.DeviceArray(self.q, tgt_host.shape, np.float32), len(tgt_host))
        rs.points.upload(src_host, sync=False)
        rt.points.upload(tgt_host, sync=False)
        self.q2.wait()
        self.q.wait()
        self.resident.append((rs, rt))

    def _chain(self, q, vg, raw, nn, after=None, done=None):
        spx = self.spx
        if after is not None:
            q.wait_event(after)  # nothing of this chain starts before the step's start event
        cloud = vg.downsampling(raw)
        tree = spx.KDTree.build(q, cloud)
        tree.knn_search_async(cloud, K_COV, nn)
        spx.covariance.estimate(nn, cloud)
        if done is not None:
            done.record(q)  # the other queue waits for this on the device, the host does not
        return cloud, tree

    def stream_upload(self, slot, src_xyz_host, tgt_xyz_host):
        """H2D of one pair's raw clouds (pinned packed-xyz source) into buffer set `slot`, on the copy queue, and their
        expansion to xyz1 on the device"""
        spx = self.spx
        rs, rt, ev = self.stream_raw[slot]
        xs, xt = self.stream_xyz[slot]
        L = spx.lib()
        spx._lib.check(L.spx_memcpy_h2d(self.qc.handle, xt.ptr, tgt_xyz_host.ctypes.data, tgt_xyz_host.nbytes))
        rt.set_points_xyz(xt, len(tgt_xyz_host))
        spx._lib.check(L.spx_memcpy_h2d(self.qc.handle, xs.ptr, src_xyz_host.ctypes.data, src_xyz_host.nbytes))
        rs.set_points_xyz(xs, len(src_xyz_host))
        ev.record(self.qc)

    def run_streamed(self, slot):
        """process the pair in buffer set `slot` once its upload has landed"""
        rs, rt, ev = self.stream_raw[slot]
        fut = self.pool.submit(self._chain, self.q2, self.vg2, rs, self.nn_s, ev, self.src_done)
        tgt, tree_t = self._chain(self.q, self.vg, rt, self.nn_t, ev)
        src, tree_s = fut.result()
        self.q.wait_event(self.src_done)
        res = self.reg.align(src, tgt, tree_t)
        self.last = (src, tgt, tree_t, res, self.nn_s, self.nn_t)
        tree_s.close()
        return res

    def feeders_async(self, which, slot, start_event=None, streamed=False):
        """both chains of one pair (resident buffer set `which`, or streamed buffer set `which` once its upload has
        landed) on q / q2, each on its own pool thread; returns the two futures"""
        if streamed:
            rs, rt, ev = self.stream_raw[which]
        else:
            (rs, rt), ev = self.resident[which], start_event
        nn_s, nn_t = self.nn_pipe[slot]
        ds, dt_ = self.done_pipe[slot]
        return (self.pool.submit(self._chain, self.q2, self.vg2, rs, nn_s, ev, ds),
                self.pool_t.submit(self._chain, self.q, self.vg, rt, nn_t, ev, dt_))

    def align_pipelined(self, futs, slot):
        """align of the pair whose feeders are `futs`, on the third queue (the feeders of the next pair may already
        be running on q / q2)"""
        src, tree_s = futs[0].result()
        tgt, tree_t = futs[1].result()
        ds, dt_ = self.done_pipe[slot]
        self.q3.wait_event(ds)
        self.q3.wait_event(dt_)
        res = self.reg3.align(src, tgt, tree_t)
        self.last = (src, tgt, tree_t, res, *self.nn_pipe[slot])
        tree_s.close()
        tree_t.close()
        return res

    def run(self, which, start_event=None):
        rs, rt = self.resident[which]
        fut = self.pool.submit(self._chain, self.q2, self.vg2, rs, self.nn_s, start_event, self.src_done)
        tgt, tree_t = self._chain(self.q, self.vg, rt, self.nn_t)
        src, tree_s = fut.result()
        # the source chain's last kernels (covariances) must be done before the align reads them: a
        # device-side wait, so that the align's set-up launches queue up behind the running chains
        self.q.wait_event(self.src_done)
        res = self.reg.align(src, tgt, tree_t)  # synchronises (result comes back to the host)
        self.last = (src, tgt, tree_t, res, self.nn_s, self.nn_t)
        tree_s.close()
        return res


def rotating_pairs(rank):
    """the N_ROTATE distinct (target_raw, source_raw, T_gt) of this rank (scene seeds 42 + 4 rank + j)"""
    if TINY:
        return [synthetic.kitti_pair(42 + j, sweeps=1, azimuth_steps=256) for j in range(N_ROTATE)]
    return [synthetic.kitti_pair(42 + N_ROTATE * rank + j) for j in range(N_ROTATE)]


def cpu_pair(oracle, src_raw, tgt_raw):
    """The reference's CPU path for one pair, restated (oracle port): std::sort voxel grid, host
    KD-tree build, KD-tree KNN k=10, covariance, KD-tree NN + GICP linearise per iteration."""
    src = oracle.voxel_downsample(src_raw, VOXEL, 1, unstable=True)
    tgt = oracle.voxel_downsample(tgt_raw, VOXEL, 1, unstable=True)
    ts, tt = oracle.KDTree(src), oracle.KDTree(tgt)
    idx_s, _ = ts.knn(src, K_COV, mode=1)
    idx_t, _ = tt.knn(tgt, K_COV, mode=1)
    cs, ct = oracle.covariance(src, idx_s), oracle.covariance(tgt, idx_t)
    P = oracle.default_params(reg_type=3, loss=1, opt_method=0, max_iterations=20, robust_default_scale=10.0,
                              sum_mode=1, knn_mode=1)
    return oracle.align(P, src, cs, tgt, ct, None, tt), len(src), len(tgt)


def timing_oracle():
    """the oracle's -O3 -march=native build with every host thread (torchrun exports OMP_NUM_THREADS=1 to its
    workers: the CPU baseline must not inherit that)"""
    import oracle
    try:
        oracle.use_fast_build()
        build = "-O3 -march=native"
    except Exception as e:  # falls back to the parity build (still a valid, slower, baseline), and says so
        build = f"-O2 parity build; the -O3 -march=native build failed: {e!r}"
    cores = os.cpu_count() or 1
    oracle.set_num_threads(cores)
    return oracle, oracle.num_threads(), build


def pair_config(ns_list, nt_list):
    """the `config` object: the same keys and values from both arms (the clouds are bit-identical).  What an arm
    MEASURED — e.g. how many iterations its aligns took: a borderline 1e-3 criterion can fall either side between the
    GPU path and the CPU port's unstable std::sort / KD-tree tie order — is reported next to it, not inside it."""
    return {"workload": WORKLOADS["pair"], "pairs_rotated": N_ROTATE, "n_src": [int(x) for x in ns_list],
            "n_tgt": [int(x) for x in nt_list], "voxel_m": VOXEL, "k_cov": K_COV}


def run_reference(ctx):
    """--impl reference: the reference's own CPU implementation of the path.  The SYCL build is not possible in
    this image (no SYCL compiler, no Eigen: DESIGN.md), so this is the oracle port with every host thread, on the
    same rotating pairs and settings; rank 0 alone runs it."""
    args = ctx.args
    if ctx.rank != 0:
        return
    oracle, cores, build = timing_oracle()
    pairs = rotating_pairs(0)
    for w in range(args.warmup):
        cpu_pair(oracle, pairs[w % N_ROTATE][1], pairs[w % N_ROTATE][0])
    stats = {}
    t0 = time.perf_counter()
    iters = 0
    for s in range(args.steps):
        tgt_raw, src_raw, _ = pairs[s % N_ROTATE]
        r, ns, nt = cpu_pair(oracle, src_raw, tgt_raw)
        stats[s % N_ROTATE] = (ns, nt, r["iterations"] + 1)
        iters += r["iterations"] + 1
    dt = time.perf_counter() - t0
    for j in range(N_ROTATE):  # the config names all rotating pairs even when fewer steps were timed
        if j not in stats:
            r, ns, nt = cpu_pair(oracle, pairs[j][1], pairs[j][0])
            stats[j] = (ns, nt, r["iterations"] + 1)
    value = args.steps / dt
    metric, unit, hib, scaling = METRICS["pair"]
    line = {
        "impl": "reference", "metric": metric, "value": value, "unit": unit, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": hib,
        "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": pair_config([stats[j][0] for j in range(N_ROTATE)], [stats[j][1] for j in range(N_ROTATE)]),
        "icp_iterations_per_pair": [int(stats[j][2]) for j in range(N_ROTATE)],
        "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": "port",
                         "sample": f"{args.steps} whole pairs (full pipeline) on {cores} host threads, {build}"},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "ms_per_iter": 1e3 * dt / max(iters, 1),
    }
    emit(line)


def workload_pair(ctx):
    args, spx, q = ctx.args, ctx.spx, ctx.q
    # every rank drives its queues from three host threads; only when those outnumber the host's cores do the queues wait
    # on an OS primitive instead of spinning (SPX_BENCH_SYNC=spin|block overrides).  Measured, 8 ranks on 32 cores:
    # spinning 8302 pairs/s (0.964 ms/step), blocking 6567 (1.218) — profiles/r2r_bench_8gpu*.json
    sync_mode = os.environ.get("SPX_BENCH_SYNC", "block" if 3 * ctx.world > (os.cpu_count() or 1) else "spin")
    pairs = rotating_pairs(ctx.rank)
    pipe = PairPipeline(spx, q, [len(p[1]) for p in pairs], [len(p[0]) for p in pairs])
    if sync_mode == "block":
        for qq in (q, pipe.q2, pipe.qc, pipe.q3):
            qq.set_blocking_sync(True)
    pins = []
    for tgt_raw, src_raw, _ in pairs:
        ps, pt = spx.PinnedArray((len(src_raw), 3)), spx.PinnedArray((len(tgt_raw), 3))
        ps.array[...] = src_raw[:, :3]
        pt.array[...] = tgt_raw[:, :3]
        pins.append((ps, pt))
        pipe.add_resident(src_raw, tgt_raw)

    W = max(args.warmup, N_ROTATE + 1)
    for w in range(W):
        pipe.run(w % N_ROTATE)
    # ---------------- device-resident timing
    sampler = ClockSampler(ctx.local)
    if ctx.rank == 0:  # one sampler per job: the JSON line reports rank 0's GPU
        sampler.start()
    ev = [(spx.Event(), spx.Event()) for _ in range(args.steps)]
    loop_ms, launches, iters_done = [], 0, 0
    per_pair = {}
    ctx.barrier(pipe.q2, pipe.qc)
    launches0 = spx.kernel_launch_count()
    wall0 = time.perf_counter()
    for s in range(args.steps):
        ctx.l2_flush()
        ev[s][0].record(q)
        res = pipe.run(s % N_ROTATE, ev[s][0])
        ev[s][1].record(q)
        t = pipe.reg.last_timing()
        loop_ms.append(t["loop_ms"])
        launches += t["launches"]
        iters_done += t["iterations"]
        per_pair[s % N_ROTATE] = (pipe.last[0].size(), pipe.last[1].size(), t["iterations"], res)
    ctx.barrier(pipe.q2, pipe.qc)
    wall = time.perf_counter() - wall0
    serial_launches = spx.kernel_launch_count() - launches0
    step_ms = [a.elapsed_ms(b) for a, b in ev]
    serial_ms = float(np.sum(step_ms))
    # ---------------- throughput: two pairs in flight (the feeders of pair s+1 overlap the align of pair s)
    def pipelined(n_steps, streamed):
        a, b = spx.Event(), spx.Event()
        ctx.barrier(pipe.q2, pipe.qc, pipe.q3)
        ctx.l2_flush()
        a.record(q)
        for qq in (pipe.q2, pipe.qc, pipe.q3):
            qq.wait_event(a)
        if streamed:
            pipe.stream_upload(0, pins[0][0].array, pins[0][1].array)
            if n_steps > 1:
                pipe.stream_upload(1, pins[1 % N_ROTATE][0].array, pins[1 % N_ROTATE][1].array)
        futs = pipe.feeders_async(0, 0, a, streamed)
        marks = [time.perf_counter()]
        for s in range(n_steps):
            nxt = None
            if streamed and s + 2 < n_steps:
                # buffer set (s+2) % 3 was last read by the feeders of pair s-1: they are done (their align returned)
                pipe.stream_upload((s + 2) % STREAM_SLOTS, pins[(s + 2) % N_ROTATE][0].array,
                                   pins[(s + 2) % N_ROTATE][1].array)
            if s + 1 < n_steps:
                if streamed:
                    nxt = pipe.feeders_async((s + 1) % STREAM_SLOTS, (s + 1) % 2, None, True)
                else:
                    nxt = pipe.feeders_async((s + 1) % N_ROTATE, (s + 1) % 2, None, False)
            pipe.align_pipelined(futs, s % 2)
            marks.append(time.perf_counter())  # the align returned: this pair's result is on the host
            futs = nxt
        b.record(pipe.q3)
        ctx.barrier(pipe.q2, pipe.qc, pipe.q3)
        step_hist.append(np.diff(marks) * 1e3)
        return float(a.elapsed_ms(b))

    step_hist = []

    def spread(ms):
        """median / worst host-observed step of one pipelined run (the mean is the reported figure)"""
        return {"median_ms": float(np.median(ms)), "p99_ms": float(np.percentile(ms, 99)), "max_ms": float(np.max(ms))}

    pipelined(4, False)
    launches1 = spx.kernel_launch_count()
    total_ms = pipelined(args.steps, False)
    gpu_launches = spx.kernel_launch_count() - launches1
    clocks = sampler.stop()
    for j in range(N_ROTATE):
        if j not in per_pair:
            res = pipe.run(j)
            per_pair[j] = (pipe.last[0].size(), pipe.last[1].size(), pipe.reg.last_timing()["iterations"], res)
    # ---------------- end to end from host buffers (streaming: upload of pair s+1 overlaps pair s)
    # Every step's inputs are copied from pinned host memory inside the timed region and every
    # step's result struct is read back (align synchronises); one bracket around the K steps because
    # consecutive steps overlap.
    value_spread = spread(step_hist[-1])
    pipelined(4, True)
    e2e_ms = pipelined(args.steps, True)
    e2e_spread = spread(step_hist[-1])
    outputs = last_step_outputs(pipe) if args.dump_outputs else None
    serial_ms, = ctx.max_over_ranks(serial_ms)
    total_ms, e2e_ms = ctx.max_over_ranks(total_ms, e2e_ms)
    gpu_launches = int(ctx.sum_over_ranks(float(gpu_launches))[0])

    ns_l = [per_pair[j][0] for j in range(N_ROTATE)]
    nt_l = [per_pair[j][1] for j in range(N_ROTATE)]
    it_l = [per_pair[j][2] for j in range(N_ROTATE)]
    value = ctx.world * args.steps / (total_ms * 1e-3)
    e2e = ctx.world * args.steps / (e2e_ms * 1e-3)
    # algorithmic bytes actually processed by the timed align launches (SURVEY.md §8(d)): per iteration 192 N_s + 16 N_t
    alg_total = 0.0
    for s in range(args.steps):
        j = s % N_ROTATE
        alg_total += it_l[j] * (192 * ns_l[j] + 16 * nt_l[j])
    kern_ms = float(np.sum(loop_ms)) / max(iters_done, 1)   # per iteration
    launch_ms = float(np.sum(loop_ms)) / max(launches, 1)   # per launch of the align kernel (all iterations)
    achieved = alg_total / (float(np.sum(loop_ms)) * 1e-3) / 1e9
    traffic = None
    try:  # dram__bytes_read.sum + dram__bytes_write.sum of that kernel from the committed ncu --set full capture
        traffic = float(json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))["dram_bytes_per_launch"])
    except Exception:
        pass
    errs = []
    for j in range(N_ROTATE):
        dT = np.linalg.inv(pairs[j][2].astype(np.float64)) @ per_pair[j][3].T.astype(np.float64)
        errs.append(float(np.linalg.norm(dT[:3, 3])))
    raw_bytes = int(np.mean([ps.array.nbytes + pt.array.nbytes for ps, pt in pins]))
    metric, unit, hib, scaling = METRICS["pair"]
    line = {
        "metric": metric, "value": value, "unit": unit, "n_gpus": ctx.world, "steps": args.steps,
        "warmup": W, "ms_per_step": total_ms / args.steps, "higher_is_better": hib, "scaling": scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": pair_config(ns_l, nt_l),
        "icp_iterations_per_pair": [int(x) for x in it_l],
        "details": {"n_src_raw": [int(len(p[1])) for p in pairs], "n_tgt_raw": [int(len(p[0])) for p in pairs],
                    "l2": "flushed before every step (256 MiB memset outside the per-step events); consecutive steps work "
                          "on different pairs",
                    "gpu": ctx.info["name"], "sm_count": ctx.info["sm_count"], "host_sync": sync_mode,
                    "host_cores": os.cpu_count(), "pose_error_vs_gt_m": errs},
        "ms_per_iter": kern_ms,
        "align_loop_ms": float(np.mean(loop_ms)),
        "latency_ms_per_pair": serial_ms / args.steps,
        "step_spread": {"value": value_spread, "e2e": e2e_spread,
                        "note": "host-observed time between consecutive results of the pipelined runs"},
        "pipeline": "value / e2e: two pairs in flight (both feeder chains of pair s+1 on two queues while the align of pair "
                    "s runs on a third), CUDA events around the K steps; latency_ms_per_pair, ms_per_iter and roofline: one "
                    "pair at a time, L2 flushed before every step, events around every step / align launch",
        "wall_s": wall,
        "e2e": {"value": e2e, "unit": unit, "h2d_bytes_per_step": raw_bytes,
                "d2h_bytes_per_step": 428 + 2 * 8 + 4 * 8,
                "note": "streaming: the H2D of pair s+2 (copy queue, three buffer sets) and the feeder chains of pair s+1 "
                        "overlap the align of pair s; every step copies its own raw points in as packed xyz (12 B per point, ~49 MB, "
                        "expanded to xyz1 on the device) and reads its result struct, voxel counts and index-build scalars back"},
        "gpu_launches": int(gpu_launches),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": "align_batch_kernel<GICP> (persistent cooperative launch: nearest neighbour + "
                                                 "linearise + reduce + solve, every iteration of one align in one launch)",
                     "achieved": achieved, "peak": ctx.peak_hbm, "unit": "GB/s", "frac": achieved / ctx.peak_hbm,
                     "traffic": traffic,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy, of measured)" if ctx.peaks
                     else "fallback 6650 (of fallback)",
                     "algorithmic_bytes_per_launch": alg_total / max(launches, 1), "launch_ms": launch_ms,
                     "iterations_per_launch": iters_done / max(launches, 1),
                     "note": "algorithmic bytes = iterations x (192 N_s + 16 N_t); the 120k working set is "
                             "L2-resident (SURVEY fact 3), so the kernel is latency-bound and the HBM fraction is "
                             "small by construction (the HBM-sized evidence is extras.config5 / extras.config4); CUDA "
                             "events on the queue's stream around each launch"},
    }
    del pipe
    return line, pairs, outputs


def last_step_outputs(pipe):
    """What the last timed step handed its caller, as host arrays: both voxelised clouds with their covariances, the
    k-NN lists the covariances were estimated from, and every field of the registration result."""
    src, tgt, _, res, nn_s, nn_t = pipe.last
    out = {}
    for name, cloud, nn in (("source", src, nn_s), ("target", tgt, nn_t)):
        out[f"{name}_points"] = cloud.points_host()
        out[f"{name}_covs"] = cloud.covs_host()
        out[f"{name}_knn_indices"] = nn.indices_host()
        out[f"{name}_knn_sq_distances"] = nn.distances_host()
    for f in dataclasses.fields(res):
        if getattr(res, f.name) is not None:
            out[f"result_{f.name}"] = np.asarray(getattr(res, f.name))
    return out


def dump_outputs(path, arrays):
    """--dump-outputs: every array as <path>/<name>.npy in float32, or in float64 for integer and boolean data (which
    float64 holds exactly).  Should the whole exceed DUMP_BYTES, every array of more than 4096 rows is cut to a fixed,
    seeded sample of its rows (the same rows for arrays of the same length)."""
    out = {k: np.asarray(v, np.float64 if np.asarray(v).dtype.kind in "biu" else np.float32) for k, v in arrays.items()}
    big = [k for k, a in out.items() if a.ndim and len(a) > 4096]
    small_bytes = sum(a.nbytes for k, a in out.items() if k not in big)
    big_bytes = sum(out[k].nbytes for k in big)
    if small_bytes + big_bytes > DUMP_BYTES:
        keep = (DUMP_BYTES - small_bytes) / big_bytes
        for k in big:
            n = len(out[k])
            out[k] = out[k][np.sort(np.random.default_rng(n).choice(n, int(n * keep), replace=False))]
    os.makedirs(path, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(path, k + ".npy"), a)


def add_cpu_baseline(line, pairs):
    oracle, cores, build = timing_oracle()
    t0 = time.perf_counter()
    n_cpu = 0
    r = None
    while n_cpu < 1 or (time.perf_counter() - t0 < 10.0 and n_cpu < N_ROTATE):
        tgt_raw, src_raw, _ = pairs[n_cpu % N_ROTATE]
        r, _, _ = cpu_pair(oracle, src_raw, tgt_raw)
        n_cpu += 1
    dt = time.perf_counter() - t0
    line["cpu_baseline"] = {"value": n_cpu / dt, "unit": "pairs/s", "cores": cores, "kind": "port",
                            "sample": f"{n_cpu} whole pair(s), full pipeline, oracle port ({build}) on {cores} threads",
                            "ms_per_pair": 1e3 * dt / n_cpu, "icp_iterations": r['iterations'] + 1}


# ------------------------------------------------------------------ config 5: batched pairs inside one GPU
def make_batch_inputs(ctx, P, scenes=4):
    """P raw scan pairs: `scenes` synthetic scenes (8 accumulated sweeps, ~1.0 M raw points -> ~64 k after the
    voxel grid), every pair its own random motion (|t| <= 0.6 m, <= 1 deg) and its own random 90 % subsample of the
    scene as the source; every pair gets its OWN copy of the target in device memory (independent pairs: nothing
    is shared or de-duplicated).  Host arrays are kept for the end-to-end leg."""
    rs = np.random.RandomState(1000 + ctx.rank)
    base = []
    for s in range(scenes):
        kw = dict(sweeps=1, azimuth_steps=256) if TINY else dict(sweeps=8)
        tgt_raw, _, _ = synthetic.kitti_pair(100 + scenes * ctx.rank + s, **kw)
        base.append(tgt_raw)
    host = []
    for j in range(P):
        tgt_raw = base[j % scenes]
        T = synthetic.random_pose(rs, 0.6, 1.0)
        keep = tgt_raw[rs.rand(len(tgt_raw)) < 0.9].astype(np.float64)
        src_raw = (keep @ np.linalg.inv(T).T).astype(np.float32)
        src_raw[:, 3] = 1.0
        host.append((src_raw, tgt_raw, T))
    return host


def odometry_params(pl, spx):
    """settings of the odometry extra (and of tests/test_gpu_odometry.py): 0.4 m voxel grid -> 8000 points, GICP + Huber
    against a 0.5 m VoxelHashMap submap, 3000-point registration sampling"""
    P = pl.Parameters()
    P.submap.map_type = pl.SubmapMapType.VOXEL_HASH_MAP
    P.submap.voxel_size = 0.5
    P.submap.point_random_sampling_num = 6000
    P.submap.max_distance_range = 60.0
    P.submap.keyframe.distance_threshold = 0.3
    P.scan.downsampling.polar.enable = False
    P.scan.downsampling.voxel.enable = True
    P.scan.downsampling.voxel.size = 0.4
    P.scan.downsampling.random.num = 8000
    P.scan.preprocess.box_filter.min = 1.0
    P.scan.preprocess.box_filter.max = 80.0
    P.registration.factor.robust.type = spx.RobustLossType.HUBER
    P.registration.factor.robust.default_scale = 1.0
    P.registration_sampling.num = 3000
    return P


def workload_odometry(ctx, frames=30, warm=5):
    """SURVEY.md §8(f) rank 2, the production caller of the path: LiDAROdometryPipeline::process on a synthetic drive
    (one 64 x 1024 revolution per frame; raw scans resident, as a driver would have uploaded them).  frames/s over the
    frames after `warm`, host clock around the loop (every process() ends with its result on the host)."""
    from sycl_points_b200 import pipeline as pl
    spx, q = ctx.spx, ctx.q
    poses, scans = synthetic.drive(frames if not TINY else 4, azimuth_steps=1024 if not TINY else 256)
    P = odometry_params(pl, spx)
    P.initial_pose = poses[0]
    pipe = pl.LiDAROdometryPipeline(P, q)
    clouds = [spx.PointCloudShared(q, s) for s in scans]
    q.wait()
    worst, t0 = 0.0, None
    warm = min(warm, len(scans) - 1)
    for k in range(len(scans)):
        if k == warm:
            q.wait()
            t0 = time.perf_counter()
        rc = pipe.process(clouds[k], 0.1 * k)
        if rc not in (pl.ResultType.first_frame, pl.ResultType.success):
            raise RuntimeError(f"odometry frame {k}: {pipe.get_error_message()}")
        worst = max(worst, float(np.linalg.norm(pipe.get_odom()[:3, 3] - poses[k][:3, 3])))
    q.wait()
    dt = time.perf_counter() - t0
    n = len(scans) - warm
    med = {name: float(np.median(v[warm:])) for name, v in pipe.get_total_processing_times().items() if len(v) > warm}
    return {"frames_per_s": n / dt, "ms_per_frame": 1e3 * dt / n, "frames_timed": n, "points_per_scan": int(len(scans[0])),
            "worst_position_error_m": worst, "keyframes": len(pipe.get_keyframe_poses()),
            "submap_points": int(pipe.get_submap_point_cloud().size()), "stage_median_ms": med}


def workload_batch(ctx, steps, warmup, P=64, e2e_steps=None, lanes=0):
    spx, q = ctx.spx, ctx.q
    host = make_batch_inputs(ctx, P)
    dev = [(spx.PointCloudShared(q, s), spx.PointCloudShared(q, t), None) for s, t, _ in host]
    params = spx.RegistrationParams()
    params.robust.type = spx.RobustLossType.HUBER
    params.robust.default_scale = 10.0
    if lanes <= 0:
        lanes = max(2, min(8, (os.cpu_count() or 8) // max(1, min(ctx.world, 8))))
    ba = spx.BatchAligner(q, params, VOXEL, K_COV, lanes=lanes)
    for _ in range(max(warmup, 1)):
        res, ns, nt = ba.align(dev)
    a, b = spx.Event(), spx.Event()
    ctx.barrier()
    ctx.l2_flush()
    l0 = spx.kernel_launch_count()
    align_ms, iters = [], []
    a.record(q)
    for _ in range(steps):
        res, ns, nt = ba.align(dev)
        t = ba.last_timing()
        align_ms.append(t["align_ms"])
    b.record(q)
    ctx.barrier()
    launches = spx.kernel_launch_count() - l0
    total_ms = a.elapsed_ms(b)
    # end to end: every step uploads its 2P raw clouds from pinned host memory and reads the P results back
    e2e_ms, h2d = None, int(sum(s.nbytes + t.nbytes for s, t, _ in host))
    if e2e_steps:
        pins = []
        for s, t, _ in host:
            ps, pt = spx.PinnedArray(s.shape), spx.PinnedArray(t.shape)
            ps.array[...] = s
            pt.array[...] = t
            pins.append((ps, pt))
        L = spx.lib()
        c, d = spx.Event(), spx.Event()
        ctx.barrier()
        c.record(q)
        for _ in range(e2e_steps):
            for (ps, pt), (ds, dt_, _) in zip(pins, dev):
                spx._lib.check(L.spx_memcpy_h2d(q.handle, ds.points.ptr, ps.array.ctypes.data, ps.array.nbytes))
                spx._lib.check(L.spx_memcpy_h2d(q.handle, dt_.points.ptr, pt.array.ctypes.data, pt.array.nbytes))
            ba.align(dev)
        d.record(q)
        ctx.barrier()
        e2e_ms = c.elapsed_ms(d)
        del pins
    total_ms, = ctx.max_over_ranks(total_ms)
    its = np.array([r.iterations + 1 for r in res])
    errs = [float(np.linalg.norm((np.linalg.inv(T) @ r.T.astype(np.float64))[:3, 3])) for (_, _, T), r in zip(host, res)]
    point_iters = float(np.sum(ns.astype(np.float64) * its))
    alg = 192.0 * point_iters + 16.0 * float(nt.sum())  # per batched launch (SURVEY.md §8(d))
    kern_ms = float(np.median(align_ms))
    out = {
        "pairs_per_s": ctx.world * P * steps / (total_ms * 1e-3), "ms_per_batch": total_ms / steps, "pairs_per_batch": P,
        "lanes": lanes, "n_src_mean": float(ns.mean()), "n_tgt_mean": float(nt.mean()), "iterations_mean": float(its.mean()),
        "iterations_max": int(its.max()), "align_kernel_ms": kern_ms,
        "align_us_per_pair_iteration": 1e3 * kern_ms / float(its.sum()),
        "align_algorithmic_gbs": alg / (kern_ms * 1e-3) / 1e9, "align_frac_of_hbm_peak": alg / (kern_ms * 1e-3) / 1e9 / ctx.peak_hbm,
        "converged": int(sum(r.converged for r in res)), "pose_error_vs_gt_m_max": max(errs),
        "gpu_launches_per_batch": launches / steps, "h2d_bytes_per_batch": h2d,
    }
    if e2e_ms is not None:
        e2e_ms, = ctx.max_over_ranks(e2e_ms)
        out["e2e_pairs_per_s"] = ctx.world * P * e2e_steps / (e2e_ms * 1e-3)
    ba.close()
    return out


# ------------------------------------------------------------------ config 3: KNN, queries sharded
def workload_knn(ctx, steps, warmup, method, nq=1_000_000, nt=1_000_000, k=20, e2e=False):
    spx, q = ctx.spx, ctx.q
    from sycl_points_b200.multi_gpu import shard_of
    if TINY:
        nq = nt = 4096
    Qh, Th = synthetic.knn_config3(nq, nt)
    lo, hi = shard_of(nq, ctx.rank, ctx.world)
    Q, T = spx.PointCloudShared(q, Qh[lo:hi]), spx.PointCloudShared(q, Th)
    res = spx.KNNResult()
    tree = None
    build_ms = None
    if method == "index":
        a, b = spx.Event(), spx.Event()
        tree = spx.KDTree.build(q, T)
        tree.close()
        q.wait()
        a.record(q)
        tree = spx.KDTree.build(q, T)
        b.record(q)
        build_ms = a.elapsed_ms(b)

    def once():
        if method == "index":
            tree.knn_search_async(Q, k, res)
            return res
        return spx.knn_search_bruteforce(q, Q, T, k)

    for _ in range(max(warmup, 1)):
        r = once()
    a, b = spx.Event(), spx.Event()
    ctx.barrier()
    l0 = spx.kernel_launch_count()
    a.record(q)
    for _ in range(steps):
        r = once()
    b.record(q)
    ctx.barrier()
    launches = spx.kernel_launch_count() - l0
    ms, = ctx.max_over_ranks(a.elapsed_ms(b) / steps)
    out = {"method": method, "nq": nq, "nt": nt, "k": k, "ms": ms, "mqueries_per_s": nq / ms / 1e3, "queries_per_rank": hi - lo,
           "gpu_launches_per_search": launches / steps,
           "algorithmic_gbs": (16.0 * nq + 16.0 * nt * ctx.world + 8.0 * k * nq) / (ms * 1e-3) / 1e9}
    if method == "bruteforce":
        pairs = float(nq) * nt
        out["gpair_per_s"] = pairs / ms / 1e6
        # FP32 issue floor: the kernel evaluates two queries per packed f32x2 instruction: 3 sub + 1 mul + 2 fma per
        # pair of pairs + 1 compare per pair = 4 lane-instructions per pair, 148 SM x 128 lanes x clock
        lane_rate = ctx.info["sm_count"] * 128 * 1.965e9 * ctx.world
        out["frac_of_fp32_issue_floor_packed4"] = pairs * 4.0 / lane_rate / (ms * 1e-3)
        out["frac_of_fp32_issue_floor_scalar7"] = pairs * 7.0 / lane_rate / (ms * 1e-3)
    if build_ms is not None:
        out["index_build_ms"] = build_ms
    if e2e:
        pq, pt = spx.PinnedArray(Qh[lo:hi].shape), spx.PinnedArray(Th.shape)
        pq.array[...] = Qh[lo:hi]
        pt.array[...] = Th
        L = spx.lib()
        c, d = spx.Event(), spx.Event()
        ctx.barrier()
        c.record(q)
        for _ in range(steps):
            spx._lib.check(L.spx_memcpy_h2d(q.handle, Q.points.ptr, pq.array.ctypes.data, pq.array.nbytes))
            spx._lib.check(L.spx_memcpy_h2d(q.handle, T.points.ptr, pt.array.ctypes.data, pt.array.nbytes))
            if method == "index":
                tree.close()
                tree = spx.KDTree.build(q, T)
            r = once()
            r.indices_host()
            r.distances_host()
        d.record(q)
        ctx.barrier()
        e_ms, = ctx.max_over_ranks(c.elapsed_ms(d) / steps)
        out["e2e_mqueries_per_s"] = nq / e_ms / 1e3
        out["e2e_h2d_bytes"] = int(pq.array.nbytes + pt.array.nbytes)
        out["e2e_d2h_bytes"] = int((hi - lo) * k * 8)
    if tree is not None:
        tree.close()
    return out


# ------------------------------------------------------------------ config 4: dense pair, source sharded
def workload_align_sharded(ctx, reps, iters=20, factors=("GICP",)):
    spx, q = ctx.spx, ctx.q
    from sycl_points_b200.multi_gpu import Communicator, ShardedRegistration, shard_indices
    if TINY:
        tgt_raw, src_raw, T_gt = synthetic.kitti_pair(42, sweeps=1, azimuth_steps=256)
        voxel, cap = 0.25, 10**9
    else:
        tgt_raw, src_raw, T_gt = synthetic.dense_pair(42)
        voxel, cap = 0.05, 2_000_000
    vg = spx.VoxelGrid(q, voxel)
    src_full = vg.downsampling(spx.PointCloudShared(q, src_raw)).points_host()[:cap]
    tgt_full = vg.downsampling(spx.PointCloudShared(q, tgt_raw)).points_host()[:cap]
    del src_raw, tgt_raw
    src, tgt = spx.PointCloudShared(q, src_full), spx.PointCloudShared(q, tgt_full)
    ts, tt = spx.KDTree.build(q, src), spx.KDTree.build(q, tgt)
    spx.covariance.estimate(ts.knn_search(src, K_COV), src)
    nn_t = tt.knn_search(tgt, K_COV)
    spx.covariance.estimate(nn_t, tgt)
    spx.covariance.estimate_normals(nn_t, tgt)
    ts.close()
    ns, nt = src.size(), tgt.size()
    sel = shard_indices(ns, ctx.rank, ctx.world)
    shard = spx.PointCloudShared(q, src_full[sel], src.covs_host()[sel]) if ctx.world > 1 else src
    comm = Communicator(q, ctx.rank, ctx.world) if ctx.world > 1 else None
    out = {"n_src": ns, "n_tgt": nt, "iterations": iters, "shard_points": int(len(sel))}
    for name, per_pt in (("POINT_TO_PLANE", 80), ("GICP", 192)):
        if name not in factors:
            continue
        params = spx.RegistrationParams(reg_type=spx.RegType[name], max_iterations=iters)
        params.robust.type = spx.RobustLossType.HUBER
        params.criteria.translation = params.criteria.rotation = 0.0
        if ctx.world > 1:
            reg = ShardedRegistration(q, params, comm=comm, mode="p2p")
            run = lambda: reg.align(shard, tgt, tt)  # noqa: E731
        else:
            reg = spx.Registration(q, params)
            run = lambda: reg.align(src, tgt, tt)  # noqa: E731
        res = run()
        ms = []
        for _ in range(reps):
            ctx.barrier()
            res = run()
            ms.append(ctx.max_over_ranks(reg.last_timing()["loop_ms"])[0])
        per_iter = float(np.median(ms)) / iters
        alg = per_pt * ns + 16 * nt
        dT = np.linalg.inv(T_gt.astype(np.float64)) @ res.T.astype(np.float64)
        out[name] = {"ms_per_iter": per_iter, "algorithmic_gbs": alg / (per_iter * 1e-3) / 1e9,
                     "frac_of_hbm_peak_per_gpu": alg / (per_iter * 1e-3) / 1e9 / (ctx.peak_hbm * ctx.world),
                     "exchange": "in-kernel NVLink mailbox (store row -> flag -> fold in rank order)" if ctx.world > 1 else "none (1 GPU)",
                     "pose_error_vs_gt_m": float(np.linalg.norm(dT[:3, 3])), "inlier": int(res.inlier)}
    tt.close()
    return out


# ------------------------------------------------------------------ output
_JSON_FD = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries loaded later write there too (NCCL prints its
    version banner on fd 1), so fd 1 is pointed at stderr for the whole run and the line goes out
    through a saved duplicate of the original stdout."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def generic_line(ctx, workload, value, ms_per_step, steps, warmup, extra):
    metric, unit, hib, scaling = METRICS[workload]
    line = {"metric": metric, "value": value, "unit": unit, "n_gpus": ctx.world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": hib, "scaling": scaling, "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": WORKLOADS[workload]}}
    line.update(extra)
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="spx", choices=["spx", "reference"])
    ap.add_argument("--workload", default="pair", choices=list(WORKLOADS))
    ap.add_argument("--pairs", type=int, default=64, help="pairs per batch and rank (--workload batch)")
    ap.add_argument("--lanes", type=int, default=0, help="feeder lanes of spx_align_batch (0 = from the host's cores)")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (--workload pair)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "spx" or args.workload != "pair"):
        ap.error("--dump-outputs needs --impl spx --workload pair")
    claim_stdout()
    ctx = Ctx(args)

    if args.impl == "reference":
        run_reference(ctx)
        return
    ctx.init_gpu()
    W = max(args.warmup, 3)
    if args.workload == "pair":
        line, pairs, outputs = workload_pair(ctx)
        if outputs is not None and ctx.rank == 0:
            dump_outputs(args.dump_outputs, outputs)
        if not args.no_extras:
            extras = {}
            t0 = time.perf_counter()
            try:
                extras["config3_knn_index"] = workload_knn(ctx, 5, 2, "index")
                extras["config3_knn_bruteforce"] = workload_knn(ctx, 1, 1, "bruteforce")
                extras["config5_batch"] = workload_batch(ctx, 3, 1, P=64, lanes=args.lanes)
                extras["config4_align_sharded"] = workload_align_sharded(ctx, 3)
                if ctx.rank == 0:
                    extras["odometry_loop"] = workload_odometry(ctx)
            except Exception as e:  # the headline line must go out whatever happens to an extra
                extras["error"] = repr(e)
            extras["seconds"] = time.perf_counter() - t0
            line["extras"] = extras
        if ctx.rank == 0 and ctx.world == 1 and not args.no_cpu_baseline:
            add_cpu_baseline(line, pairs)
    elif args.workload == "batch":
        r = workload_batch(ctx, args.steps, W, P=args.pairs, e2e_steps=args.steps, lanes=args.lanes)
        line = generic_line(ctx, "batch", r["pairs_per_s"], r["ms_per_batch"], args.steps, W, {
            "config": {"workload": WORKLOADS["batch"], "pairs_per_batch": args.pairs, "n_src_mean": r["n_src_mean"],
                       "n_tgt_mean": r["n_tgt_mean"], "iterations_mean": r["iterations_mean"]},
            "e2e": {"value": r.get("e2e_pairs_per_s"), "unit": "pairs/s", "h2d_bytes_per_step": r["h2d_bytes_per_batch"],
                    "d2h_bytes_per_step": 428 * args.pairs},
            "gpu_launches": int(r["gpu_launches_per_batch"] * args.steps),
            "roofline": {"bound": "hbm", "kernel": "align_batch_kernel<GICP> (one launch for all pairs of a batch)",
                         "achieved": r["align_algorithmic_gbs"], "peak": ctx.peak_hbm, "unit": "GB/s",
                         "frac": r["align_frac_of_hbm_peak"], "traffic": None, "launch_ms": r["align_kernel_ms"]},
            "details": r})
    elif args.workload in ("knn_index", "knn_bf"):
        method = "index" if args.workload == "knn_index" else "bruteforce"
        r = workload_knn(ctx, args.steps, W if method == "index" else 1, method, e2e=True)
        line = generic_line(ctx, args.workload, r["mqueries_per_s"], r["ms"], args.steps, W, {
            "e2e": {"value": r.get("e2e_mqueries_per_s"), "unit": "Mqueries/s", "h2d_bytes_per_step": r.get("e2e_h2d_bytes"),
                    "d2h_bytes_per_step": r.get("e2e_d2h_bytes")},
            "gpu_launches": int(r["gpu_launches_per_search"] * args.steps),
            "roofline": {"bound": "hbm", "kernel": "grid_knn_reg_*<20>" if method == "index" else "knn_bruteforce_kernel<2,packed,TMA-staged,batch 2>",
                         "achieved": r["algorithmic_gbs"], "peak": ctx.peak_hbm * ctx.world, "unit": "GB/s",
                         "frac": r["algorithmic_gbs"] / (ctx.peak_hbm * ctx.world), "traffic": None,
                         "note": "the brute force is FP32-issue bound and the index L2-latency bound (SURVEY.md §8(d)); see details"},
            "details": r})
    else:
        r = workload_align_sharded(ctx, args.steps, factors=("POINT_TO_PLANE", "GICP"))
        g = r["GICP"]
        line = generic_line(ctx, "align_sharded", g["ms_per_iter"], g["ms_per_iter"] * r["iterations"], args.steps, 1, {
            "config": {"workload": WORKLOADS["align_sharded"], "n_src": r["n_src"], "n_tgt": r["n_tgt"]},
            "roofline": {"bound": "hbm", "kernel": "align_gn_kernel<GICP,sharded> / split search + linearize kernels (1 GPU)",
                         "achieved": g["algorithmic_gbs"], "peak": ctx.peak_hbm * ctx.world, "unit": "GB/s",
                         "frac": g["frac_of_hbm_peak_per_gpu"], "traffic": None},
            "details": r})
    if ctx.rank == 0:
        emit(line)
    if ctx.dist is not None:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()

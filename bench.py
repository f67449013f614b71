#!/usr/bin/env python
"""bench.py -- NICP 640x480 alignments/s on 1/2/4/8 B200 (BASELINE.json metric).

Workload (config 4 of BASELINE.json, the one the metric's multi-GPU numbers are quoted on):
batched loop-closure candidate verification of 8192 independent 640x480 frame pairs per step
(64 "current" frames x 128 candidate "reference" frames, guesses perturbed by U(+-5 cm, +-3 deg),
10 outer iterations, parameters of pwn_core/conf/pwn_aligner_1_1.conf).  The pairs are sharded over the
ranks as rectangular blocks of the current x candidate grid (shard_grid: 1x2, 2x2, 2x4 blocks at 2, 4, 8
ranks, so that a rank prepares as few frames as possible; current-major inside a block; SURVEY.md 8e):
the total work is fixed, scaling is strong.

One JSON line on rank 0:
  value     whole-job alignments/s with the clouds already resident in HBM (device-timed, CUDA events
            on the library's stream, max over ranks)
  e2e       the same metric through the C-ABI with HOST buffers: every step uploads the raw 16-bit
            depth frames the rank needs from pinned memory (192 at N = 1, 64 at N = 8), builds their clouds, aligns
            its pairs and reads the 256-byte result records back
  configs   (N = 1) BASELINE configs 1, 2, 3, 5 through tools/bench_configs.py, each with its own CPU sample
  roofline  the fused correspondence+linearise kernel: algorithmic bytes / live CUDA-event time
  cpu_baseline  the CPU oracle (restatement of pwn_core; the reference itself cannot be built here)
            timed on this box's host cores on a bounded sample of the same workload

`--impl reference` times the CPU path only (rank 0), same metric/config.
`--dump-outputs DIR` writes the result records of the last timed step (one per pair, 2 MB at the default 8192 pairs),
one .npy per field, in the job's pair order whatever the number of GPUs; the workload is seeded, so two builds run with
the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ROWS, COLS = 480, 640
CONF = dict(minD=0.5, maxD=4.5, minImageRadius=10, maxImageRadius=30, minPoints=50, curvatureThreshold=0.2,
            worldRadius=0.1, omegaCurvatureThreshold=0.02, inlierDistanceThreshold=1.0,
            inlierNormalAngularThreshold=0.95, inlierCurvatureRatioThreshold=1.3, flatCurvatureThreshold=0.02,
            inlierMaxChi2=9000.0, outerIterations=10, innerIterations=1)
METRIC = "nicp_640x480_alignments_per_s"
UNIT = "alignments/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--currents", type=int, default=64, help="current frames of the whole job (sharded over the ranks)")
    ap.add_argument("--candidates", type=int, default=128, help="candidate frames every current is verified against")
    ap.add_argument("--no-configs", action="store_true", help="skip the configs block (BASELINE configs 1, 2, 3, 5)")
    ap.add_argument("--tracking-frames", type=int, default=2000)
    ap.add_argument("--cpu-sample-pairs", type=int, default=12)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-threads", type=int, default=0, help="threads of the CPU arm (0 = all host cores)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result records of the last timed step as DIR/<field>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU path (--impl ours)")
    return args


DUMP_MAX_BYTES = 64 << 20


def job_pair_ids(n_cur, n_cand, world):
    """the job's pair index (current-major over the current x candidate grid) of every record, in the order the ranks'
    blocks are gathered (rank-major, current-major inside a block)"""
    split_cur, split_cand = shard_grid(n_cur, n_cand, world)
    bc, bk = n_cur // split_cur, n_cand // split_cand
    ids = [(r // split_cand * bc + ci) * n_cand + r % split_cand * bk + ri
           for r in range(world) for ci in range(bc) for ri in range(bk)]
    return np.array(ids, np.int64)


def dump_outputs(records, pair_ids, out_dir):
    """One .npy per field of the RESULT_DTYPE records (include/nicp_b200.h: nicp_align_result), rows in the job's pair
    order (pair_ids: the pair index of each record), so that runs on any number of GPUs line up.  T and omega stay
    column-major as the C-ABI returns them; integer fields are stored as float64, which holds them exactly.  `reserved`
    holds the kernels' work counters, not a result, and is left out.  A job whose records would exceed DUMP_MAX_BYTES is
    written as a fixed, seeded sample of pairs, listed in pair_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    records = records[np.argsort(pair_ids)]
    names = [n for n in records.dtype.names if n != "reserved"]
    per_record = sum(8 * int(np.prod(records.dtype[n].shape, dtype=np.int64)) for n in names)
    if len(records) * per_record > DUMP_MAX_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(len(records), DUMP_MAX_BYTES // per_record - 1, replace=False))
        records = records[keep]
        np.save(os.path.join(out_dir, "pair_index.npy"), keep.astype(np.float64))
    for name in names:
        a = records[name]
        a = a.astype(np.float64) if a.dtype.kind in "iu" else a.astype(np.float32)
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


# ---------------------------------------------------------------------------------------------------
def _render(args):
    from g2o_frontend_b200 import synth
    pose, seed = args
    return synth.render_depth_u16(pose, ROWS, COLS, seed=seed)


def render_frames(jobs, procs=None):
    """(pose, seed) -> raw 16-bit frames; a process pool when there are many (0.1 s per frame in numpy)"""
    procs = procs or min(os.cpu_count() or 1, 32)
    if procs > 1 and len(jobs) >= 32:
        import multiprocessing as mp
        with mp.get_context("fork").Pool(procs) as pool:
            return pool.map(_render, jobs, chunksize=4)
    return [_render(j) for j in jobs]


def make_workload(n_cur, n_cand, rank, cur_slice=None, procs=None, cand_slice=None):
    """poses + raw frames + pair list + guesses (deterministic in `rank`, the seed of the job).  cur_slice = (lo, hi) /
    cand_slice = (lo, hi): only those currents / candidates are rendered and paired (a rank's block of the job's
    current x candidate grid); pair indices are relative to the slices."""
    from g2o_frontend_b200 import synth
    rng = np.random.default_rng(1000 + rank)
    cur_poses = [synth.perturbed_pose(rng, np.eye(4), 0.25, 6.0) for _ in range(n_cur)]
    cand_poses = [synth.perturbed_pose(rng, np.eye(4), 0.25, 6.0) for _ in range(n_cand)]
    lo, hi = cur_slice if cur_slice else (0, n_cur)
    clo, chi = cand_slice if cand_slice else (0, n_cand)
    frames = render_frames([(cur_poses[i], 10 * rank + i) for i in range(lo, hi)] +
                           [(cand_poses[i], 5000 + 10 * rank + i) for i in range(clo, chi)], procs)
    raws_cur, raws_cand = frames[:hi - lo], frames[hi - lo:]
    pairs, guesses = [], []
    for ci, cp in enumerate(cur_poses):
        for ri, rp in enumerate(cand_poses):
            T_true = np.linalg.inv(rp) @ cp  # reference <- current
            g = synth.perturbed_pose(rng, T_true, 0.05, 3.0)  # drawn for every pair so that a shard sees the job's guesses
            if lo <= ci < hi and clo <= ri < chi:
                guesses.append(g)
                pairs.append((ri - clo, ci - lo))
    return raws_cur, raws_cand, np.array(pairs), np.stack(guesses).astype(np.float32)


def shard_grid(n_cur, n_cand, world):
    """The job's current x candidate grid cut into `world` rectangular blocks (a splits of the currents x b of the
    candidates, a b = world) so that a rank prepares as few frames as possible: its n_cur / a currents and n_cand / b
    candidates.  Pairs that share a current cloud stay contiguous inside a block (SURVEY.md 8e)."""
    best = None
    for a in range(1, world + 1):
        if world % a:
            continue
        b = world // a
        if n_cur % a or n_cand % b:
            continue
        frames = n_cur // a + n_cand // b
        if best is None or frames < best[0] or (frames == best[0] and a > best[1]):
            best = (frames, a, b)
    if best is None:
        raise SystemExit("--currents (%d) x --candidates (%d) cannot be cut into %d equal blocks" % (n_cur, n_cand, world))
    return best[1], best[2]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)"""

    def __init__(self, indices):
        """indices: the GPUs to watch (one nvidia-smi process for all of them, started by rank 0 only); None = off"""
        self.index = None if indices is None else ",".join(str(i) for i in indices)
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        if self.index is None:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.index, "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------------
def cpu_reference_run(steps, warmup, sample_pairs, n_threads=None):
    """The reference arm: the CPU restatement of pwn_core (oracle, performance build: the reference's
    own flags + OpenMP) on this box's host cores.  Each step = 1 cloud build from a raw frame +
    `sample_pairs` alignments (the workload's ratio of 80 cloud builds per 1024 alignments)."""
    from oracle import pwn_oracle as O
    from g2o_frontend_b200 import synth
    cores = n_threads or os.cpu_count() or 1
    # the finder drops rows % numThreads (correspondencefinder.cpp:38): use a divisor of 480
    while ROWS % cores:
        cores -= 1
    # through the library (omp_set_num_threads), not the environment: libgomp reads OMP_NUM_THREADS once, when it is
    # loaded, and torch.distributed.run exports OMP_NUM_THREADS=1 to every rank; `cores` is what the team really has
    cores = O.set_threads(cores, fast=True)
    raws_cur, raws_cand, pairs, guesses = make_workload(1, sample_pairs, 0)
    K = synth.K_KINECT
    sp = O.default_stats_params(minImageRadius=CONF["minImageRadius"], maxImageRadius=CONF["maxImageRadius"],
                                minPoints=CONF["minPoints"], curvatureThreshold=CONF["curvatureThreshold"],
                                worldRadius=CONF["worldRadius"], omegaCurvatureThreshold=CONF["omegaCurvatureThreshold"])
    cp = O.default_corr_params(inlierDistanceThreshold=CONF["inlierDistanceThreshold"],
                               inlierNormalAngularThreshold=CONF["inlierNormalAngularThreshold"],
                               flatCurvatureThreshold=CONF["flatCurvatureThreshold"],
                               inlierCurvatureRatioThreshold=CONF["inlierCurvatureRatioThreshold"])

    def build(raw):
        d = O.depth_u16_to_f32(raw, fast=True)
        return O.depth_to_cloud(d, K, CONF["minD"], CONF["maxD"], sp, fast=True)[0]

    cur = build(raws_cur[0])
    cands = [build(r) for r in raws_cand]
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        cur = build(raws_cur[0])  # the step's share of cloud building
        for j, (ri, ci) in enumerate(pairs):
            ap = O.make_align_params(K, ROWS, COLS, CONF["minD"], CONF["maxD"], cp, guess=guesses[j],
                                     max_chi2=CONF["inlierMaxChi2"], num_threads=cores)
            O.align(cands[ri], cur, ap, fast=True, want_trace=False)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    total = float(np.sum(times))
    value = sample_pairs * len(times) / total
    return value, cores, total / len(times) * 1e3


def cpu_reference_sources_run(sample_pairs, n_threads=None):
    """The reference's OWN sources (g2o_frontend/pwn_core/*.cpp compiled from /root/reference against the Eigen / OpenCV
    stand-ins of oracle/shim with the reference's flags: oracle/_ref/libpwn_core_ref_fast.so) on the same bounded sample:
    1 cloud build + `sample_pairs` alignments.  Reported next to the oracle port, which is the faster of the two and stays
    the baseline (the stand-in evaluates Eigen expressions eagerly, without Eigen's SIMD).  None if the library is absent."""
    import ctypes as C
    so = os.path.join(ROOT, "oracle", "_ref", "libpwn_core_ref_fast.so")
    if not os.path.exists(so):
        return None
    from oracle import pwn_oracle as O
    from g2o_frontend_b200 import synth
    O.lib()  # liboracle.so first: the stand-in's numerical kernels resolve against it
    R = C.CDLL(so)
    R.refcore_depth_to_cloud.restype = C.c_void_p
    cores = n_threads or os.cpu_count() or 1
    while ROWS % cores:
        cores -= 1
    R.refcore_set_threads(cores)
    fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
    cm = lambda M: np.ascontiguousarray(np.asarray(M, np.float32).T.reshape(-1))
    raws_cur, raws_cand, pairs, guesses = make_workload(1, sample_pairs, 0)
    sp = np.array([CONF["worldRadius"], CONF["minImageRadius"], CONF["maxImageRadius"], CONF["minPoints"],
                   CONF["curvatureThreshold"], CONF["omegaCurvatureThreshold"]], np.float32)
    eye = cm(np.eye(4))
    K9 = cm(synth.K_KINECT)

    def build(raw):
        d = np.ascontiguousarray(O.depth_u16_to_f32(raw, fast=True), np.float32)
        return C.c_void_p(R.refcore_depth_to_cloud(fp(d), ROWS, COLS, fp(K9), C.c_float(CONF["minD"]), C.c_float(CONF["maxD"]),
                                                   fp(sp), fp(eye), None, None, None))

    cands = [build(r) for r in raws_cand]
    fpar = np.array([CONF["inlierDistanceThreshold"], CONF["inlierNormalAngularThreshold"], CONF["flatCurvatureThreshold"],
                     CONF["inlierCurvatureRatioThreshold"]], np.float32)
    T = np.zeros(16, np.float32)
    t0 = time.perf_counter()
    cur = build(raws_cur[0])
    for j, (ri, ci) in enumerate(pairs):
        R.refcore_align(cands[ri], cur, fp(K9), ROWS, COLS, C.c_float(CONF["minD"]), C.c_float(CONF["maxD"]), fp(fpar),
                        C.c_float(CONF["inlierMaxChi2"]), 1, CONF["outerIterations"], CONF["innerIterations"], fp(cm(guesses[j])),
                        fp(eye), fp(eye), None, 0, fp(T), None, None, None, None, None, None, None, None, None)
    dt = time.perf_counter() - t0
    for h in cands + [cur]:
        R.refcore_cloud_free(h)
    return {"value": sample_pairs / dt, "unit": UNIT, "cores": cores,
            "note": "g2o_frontend/pwn_core sources compiled against the Eigen/OpenCV stand-ins of oracle/shim "
                    "(-O3 -march=x86-64-v3 -fopenmp), 1 cloud build + %d alignments" % sample_pairs}


class CpuLeg:
    """The CPU oracle (performance build, all host threads) as the baseline of the secondary configurations
    (tools/bench_configs.py): cloud builds, alignments, pyramids, rig alignments.  Part of the cpu_baseline leg."""

    def __init__(self, threads=None):
        from oracle import pwn_oracle as O
        from g2o_frontend_b200 import synth
        self.O, self.synth = O, synth
        cores = threads or os.cpu_count() or 1
        while ROWS % cores:  # the finder drops rows % numThreads (correspondencefinder.cpp:38)
            cores -= 1
        self.cores = O.set_threads(cores, fast=True)

    def sp(self, minr, maxr, minp):
        return self.O.default_stats_params(minImageRadius=minr, maxImageRadius=maxr, minPoints=minp,
                                           curvatureThreshold=CONF["curvatureThreshold"], worldRadius=CONF["worldRadius"],
                                           omegaCurvatureThreshold=CONF["omegaCurvatureThreshold"])

    def cp(self, dist):
        return self.O.default_corr_params(inlierDistanceThreshold=dist,
                                          inlierNormalAngularThreshold=CONF["inlierNormalAngularThreshold"],
                                          flatCurvatureThreshold=CONF["flatCurvatureThreshold"],
                                          inlierCurvatureRatioThreshold=CONF["inlierCurvatureRatioThreshold"])

    def K(self, step):
        return self.synth.scaled_K(self.synth.K_KINECT, np.float32(1.0) / np.float32(step))

    def cloud(self, raw, step, minr, maxr, minp):
        O = self.O
        d = O.depth_u16_to_f32(raw, fast=True)
        if step > 1:
            d = O.depth_scale(d, step, fast=True)
        return O.depth_to_cloud(d, self.K(step), CONF["minD"], CONF["maxD"], self.sp(minr, maxr, minp), fast=True)[0]

    def align(self, ref, cur, step, dist, guess=None):
        O = self.O
        ap = O.make_align_params(self.K(step), ROWS // step, COLS // step, CONF["minD"], CONF["maxD"], self.cp(dist), guess=guess,
                                 max_chi2=CONF["inlierMaxChi2"], num_threads=self.cores)
        return O.align(ref, cur, ap, fast=True, want_trace=False)

    def multi_pair_align_seconds(self, cams, depthA, depthB):
        """one alignment of a MultiPointProjector rig pair (clouds prebuilt, not timed)"""
        O = self.O
        om = O.make_multi(cams)
        osp = self.sp(10, 30, 50)
        oA, oB = O.multi_depth_to_cloud(om, depthA, osp)[0], O.multi_depth_to_cloud(om, depthB, osp)[0]
        rows, cols = O.multi_image_size(om)
        oap = O.make_align_params(cams[0]["K"], rows, cols, CONF["minD"], CONF["maxD"], self.cp(1.0),
                                  max_chi2=CONF["inlierMaxChi2"], num_threads=self.cores, multi=om)
        t0 = time.perf_counter()
        O.align(oA, oB, oap, fast=True, want_trace=False)
        return time.perf_counter() - t0


def workload_config(n_cur, n_cand, world):
    """the `config` object both arms report (same workload name; the reference arm times a bounded sample of it)"""
    n_pairs = n_cur * n_cand
    P = ROWS * COLS
    split_cur, split_cand = shard_grid(n_cur, n_cand, world)
    return {"workload": "batched loop-closure candidate verification (BASELINE config 4): %d pairs/step = "
                        "%d current x %d candidate 640x480 frames, 10 outer iterations, "
                        "pwn_aligner_1_1.conf parameters" % (n_pairs, n_cur, n_cand),
            "pairs_total_per_step": n_pairs, "pairs_per_gpu_per_step": n_pairs // world, "rows": ROWS, "cols": COLS,
            "l2_policy": "inputs larger than L2 (%.1f GB of clouds + %.1f GB of z-buffers per GPU and step)" %
                         ((n_cur // split_cur + n_cand // split_cand) * P * 124 / 1e9, 256 * P * 32 / 1e9),
            "parallelism": "pair-sharded x%d (%d x %d blocks of the current x candidate grid, current-major inside a block; no "
                           "data-path collective, one all-gather of the 256-byte records)" % (world, split_cur, split_cand)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.cpu_sample_pairs
    value, cores, ms = cpu_reference_run(args.steps, args.warmup, n, args.cpu_threads or None)
    sample = ("per step: 1 cloud build from a raw 640x480 frame + %d alignments (10 iterations) of the "
              "loop-closure workload, CPU oracle performance build (-O3 -march=x86-64-v3 -fopenmp)" % n)
    try:
        ref_src = cpu_reference_sources_run(min(n, 4), args.cpu_threads or None)
    except Exception as e:  # the baseline is the port; this figure is informative
        ref_src = {"value": None, "note": "failed: %s" % e}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.currents, args.candidates, int(os.environ.get("WORLD_SIZE", "1"))),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "reference_sources": ref_src},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ---------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from g2o_frontend_b200 import capi, sharding, synth

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the NICP path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    n_cur_total, n_cand_total = args.currents, args.candidates
    # this rank's block of the job (SURVEY.md 8e): a rectangle of the current x candidate grid, so that it prepares
    # n_cur + n_cand frames for n_cur x n_cand pairs (at 8 ranks: 32 + 32 frames instead of 8 + 128)
    split_cur, split_cand = shard_grid(n_cur_total, n_cand_total, world)
    n_cur, n_cand = n_cur_total // split_cur, n_cand_total // split_cand
    rc, rk = rank // split_cand, rank % split_cand
    n_pairs = n_cur * n_cand
    n_pairs_total = n_cur_total * n_cand_total
    raws_cur, raws_cand, pairs, guesses = make_workload(n_cur_total, n_cand_total, 0, (rc * n_cur, (rc + 1) * n_cur),
                                                        procs=max(1, min(32, (os.cpu_count() or 1) // world)),
                                                        cand_slice=(rk * n_cand, (rk + 1) * n_cand))
    n_frames = n_cur + n_cand
    # pinned host staging of the raw frames (what a tracker would hand over)
    pinned = torch.empty((n_frames, ROWS, COLS), dtype=torch.int16).pin_memory()
    host_raw = pinned.numpy().view(np.uint16)
    for i, r in enumerate(raws_cur + raws_cand):
        host_raw[i] = r

    ctx = capi.Context(local_rank)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=dev)
    proj = capi.make_projector(synth.K_KINECT, ROWS, COLS, CONF["minD"], CONF["maxD"])
    sp = capi.make_stats_params(CONF["worldRadius"], CONF["minImageRadius"], CONF["maxImageRadius"], CONF["minPoints"],
                                CONF["curvatureThreshold"], CONF["omegaCurvatureThreshold"])
    ap = capi.make_align_params(CONF["inlierDistanceThreshold"], CONF["inlierNormalAngularThreshold"],
                                CONF["flatCurvatureThreshold"], CONF["inlierCurvatureRatioThreshold"],
                                CONF["inlierMaxChi2"], True, CONF["outerIterations"], CONF["innerIterations"])
    clouds = [ctx.new_cloud(ROWS * COLS) for _ in range(n_frames)]

    frames = [host_raw[i] for i in range(n_frames)]  # views of the pinned buffer: uploaded in place, no host copy

    def build_clouds():
        # one launch set per sub-batch of 8 frames (nicp_raw_depth_to_cloud_batch); asynchronous
        ctx.raw_depth_to_cloud_batch(frames, proj, sp, clouds=clouds)

    refs = [clouds[n_cur + ri] for ri, ci in pairs]
    curs = [clouds[ci] for ri, ci in pairs]
    results = np.zeros(n_pairs, capi.RESULT_DTYPE)

    def align_step():
        ctx.align_batch(refs, curs, proj, ap, guesses, results=results)
        if world > 1:
            return sharding.gather_records(results, n_pairs_total, device=dev)
        return results

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- value: clouds resident in HBM ---------------------------------------------------------
    build_clouds()
    ctx.synchronize()
    for _ in range(args.warmup):
        align_step()
    ctx.set_kernel_timing(True)
    # rank 0 watches every GPU of the job (one sampler process, not one per rank)
    sampler = ClockSampler(list(range(world)) if rank == 0 else None)
    barrier()
    launches0 = ctx.launch_count()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    sumMidx = sumMacc = 0.0
    for _ in range(args.steps):
        allrec = align_step()
        sumMidx += float(results["reserved"][:, 0].sum())
        sumMacc += float(results["reserved"][:, 1].sum())
    e1.record(stream)
    barrier()
    last_step = allrec.copy()  # the e2e leg below writes into the same buffer
    clocks = sampler.stop()
    launches = ctx.launch_count() - launches0
    dev_ms = max_over_ranks(e0.elapsed_time(e1))
    kt = ctx.kernel_timing()
    ctx.set_kernel_timing(False)
    value = n_pairs_total * args.steps / (dev_ms * 1e-3)
    ok_pairs = int((allrec["status"] == 0).sum())
    mean_inliers = float(results["inliers"].mean())

    # roofline of the fused correspondence+linearise kernel (SURVEY.md 8d algorithmic bytes)
    P = ROWS * COLS
    n_launch = max(kt["corr_lin_launches"], 1)
    bytes_total = 8.0 * P * n_pairs * args.steps * CONF["outerIterations"] + 56.0 * sumMidx + 48.0 * sumMacc
    achieved = bytes_total / (kt["corr_lin_ms"] * 1e-3) / 1e9 if kt["corr_lin_ms"] > 0 else 0.0
    peak, peak_src = measured_peak()
    # DRAM traffic per launch from the committed ncu capture of this kernel on this workload shape (256 pairs per
    # launch, 640x480); null if the launch shape differs
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        pairs_per_launch = n_pairs * args.steps * CONF["outerIterations"] / n_launch
        if abs(pairs_per_launch - tj["pairs_per_launch"]) < 0.5 and (tj["rows"], tj["cols"]) == (ROWS, COLS):
            traffic, traffic_src = tj["traffic_bytes_per_launch"], tj["source"]
    except Exception:
        pass
    roofline = {"kernel": "k_corr_lin_group<0> (CorrespondenceFinder::compute + Linearizer::update fused; one warp walks the pairs "
                          "of a group that share a current cloud)", "bound": "hbm",
                "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak,
                "frac_of_nominal_8TBs": achieved / 8000.0,
                "traffic": traffic, "traffic_source": traffic_src, "avg_launch_ms": kt["corr_lin_ms"] / n_launch,
                "launches_timed": kt["corr_lin_launches"],
                "algorithmic_bytes_per_launch": bytes_total / n_launch,
                "project_avg_launch_ms": kt["project_ms"] / max(kt["project_launches"], 1),
                "share_of_step": kt["corr_lin_ms"] / dev_ms if dev_ms > 0 else None}

    # the reference-cloud projection kernel by the same accounting (SURVEY.md 8d: 12 N + 8 P bytes per pair and iteration);
    # informative, never allowed to break the line
    try:
        sizes = [c.size() for c in clouds]
        n_ref_total = float(sum(sizes[n_cur + ri] for ri, ci in pairs))
        proj_bytes = (12.0 * n_ref_total + 8.0 * P * n_pairs) * args.steps * CONF["outerIterations"]
        if kt["project_ms"] > 0:
            roofline["project"] = {"kernel": "k_project (PinholePointProjector::project, packed 64-bit red.min z-buffer)",
                                   "achieved": proj_bytes / (kt["project_ms"] * 1e-3) / 1e9, "unit": "GB/s",
                                   "frac": proj_bytes / (kt["project_ms"] * 1e-3) / 1e9 / peak,
                                   "launches_timed": kt["project_launches"]}
    except Exception:
        pass

    # ---- e2e: host buffers in, records out, every step -------------------------------------------
    def e2e_step():
        build_clouds()
        return align_step()

    for _ in range(max(1, min(args.warmup, 2))):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record(stream)
    for _ in range(args.steps):
        e2e_step()
    f1.record(stream)
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    e2e_ms = max_over_ranks(max(f0.elapsed_time(f1), wall_ms))
    e2e_value = n_pairs_total * args.steps / (e2e_ms * 1e-3)
    h2d = n_frames * ROWS * COLS * 2 + n_pairs * 64 + n_pairs * 0
    d2h = n_pairs * 256 + n_pairs * 42 * 4

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": workload_config(n_cur_total, n_cand_total, world),
                "clocks": clocks, "gpu_launches": int(launches),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "ms_per_step": e2e_ms / args.steps},
                "roofline": roofline,
                "checks": {"pairs_ok": ok_pairs, "pairs_total": int(n_pairs_total), "mean_inliers": mean_inliers}}
        if not args.no_cpu_baseline and world == 1:
            v, cores, ms = cpu_reference_run(1, 1, args.cpu_sample_pairs)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": "1 cloud build + %d alignments (10 iterations) of the same workload, CPU "
                                              "oracle performance build, 1 warm-up + 1 timed pass" % args.cpu_sample_pairs}
            # single-thread figure (SURVEY.md 8d): a fresh process, because OpenMP reads OMP_NUM_THREADS once
            try:
                import subprocess
                env = dict(os.environ, OMP_NUM_THREADS="1")
                for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
                    env.pop(k, None)
                o = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--cpu-threads", "1",
                                    "--steps", "1", "--warmup", "0", "--cpu-sample-pairs", "2"], env=env,
                                   capture_output=True, text=True, timeout=300)
                line["cpu_baseline"]["value_1_thread"] = json.loads(o.stdout.strip().splitlines()[-1])["value"]
            except Exception:
                line["cpu_baseline"]["value_1_thread"] = None
        if world == 1 and not args.no_configs:
            # BASELINE configs 1, 2, 3 and 5 on the same context (tools/bench_configs.py), each beside its CPU sample
            try:
                sys.path.insert(0, os.path.join(ROOT, "tools"))
                import bench_configs
                for c in clouds:
                    c.close()
                line["configs"] = bench_configs.run_all(ctx, None if args.no_cpu_baseline else CpuLeg(),
                                                        tracking_frames=args.tracking_frames)
            except Exception as e:
                line["configs"] = {"error": "%s: %s" % (type(e).__name__, e)}
        if args.dump_outputs:
            dump_outputs(last_step, job_pair_ids(n_cur_total, n_cand_total, world), args.dump_outputs)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


_JSON_OUT = None


def emit(line):
    """the one JSON line, on the process's original stdout"""
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    # stdout carries exactly one JSON line: anything else a library prints on file descriptor 1 (NCCL announces its
    # version there under NCCL_DEBUG=VERSION) goes to stderr
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

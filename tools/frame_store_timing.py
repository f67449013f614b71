"""Incremental loop closing with a frame store (nicp_frame_store_*) against the per-call sharded entries
(nicp_align_frames_sharded / nicp_multi_align_frames_sharded), at BASELINE config 5 rig size (4 x 1280x960, composite
1280 x 3840) and with 640x480 pinhole frames.

The closer starts with K frames.  Each of T steps adds one frame and aligns it against the K frames before it (candidates
ordered by id, the new frame as the current one), as MapCloser::process does each time the map grows.
  store:   the store holds every frame added so far; one nicp_frame_store_add + one nicp_frame_store_align per step.
  sharded: one *_align_frames_sharded call per step over the K + 1 frames that step references.
Reported per step: host wall time of the step (both calls are synchronous, so the clock stops after the device has
finished), frames prepared (store: from nicp_frame_store_counters; sharded: every frame of the call), and whether the
records of the two paths are identical.  Step 0 of the store prepares all K candidates and is reported on its own.
Rendering synthetic rig frames costs ~2 s each on the host, so rig frame f uses rendered image f mod --distinct (the
prep and align cost does not depend on which image a frame holds).  The card's name and power limit are read in the same
run.  Writes <out>/frame_store_timing.json.  Measurement tool, not part of the product."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from g2o_frontend_b200 import capi, synth  # noqa: E402
from rig_batch_timing import card  # noqa: E402


def params():
    C = bench.CONF
    sp = capi.make_stats_params(C["worldRadius"], C["minImageRadius"], C["maxImageRadius"], C["minPoints"],
                                C["curvatureThreshold"], C["omegaCurvatureThreshold"])
    ap = capi.make_align_params(C["inlierDistanceThreshold"], C["inlierNormalAngularThreshold"], C["flatCurvatureThreshold"],
                                C["inlierCurvatureRatioThreshold"], C["inlierMaxChi2"], True, C["outerIterations"], 1)
    return sp, ap


def trajectory(n, seed):
    """n poses along a slow walk, so that every frame overlaps the ones before it"""
    rng = np.random.default_rng(seed)
    base = synth.make_pose((0.1, -0.05, 0.2), (0, 1, 0), 10.0)
    return [base @ synth.perturbed_pose(rng, np.eye(4), 0.03, 1.5) for _ in range(n)]


def run(name, store, sharded, frames, poses, K, T, warm, ap):
    """store: FrameStore on its own pool; sharded(frames, ref, cur, guesses) -> records.  Returns the report of one mode."""
    n = K + T
    ids = list(range(n))
    rng = np.random.default_rng(5)
    guesses = {}

    def step_pairs(t):
        cur = K + t
        refs = list(range(cur - K, cur))  # ordered by id
        g = np.stack([synth.perturbed_pose(rng, np.linalg.inv(poses[r]) @ poses[cur], 0.02, 1.0) for r in refs])
        return cur, refs, g.astype(np.float32)

    for t in range(T):
        guesses[t] = step_pairs(t)
    # warm-up: one step of each path on throw-away ids, so module loading and scratch allocation are not timed
    for _ in range(warm):
        cur, refs, g = guesses[0]
        sharded([frames[f] for f in refs + [cur]], list(range(K)), [K] * K, g)
    store.add([-1 - f for f in range(K + 1)], [frames[f] for f in range(K + 1)])
    for _ in range(warm):
        store.align([-1 - f for f in range(K)], [-1 - K] * K, guesses[0][2], ap)
    store.remove([-1 - f for f in range(K + 1)])
    b0 = store.counters()[0]

    t0 = time.perf_counter()
    store.add(ids[:K], [frames[f] for f in range(K)])
    add_ms = (time.perf_counter() - t0) * 1e3
    steps = []
    for t in range(T):
        cur, refs, g = guesses[t]
        t0 = time.perf_counter()
        store.add([cur], [frames[cur]])
        recs_store = store.align(refs, [cur] * K, g, ap)
        ms_store = (time.perf_counter() - t0) * 1e3
        b1 = store.counters()[0]
        t0 = time.perf_counter()
        recs_sharded = sharded([frames[f] for f in refs + [cur]], list(range(K)), [K] * K, g)
        ms_sharded = (time.perf_counter() - t0) * 1e3
        steps.append({"step": t, "store_ms": ms_store, "store_frames_built": b1 - b0, "sharded_ms": ms_sharded,
                      "sharded_frames_built": K + 1, "records_identical": recs_store.tobytes() == recs_sharded.tobytes(),
                      "status_ok": int((recs_store["status"] == 0).sum()), "mean_inliers": float(recs_store["inliers"].mean())})
        b0 = b1
    steady = steps[1:]
    out = {"mode": name, "K": K, "T": T, "initial_add_ms": add_ms, "steps": steps,
           "first_step": {"store_ms": steps[0]["store_ms"], "sharded_ms": steps[0]["sharded_ms"],
                          "store_frames_built": steps[0]["store_frames_built"]},
           "all_records_identical": all(s["records_identical"] for s in steps)}
    if steady:
        ms_s = float(np.mean([s["store_ms"] for s in steady]))
        ms_h = float(np.mean([s["sharded_ms"] for s in steady]))
        out["steady_steps"] = {"steps": len(steady), "store_ms_mean": ms_s, "sharded_ms_mean": ms_h,
                               "store_frames_built_mean": float(np.mean([s["store_frames_built"] for s in steady])),
                               "speedup": ms_h / ms_s}
    return out


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", required=True, help="output directory")
    p.add_argument("--gpus", type=int, default=1, help="workers of the pool, one per GPU (GPU 0 listed again if fewer)")
    p.add_argument("--rig-steps", type=int, default=8)
    p.add_argument("--rig-cands", type=int, default=40)
    p.add_argument("--distinct", type=int, default=12, help="rendered rig images, recycled over the frames")
    p.add_argument("--pinhole-steps", type=int, default=16)
    p.add_argument("--pinhole-cands", type=int, default=40)
    p.add_argument("--warmup", type=int, default=1)
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this tool measures device time and has no CPU mode")
    os.makedirs(args.out, exist_ok=True)
    visible = torch.cuda.device_count()
    devices = [g if g < visible else 0 for g in range(args.gpus)]
    sp, ap = params()
    out = {"card": card(), "visible_gpus": visible, "devices": devices, "ap_outer_iterations": ap.outer_iterations}

    # ---- 640x480 pinhole frames
    K, T = args.pinhole_cands, args.pinhole_steps
    poses = trajectory(K + T, 11)
    frames = [synth.render_depth_u16(q, seed=200 + f) for f, q in enumerate(poses)]
    proj = capi.make_projector(synth.K_KINECT, 480, 640, bench.CONF["minD"], bench.CONF["maxD"])
    pool = capi.ShardPool(devices)
    store = capi.FrameStore(pool, proj, sp, (480, 640))
    out["pinhole_640x480"] = run("pinhole 640x480", store, lambda fr, r, c, g: pool.align_frames(fr, proj, sp, r, c, g, ap),
                                 frames, poses, K, T, args.warmup, ap)
    store.close()
    pool.close()
    print(json.dumps(out["pinhole_640x480"].get("steady_steps")), flush=True)

    # ---- config-5 rig
    K, T = args.rig_cands, args.rig_steps
    cams = synth.make_rig(4, 1280, 960)
    mp = capi.make_multi_projector(cams)
    rows, cols = capi.multi_image_size(mp)
    poses = trajectory(K + T, 12)
    rendered = [[synth.render_depth_u16(poses[f] @ c["offset"].astype(np.float64), c["height"], c["width"], c["K"],
                                        seed=100 * f + i, zmin=c["minD"], zmax=c["maxD"]) for i, c in enumerate(cams)]
                for f in range(min(args.distinct, K + T))]
    frames = [rendered[f % len(rendered)] for f in range(K + T)]
    rposes = [poses[f % len(rendered)] for f in range(K + T)]
    pool = capi.ShardPool(devices)
    store = capi.FrameStore(pool, mp, sp, [im.shape for im in frames[0]])
    out["rig_config5"] = run("rig 4 x 1280x960 (composite %d x %d)" % (rows, cols), store,
                             lambda fr, r, c, g: pool.multi_align_frames(fr, mp, sp, r, c, g, ap), frames, rposes, K, T,
                             args.warmup, ap)
    out["rig_config5"]["distinct_images"] = len(rendered)
    store.close()
    pool.close()
    print(json.dumps(out["rig_config5"].get("steady_steps")), flush=True)
    path = os.path.join(args.out, "frame_store_timing.json")
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps({k: out[k] for k in ("card", "devices")}))
    ok = out["pinhole_640x480"]["all_records_identical"] and out["rig_config5"]["all_records_identical"]
    if not ok:
        raise SystemExit("store and sharded records differ")


if __name__ == "__main__":
    main()

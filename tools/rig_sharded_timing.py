"""Rig loop closure over the GPUs of one process (nicp_multi_align_frames_sharded) at BASELINE config 5 size
(4 x 1280x960, composite 1280 x 3840): n_cur current x n_cand candidate rig frames in pinned host memory, every current
against every candidate, current-major.
  (a) pairs/s end to end (host clock around the synchronous call) through shard pools over 1, 2, 4 and 8 of the visible
      GPUs, and the scaling factor against the one-GPU pool; device counts above the visible ones are reported as not
      measured;
  (b) the same job on one context as nicp_multi_raw_depth_to_cloud_batch + nicp_multi_align_batch;
  (c) per device count, the prep / align split of worker 0's block: that block timed on one context as two synchronised
      calls (its frames built in one call, its pairs aligned in one call), host clock.  The pool does not expose the split;
      it is the evidence for preparing a frame once and copying its cloud to the other devices instead.
The records must be identical across device counts and to (b).  The card's name and power limit are read in the same run.
Writes <out>/rig_sharded_timing.json.  Measurement tool, not part of the product."""
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


def wall(fn, reps, warmup):
    """mean host milliseconds of fn(), which ends in a device synchronise, after warm-up; returns (ms, last result)"""
    for _ in range(warmup):
        out = fn()
    t0 = time.perf_counter()
    for _ in range(reps):
        out = fn()
    return (time.perf_counter() - t0) * 1e3 / reps, out


def main():
    ap_ = argparse.ArgumentParser()
    ap_.add_argument("--out", required=True, help="output directory")
    ap_.add_argument("--cur", type=int, default=4)
    ap_.add_argument("--cand", type=int, default=8)
    ap_.add_argument("--reps", type=int, default=3)
    ap_.add_argument("--warmup", type=int, default=1)
    args = ap_.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this tool measures device time and has no CPU mode")
    os.makedirs(args.out, exist_ok=True)
    C = bench.CONF
    cams = synth.make_rig(4, 1280, 960)
    mp = capi.make_multi_projector(cams)
    rows, cols = capi.multi_image_size(mp)
    sp = capi.make_stats_params(C["worldRadius"], C["minImageRadius"], C["maxImageRadius"], C["minPoints"],
                                C["curvatureThreshold"], C["omegaCurvatureThreshold"])
    ap = capi.make_align_params(C["inlierDistanceThreshold"], C["inlierNormalAngularThreshold"], C["flatCurvatureThreshold"],
                                C["inlierCurvatureRatioThreshold"], C["inlierMaxChi2"], True, C["outerIterations"], 1)
    rng = np.random.default_rng(1005)
    base = synth.make_pose((0.1, -0.05, 0.2), (0, 1, 0), 10.0)
    cur_poses = [synth.perturbed_pose(rng, base, 0.1, 4.0) for _ in range(args.cur)]
    cand_poses = [synth.perturbed_pose(rng, base, 0.1, 4.0) for _ in range(args.cand)]
    poses = cur_poses + cand_poses
    nF = len(poses)
    pinned = torch.empty((nF, len(cams), 960, 1280), dtype=torch.int16).pin_memory()
    host = pinned.numpy().view(np.uint16)
    for f, p in enumerate(poses):
        for i, c in enumerate(cams):
            host[f, i] = synth.render_depth_u16(p @ c["offset"].astype(np.float64), c["height"], c["width"], c["K"],
                                                seed=100 * f + i, zmin=c["minD"], zmax=c["maxD"])
    frames = [[host[f, i] for i in range(len(cams))] for f in range(nF)]
    ref_frame, cur_frame, guesses = [], [], []
    for ci in range(args.cur):
        for ri in range(args.cand):
            guesses.append(synth.perturbed_pose(rng, np.linalg.inv(cand_poses[ri]) @ cur_poses[ci], 0.05, 3.0))
            ref_frame.append(args.cur + ri)
            cur_frame.append(ci)
    guesses = np.stack(guesses).astype(np.float32)
    n = len(ref_frame)
    visible = torch.cuda.device_count()
    out = {"card": card(), "visible_gpus": visible, "rig": "4 x 1280x960 (composite %d x %d)" % (rows, cols),
           "pairs": n, "current_frames": args.cur, "candidate_frames": args.cand, "reps": args.reps, "warmup": args.warmup}

    # ---- (b) one context, the two batch calls
    ctx = capi.Context(0)
    clouds = [ctx.new_cloud(rows * cols) for _ in range(nF)]
    refs = [clouds[r] for r in ref_frame]
    curs = [clouds[c] for c in cur_frame]

    def one_context():
        ctx.multi_raw_depth_to_cloud_batch(frames, mp, sp, clouds=clouds)
        return ctx.multi_align_batch(refs, curs, mp, ap, guesses)

    ms, base_recs = wall(one_context, args.reps, args.warmup)
    out["one_context"] = {"ms": ms, "pairs_per_s": n / (ms * 1e-3)}

    # ---- (a) pools, and (c) worker 0's block on one context
    out["pools"] = {}
    recs_by_g = {}
    for G in (1, 2, 4, 8):
        if G > visible:
            out["pools"][str(G)] = "not measured (%d GPU%s visible)" % (visible, "" if visible == 1 else "s")
            continue
        pool = capi.ShardPool(list(range(G)))
        ms, recs = wall(lambda: pool.multi_align_frames(frames, mp, sp, ref_frame, cur_frame, guesses, ap), args.reps,
                        args.warmup)
        pool.close()
        recs_by_g[G] = recs
        lo, hi = 0, n // G  # worker 0's block
        blk_frames = sorted(set(ref_frame[lo:hi]) | set(cur_frame[lo:hi]))
        slot = {f: k for k, f in enumerate(blk_frames)}
        bclouds = clouds[:len(blk_frames)]
        brefs = [bclouds[slot[r]] for r in ref_frame[lo:hi]]
        bcurs = [bclouds[slot[c]] for c in cur_frame[lo:hi]]
        prep_ms, _ = wall(lambda: (ctx.multi_raw_depth_to_cloud_batch([frames[f] for f in blk_frames], mp, sp, clouds=bclouds),
                                   ctx.synchronize()), args.reps, args.warmup)
        align_ms, blk = wall(lambda: ctx.multi_align_batch(brefs, bcurs, mp, ap, guesses[lo:hi]), args.reps, args.warmup)
        assert blk.tobytes() == recs[lo:hi].tobytes(), G
        out["pools"][str(G)] = {"ms": ms, "pairs_per_s": n / (ms * 1e-3),
                                "worker0_block": {"pairs": hi - lo, "frames": len(blk_frames), "prep_ms": prep_ms,
                                                  "align_ms": align_ms, "prep_ms_per_frame": prep_ms / len(blk_frames),
                                                  "align_ms_per_pair": align_ms / (hi - lo)}}
    ctx.close()
    one = out["pools"]["1"]["pairs_per_s"]
    for G, v in out["pools"].items():
        if isinstance(v, dict):
            v["scaling_vs_1_gpu"] = v["pairs_per_s"] / one
    out["one_gpu_pool_vs_one_context"] = one / out["one_context"]["pairs_per_s"]
    for G, recs in recs_by_g.items():
        assert recs.tobytes() == base_recs.tobytes(), "records of the %d-GPU pool differ from the one-context run" % G
    out["records_identical_across_device_counts"] = True
    out["status_ok"] = int((base_recs["status"] == 0).sum())
    out["mean_inliers"] = float(base_recs["inliers"].mean())
    path = os.path.join(args.out, "rig_sharded_timing.json")
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()

"""Batched keyframe tracking (nicp_tracker_*) of S independent synthetic 640x480 depth sequences on one worker, against
the pipelined single-sequence loop of BASELINE config 3 (tools/bench_configs.py:config3).

For step (DepthImage_scale) 1 and 2 and S = 1, 8, 64, 256: one tracker of S sequences on a shard pool of one worker, every
step listing all S sequences.  frames/s = S x timed steps / host wall time around the synchronous step calls, after warm-up
steps; the timed window is repeated and every repeat is reported.  Sequence s walks frames start_s, start_s + 1, ... of one
rendered trajectory (the prep and align cost does not depend on which images a sequence holds), so a few hundred rendered
frames serve 256 sequences.  For the largest S the same work is also split: one nicp_raw_depth_to_cloud_batch of S frames
and one nicp_align_batch of S pairs with S distinct current clouds (the tracker's batch shape), each timed on its own
context, to show which half dominates a step.  The card's name and power limit are read in the same run.  Writes
<out>/tracker_timing.json.  Measurement tool, not part of the product."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench_configs  # noqa: E402
from g2o_frontend_b200 import capi, synth  # noqa: E402
from rig_batch_timing import card  # noqa: E402

LEVEL = {1: (1, 10, 30, 50, 1.0), 2: (2, 5, 15, 25, 0.5)}  # bench_configs.LEVELS: step, minR, maxR, minPoints, distance


def run_tracker(proj, sp, ap, step, raws, S, steps, warm, repeats):
    pool = capi.ShardPool([0])
    tr = capi.Tracker(pool, proj, sp, ap, (480, 640), S, step=step)
    span = warm + repeats * steps
    starts = [(7 * s) % (len(raws) - span) for s in range(S)]
    seqs = list(range(S))
    t = 0

    def one():
        nonlocal t
        res = tr.step(seqs, [raws[starts[s] + t] for s in seqs])
        t += 1
        return res

    for _ in range(warm):
        one()
    walls, keyframes, inliers = [], 0, []
    for _ in range(repeats):
        t0 = time.perf_counter()
        for _ in range(steps):
            res = one()
            keyframes += int(res["keyframe"].sum())
            inliers.append(float(res["record"]["inliers"].mean()))
        walls.append(time.perf_counter() - t0)
    tr.close()
    pool.close()
    rates = [S * steps / w for w in walls]
    return {"S": S, "timed_steps": steps, "warmup_steps": warm, "repeats": repeats,
            "frames_per_s": float(np.median(rates)), "frames_per_s_repeats": rates,
            "step_ms_median": float(np.median(walls)) / steps * 1e3, "keyframe_switches": keyframes,
            "mean_inliers": float(np.mean(inliers))}


def split(proj, sp, ap, step, raws, S, reps):
    """one batched prep of S frames and one batched alignment of S pairs with distinct current clouds, on a plain context"""
    ctx = capi.Context(0)
    frames = [raws[k % len(raws)] for k in range(2 * S)]
    keys = ctx.raw_depth_to_cloud_batch(frames[:S], proj, sp, step=step)
    curs = ctx.raw_depth_to_cloud_batch(frames[S:], proj, sp, step=step)
    ctx.synchronize()

    def prep():
        ctx.raw_depth_to_cloud_batch(frames[S:], proj, sp, step=step, clouds=curs)
        ctx.synchronize()

    def align():
        ctx.align_batch(keys, curs, proj, ap)

    out = {}
    for name, fn in (("prep", prep), ("align", align)):
        fn()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        out[name + "_ms"] = (time.perf_counter() - t0) / reps * 1e3
        out[name + "_us_per_frame"] = out[name + "_ms"] * 1e3 / S
    for c in keys + curs:
        c.close()
    ctx.close()
    return out


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", required=True, help="output directory")
    p.add_argument("--sizes", default="1,8,64,256")
    p.add_argument("--steps", type=int, default=12, help="timed steps per repeat")
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--repeats", type=int, default=3)
    p.add_argument("--baseline-frames", type=int, default=400, help="frames of the config-3 baseline sequence")
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this tool measures device time and has no CPU mode")
    os.makedirs(args.out, exist_ok=True)
    sizes = [int(x) for x in args.sizes.split(",")]
    out = {"card": card(), "workers": 1, "image": "640x480 raw, synthetic (synth.trajectory + render_depth_u16)",
           "new_frame_inliers_fraction": 0.4}
    span = args.warmup + args.repeats * args.steps
    _, raws = bench_configs.render_sequence(span + 96)  # 96 distinct start frames
    out["rendered_frames"] = len(raws)

    ctx = capi.Context(0)
    base = bench_configs.config3(ctx, None, args.baseline_frames)
    ctx.close()
    out["baseline_config3"] = {k: base[k] for k in ("workload", "frames", "value", "unit", "schedule", "keyframes")}
    out["baseline_config3"]["strictly_sequential_frames_per_s"] = base["strictly_sequential"]["value"]
    print(json.dumps(out["baseline_config3"]), flush=True)

    for step in (1, 2):
        s, minr, maxr, minp, dist = LEVEL[step]
        proj, sp, ap = bench_configs.params(s, minr, maxr, minp, dist)
        rows = []
        for S in sizes:
            r = run_tracker(proj, sp, ap, step, raws, S, args.steps, args.warmup, args.repeats)
            r["speedup_vs_config3"] = r["frames_per_s"] / out["baseline_config3"]["value"]
            rows.append(r)
            print(json.dumps(dict(step=step, **r)), flush=True)
        out["step%d" % step] = {"image": "%dx%d clouds" % (640 // step, 480 // step), "sizes": rows,
                                "split_at_S%d" % max(sizes): split(proj, sp, ap, step, raws, max(sizes), 5)}
        print(json.dumps(out["step%d" % step]["split_at_S%d" % max(sizes)]), flush=True)
    path = os.path.join(args.out, "tracker_timing.json")
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out["card"]))


if __name__ == "__main__":
    main()

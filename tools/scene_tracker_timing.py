"""Batched scene-based odometry (nicp_scene_tracker_*) of S independent synthetic 640x480 depth sequences on one worker,
against the chain of single C-ABI calls the localmap loop of host/pwn_simple_aligner.cpp makes, run sequence by sequence.

For step (DepthImage_scale) 4 (160x120 clouds) and step 2 (320x240), both with the parameters of pwn_aligner_1_4.conf
(tests/test_scene_tracker.py:params, the same projector, statistics, alignment and merge parameters on both sides), and
S = 1, 8, 64: one scene tracker of S sequences on a shard pool of one worker, every step listing all S sequences,
chunk_step 10.  frames/s = S x timed steps / host wall time around the synchronous step calls, after warm-up steps; the
timed window is repeated and every repeat is reported, with the split of the tracker's host time between phase 1 (prep,
render, alignment) and phase 2 (append, merges) from nicp_scene_tracker_phase_ms.  The chain
(tests/test_scene_tracker.py::Chain: nicp_raw_depth_to_cloud, nicp_depth_prepare + nicp_cloud_compute_gaussians,
nicp_project, nicp_depth_to_cloud, nicp_align, nicp_cloud_append, nicp_merge per frame, through the Python binding; a new
map empties the old one, as referenceScene.clear() does) runs the first min(S, 8) sequences one after the other on a plain
context: its rate does not depend on S.  Sequence s walks frames start_s, start_s + 1, ... of one rendered trajectory.
The card's name and power limit are read in the same run.  Writes the JSON to --out
(profiles/scene_tracker_timing_1gpu.json is this tool's output).  Measurement tool, not part of the product."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)
import bench_configs  # noqa: E402
from g2o_frontend_b200 import capi  # noqa: E402
from rig_batch_timing import card  # noqa: E402
from test_scene_tracker import ALPHA, BASELINE, Chain, params  # noqa: E402

CHUNK = 10


def starts_of(S, n_raws, span):
    return [(7 * s) % (n_raws - span) for s in range(S)]


def run_tracker(step, raws, S, steps, warm, repeats, cap):
    _, proj, sp, ap, mp = params(step)
    pool = capi.ShardPool([0])
    tr = capi.SceneTracker(pool, proj, sp, ap, (480, 640), S, cap, mp=mp, step=step, baseline=BASELINE, alpha=ALPHA,
                           chunk_step=CHUNK)
    starts = starts_of(S, len(raws), warm + repeats * steps)
    seqs = list(range(S))
    t = 0

    def one():
        nonlocal t
        res = tr.step(seqs, [raws[starts[s] + t] for s in seqs])
        t += 1
        return res

    for _ in range(warm):
        one()
    walls, phases, inliers, maps = [], [], [], []
    for _ in range(repeats):
        p0 = tr.phase_ms()
        t0 = time.perf_counter()
        for _ in range(steps):
            res = one()
            inliers.append(float(res["record"]["inliers"].mean()))
            maps.append(float(res["map_points"].mean()))
        walls.append(time.perf_counter() - t0)
        p1 = tr.phase_ms()
        phases.append((p1[0] - p0[0], p1[1] - p0[1]))
    tr.close()
    pool.close()
    rates = [S * steps / w for w in walls]
    ph1 = float(np.median([p[0] for p in phases])) / steps
    ph2 = float(np.median([p[1] for p in phases])) / steps
    return {"S": S, "timed_steps": steps, "warmup_steps": warm, "repeats": repeats,
            "frames_per_s": float(np.median(rates)), "frames_per_s_repeats": rates,
            "step_ms_median": float(np.median(walls)) / steps * 1e3, "phase1_ms_per_step": ph1,
            "phase2_ms_per_step": ph2, "phase2_share": ph2 / (ph1 + ph2), "mean_inliers": float(np.mean(inliers)),
            "mean_map_points": float(np.mean(maps))}


def run_chain(step, raws, S, steps, warm, repeats):
    ctx = capi.Context(0)
    n = min(S, 8)
    starts = starts_of(n, len(raws), warm + repeats * steps)
    chains = [Chain(ctx, step, CHUNK) for _ in range(n)]
    for s, ch in enumerate(chains):
        for t in range(warm):
            ch.frame(raws[starts[s] + t])
    walls = []
    for rep in range(repeats):
        t0 = time.perf_counter()
        for s, ch in enumerate(chains):
            for t in range(steps):
                ch.frame(raws[starts[s] + warm + rep * steps + t])
        walls.append(time.perf_counter() - t0)
    ctx.close()
    rates = [n * steps / w for w in walls]
    return {"sequences": n, "frames_per_s": float(np.median(rates)), "frames_per_s_repeats": rates}


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", required=True, help="output JSON file")
    p.add_argument("--sizes", default="1,8,64")
    p.add_argument("--steps", type=int, default=10, help="timed steps per repeat")
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--repeats", type=int, default=3)
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this tool measures device time and has no CPU mode")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    sizes = [int(x) for x in args.sizes.split(",")]
    out = {"card": card(), "workers": 1, "chunk_step": CHUNK, "parameters": "pwn_aligner_1_4.conf radii at both steps",
           "image": "640x480 raw, synthetic (synth.trajectory + render_depth_u16)"}
    span = args.warmup + args.repeats * args.steps
    _, raws = bench_configs.render_sequence(span + 64)
    out["rendered_frames"] = len(raws)
    for step in (4, 2):
        proj = params(step)[1]
        cap = 16 * proj.rows * proj.cols  # a chunk of 10 frames after merging fits with room to spare
        chain = run_chain(step, raws, max(sizes), args.steps, args.warmup, args.repeats)
        print(json.dumps(dict(step=step, chain=chain)), flush=True)
        rows = []
        for S in sizes:
            r = run_tracker(step, raws, S, args.steps, args.warmup, args.repeats, cap)
            r["ratio_vs_chain"] = r["frames_per_s"] / chain["frames_per_s"]
            rows.append(r)
            print(json.dumps(dict(step=step, **r)), flush=True)
        out["step%d" % step] = {"image": "%dx%d clouds" % (640 // step, 480 // step), "map_capacity": cap,
                                "chain_single_calls": chain, "sizes": rows}
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out["card"]))


if __name__ == "__main__":
    main()

"""Local maps from raw 640x480 frames: nicp_raw_depth_to_local_map against the chain of single calls it replaces, per
frame nicp_raw_depth_to_cloud + nicp_depth_prepare + nicp_cloud_compute_gaussians + nicp_cloud_append, then nicp_merge and
nicp_voxelize.  N = 8, 32 and 128 frames along synth.trajectory at steps 1 and 2.

Per (step, N), each path is timed twice: appends only (time per frame), and with Merger::merge (identity transform, default
parameters) and voxel thinning (--voxel) behind them, whose difference is the merge + voxelize share.  Every call of both
paths ends in a device synchronisation, so a host clock around it measures the device work and the host round trips
together.  The map is emptied between repetitions (no reallocation); one warm-up run per path and shape.  The final maps
of the two paths are compared byte for byte.  The card's name and power limit are read in the same run.  Writes
<out>/local_map_timing.json.  Measurement tool, not part of the product."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from g2o_frontend_b200 import capi, synth  # noqa: E402
from rig_batch_timing import card  # noqa: E402

BASELINE, ALPHA = 0.075, 0.1


def camera(step):
    C = bench.CONF
    K = synth.scaled_K(synth.K_KINECT, 1.0 / step)
    proj = capi.make_projector(K, 480 // step, 640 // step, C["minD"], C["maxD"])
    sp = (capi.make_stats_params(C["worldRadius"], C["minImageRadius"], C["maxImageRadius"], C["minPoints"],
                                 C["curvatureThreshold"], C["omegaCurvatureThreshold"]) if step == 1 else
          capi.make_stats_params(C["worldRadius"], 3, 6, 10, C["curvatureThreshold"], C["omegaCurvatureThreshold"]))
    return proj, sp


def empty(cl):
    cl.upload(np.zeros((0, 4), np.float32))


def chain(ctx, raws, poses, step, cl, fc, full, vres):
    proj, sp = camera(step)
    for raw, T in zip(raws, poses):
        ctx.raw_depth_to_cloud(raw, proj, sp, step=step, cloud=fc)
        fc.compute_gaussians(ctx.depth_prepare(raw, step=step), proj, BASELINE, ALPHA)
        cl.append(fc, T)
    if full:
        cl.merge(proj, np.eye(4, dtype=np.float32), capi.make_merge_params())
        cl.voxelize(vres)


def entry(ctx, raws, poses, step, cl, full, vres):
    proj, sp = camera(step)
    ctx.raw_depth_to_local_map(raws, proj, sp, poses, cl, step=step, baseline=BASELINE, alpha=ALPHA,
                               merge_params=capi.make_merge_params() if full else None,
                               voxel_resolution=vres if full else 0.0)


def timed(ctx, fn, cl, reps):
    """median host ms of fn() over reps runs on an emptied map (one warm-up run first)"""
    out = []
    for r in range(reps + 1):
        empty(cl)
        ctx.synchronize()
        t0 = time.perf_counter()
        fn()
        ctx.synchronize()
        if r:
            out.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(out)), out


def snapshot(cl):
    d = cl.download()
    g, f = cl.download_gaussians()
    return [cl.size()] + [d[k].tobytes() for k in ("points", "normals", "curvature", "omega_p", "omega_n")] + [g.tobytes(), f.tobytes()]


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", required=True, help="output directory")
    p.add_argument("--frames", type=int, nargs="+", default=[8, 32, 128])
    p.add_argument("--steps", type=int, nargs="+", default=[1, 2])
    p.add_argument("--reps", type=int, default=3)
    p.add_argument("--voxel", type=float, default=0.05, help="voxel side in metres")
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this tool measures device time and has no CPU mode")
    os.makedirs(args.out, exist_ok=True)
    nmax = max(args.frames)
    poses = [q.astype(np.float32) for q in synth.trajectory(nmax, seed=7)]
    raws = [synth.render_depth_u16(q, seed=300 + i, dropout=0.05) for i, q in enumerate(poses)]
    out = {"card": card(), "reps": args.reps, "voxel_resolution": args.voxel, "merge": "identity transform, default params",
           "runs": []}
    ctx = capi.Context(0)
    for step in args.steps:
        P = (480 // step) * (640 // step)
        fc = ctx.new_cloud(P)  # the chain's frame cloud, reused frame to frame
        for n in args.frames:
            fr, po = raws[:n], poses[:n]
            a, b = ctx.new_cloud(n * P), ctx.new_cloud(n * P)
            chain_app, chain_app_runs = timed(ctx, lambda: chain(ctx, fr, po, step, a, fc, False, args.voxel), a, args.reps)
            entry_app, entry_app_runs = timed(ctx, lambda: entry(ctx, fr, po, step, b, False, args.voxel), b, args.reps)
            appended = b.size()
            chain_tot, _ = timed(ctx, lambda: chain(ctx, fr, po, step, a, fc, True, args.voxel), a, args.reps)
            entry_tot, _ = timed(ctx, lambda: entry(ctx, fr, po, step, b, True, args.voxel), b, args.reps)
            run = {"step": step, "image": "%dx%d" % (640 // step, 480 // step), "frames": n, "appended_points": appended,
                   "final_points": b.size(),
                   "chain": {"append_ms_per_frame": chain_app / n, "total_ms": chain_tot, "append_ms": chain_app,
                             "merge_voxelize_ms": chain_tot - chain_app,
                             "merge_voxelize_share": (chain_tot - chain_app) / chain_tot, "append_runs_ms": chain_app_runs},
                   "entry": {"append_ms_per_frame": entry_app / n, "total_ms": entry_tot, "append_ms": entry_app,
                             "merge_voxelize_ms": entry_tot - entry_app,
                             "merge_voxelize_share": (entry_tot - entry_app) / entry_tot, "append_runs_ms": entry_app_runs},
                   "append_speedup": chain_app / entry_app, "total_speedup": chain_tot / entry_tot,
                   "maps_identical": snapshot(a) == snapshot(b)}
            out["runs"].append(run)
            print(json.dumps({k: run[k] for k in ("step", "frames", "append_speedup", "total_speedup", "maps_identical")}
                             | {"chain_ms_per_frame": run["chain"]["append_ms_per_frame"],
                                "entry_ms_per_frame": run["entry"]["append_ms_per_frame"],
                                "entry_merge_voxelize_share": run["entry"]["merge_voxelize_share"]}), flush=True)
            a.close()
            b.close()
        fc.close()
    ctx.close()
    with open(os.path.join(args.out, "local_map_timing.json"), "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out["card"]))
    if not all(r["maps_identical"] for r in out["runs"]):
        raise SystemExit("the entry and the chain built different maps")


if __name__ == "__main__":
    main()

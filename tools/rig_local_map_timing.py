"""Local maps from raw rig frames: nicp_multi_raw_depth_to_local_map against the chain of single calls it replaces, per
frame nicp_multi_raw_depth_to_cloud_batch (one frame) + nicp_depth_prepare of every camera + the host transpose into the
composite + nicp_multi_cloud_compute_gaussians + nicp_cloud_append, then nicp_merge (pinhole view of camera 0) and
nicp_voxelize.

Rigs: the BASELINE config-5 rig (synth.make_rig(4, 1280, 960), composite 1280 x 3840, one frame per launch set at step 1,
two at step 2) and a small rig of four 160x120 cameras (composite 160 x 480, eight frames per launch set).  Per (rig, step,
N), each path is timed with appends only and with merge + voxelize behind them.  Every call of both paths ends in a device
synchronisation; a CUDA event pair on the context's stream around the call measures it, host round trips included.  The map
is emptied between repetitions (no reallocation); one warm-up run per path and shape.  The final maps of the two paths are
compared byte for byte.  The card's name and power limit are read in the same run.  Writes <out>/rig_local_map_timing.json.
Measurement tool, not part of the product."""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from g2o_frontend_b200 import capi, synth  # noqa: E402
from rig_batch_timing import card  # noqa: E402

BASELINE, ALPHA = 0.075, 0.1


def rig(kind, step):
    """the rig after scaling (what the projector describes) and the stats parameters"""
    if kind == "config5":
        cams = synth.make_rig(4, 1280 // step, 960 // step, K=synth.scaled_K(synth.K_KINECT, 2.0 / step))
    else:
        cams = synth.make_rig(4, 160, 120, K=synth.scaled_K(synth.K_KINECT, 160 / 640.0))
    return cams, capi.make_stats_params(0.1, 3, 6, 10, 0.2, 0.02)


def raw_frame(pose, cams, step, seed):
    return [synth.render_depth_u16(pose @ c["offset"].astype(np.float64), c["height"] * step, c["width"] * step,
                                   synth.scaled_K(c["K"], step), seed=seed + 17 * i, dropout=0.02, zmin=c["minD"],
                                   zmax=c["maxD"]) for i, c in enumerate(cams)]


def composite(ctx, frame, cams, step):
    out = np.zeros((max(c["width"] for c in cams), sum(c["height"] for c in cams)), np.float32)
    off = 0
    for r, c in zip(frame, cams):
        out[:c["width"], off:off + c["height"]] = ctx.depth_prepare(r, step=step).T
        off += c["height"]
    return out


def merge_view(cams):
    c = cams[0]
    return capi.make_projector(c["K"], c["height"], c["width"], c["minD"], c["maxD"])


def empty(cl):
    cl.upload(np.zeros((0, 4), np.float32))


def chain(ctx, cams, sp, frames, poses, step, cl, fc, full, vres):
    mp = capi.make_multi_projector(cams)
    for fr, T in zip(frames, poses):
        ctx.multi_raw_depth_to_cloud_batch([fr], mp, sp, step=step, clouds=[fc])
        fc.multi_compute_gaussians(composite(ctx, fr, cams, step), mp, BASELINE, ALPHA)
        cl.append(fc, T)
    if full:
        cl.merge(merge_view(cams), np.eye(4, dtype=np.float32), capi.make_merge_params())
        cl.voxelize(vres)


def entry(ctx, cams, sp, frames, poses, step, cl, full, vres):
    ctx.multi_raw_depth_to_local_map(frames, capi.make_multi_projector(cams), sp, poses, cl, step=step, baseline=BASELINE,
                                     alpha=ALPHA, merge_proj=merge_view(cams),
                                     merge_params=capi.make_merge_params() if full else None,
                                     voxel_resolution=vres if full else 0.0)


def timed(ctx, stream, fn, cl, reps):
    """median ms of fn() over reps runs on an emptied map (one warm-up run first), CUDA events on the context's stream"""
    out = []
    for r in range(reps + 1):
        empty(cl)
        ctx.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        e1.synchronize()
        if r:
            out.append(e0.elapsed_time(e1))
    return float(np.median(out)), out


def snapshot(cl):
    d = cl.download()
    g, f = cl.download_gaussians()
    return [cl.size()] + [d[k].tobytes() for k in ("points", "normals", "curvature", "omega_p", "omega_n")] + [g.tobytes(), f.tobytes()]


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", required=True, help="output directory")
    p.add_argument("--cases", nargs="+", default=["config5:1:4", "config5:2:8", "small:1:8", "small:1:32"],
                   help="rig:step:frames")
    p.add_argument("--reps", type=int, default=3)
    p.add_argument("--voxel", type=float, default=0.05, help="voxel side in metres")
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this tool measures device time and has no CPU mode")
    os.makedirs(args.out, exist_ok=True)
    out = {"card": card(), "reps": args.reps, "voxel_resolution": args.voxel,
           "merge": "pinhole view of camera 0, identity transform, default params", "runs": []}
    ctx = capi.Context(0)
    stream = torch.cuda.ExternalStream(ctx.stream())
    rng = np.random.default_rng(5)
    base = synth.make_pose((0.1, -0.05, 0.2), (0, 1, 0), 10.0)
    for case in args.cases:
        kind, step, n = case.split(":")
        step, n = int(step), int(n)
        cams, sp = rig(kind, step)
        poses = [synth.perturbed_pose(rng, base, 0.04, 3.0).astype(np.float32) for _ in range(n)]
        frames = [raw_frame(q, cams, step, 300 + 5 * i) for i, q in enumerate(poses)]
        P = max(c["width"] for c in cams) * sum(c["height"] for c in cams)
        fc = ctx.new_cloud(P)  # the chain's frame cloud, reused frame to frame
        a, b = ctx.new_cloud(n * P), ctx.new_cloud(n * P)
        run_c = lambda full: (lambda: chain(ctx, cams, sp, frames, poses, step, a, fc, full, args.voxel))
        run_e = lambda full: (lambda: entry(ctx, cams, sp, frames, poses, step, b, full, args.voxel))
        chain_app, chain_app_runs = timed(ctx, stream, run_c(False), a, args.reps)
        entry_app, entry_app_runs = timed(ctx, stream, run_e(False), b, args.reps)
        appended = b.size()
        chain_tot, _ = timed(ctx, stream, run_c(True), a, args.reps)
        entry_tot, _ = timed(ctx, stream, run_e(True), b, args.reps)
        run = {"rig": kind, "step": step, "composite": "%dx%d" % (max(c["width"] for c in cams), sum(c["height"] for c in cams)),
               "frames": n, "appended_points": appended, "final_points": b.size(),
               "chain": {"append_ms_per_frame": chain_app / n, "total_ms": chain_tot, "append_ms": chain_app,
                         "append_runs_ms": chain_app_runs},
               "entry": {"append_ms_per_frame": entry_app / n, "total_ms": entry_tot, "append_ms": entry_app,
                         "append_runs_ms": entry_app_runs},
               "append_speedup": chain_app / entry_app, "total_speedup": chain_tot / entry_tot,
               "maps_identical": snapshot(a) == snapshot(b)}
        out["runs"].append(run)
        print(json.dumps({k: run[k] for k in ("rig", "step", "frames", "append_speedup", "total_speedup", "maps_identical")}
                         | {"chain_ms_per_frame": run["chain"]["append_ms_per_frame"],
                            "entry_ms_per_frame": run["entry"]["append_ms_per_frame"]}), flush=True)
        for c in (a, b, fc):
            c.close()
    ctx.close()
    with open(os.path.join(args.out, "rig_local_map_timing.json"), "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out["card"]))
    if not all(r["maps_identical"] for r in out["runs"]):
        raise SystemExit("the entry and the chain built different maps")


if __name__ == "__main__":
    main()

"""Rig (MultiPointProjector, BASELINE config 5: 4 x 1280x960, composite 1280 x 3840) batch entry points against the
single-frame / single-pair loops they replace, on one GPU, in one process:
  (a) rig frames/s through nicp_multi_raw_depth_to_cloud_batch from pinned raw frames, for every frames-per-launch-set
      setting (NICP_PREP_BATCH, capped by the library's rule), against a loop of nicp_multi_depth_to_cloud over composites
      converted on the host (the host conversion is timed separately);
  (b) rig pairs/s through nicp_multi_align_batch (n_cur current x n_cand candidate frames, guesses perturbed from the true
      relative pose as in bench.make_workload) against a loop of nicp_multi_align.
Device time from CUDA events on the context's stream, after warm-up.  Algorithmic bytes per SURVEY.md 8d: prep 88 P + 76 N
per frame, align (12 N_c + 8 P) + outer (12 N_r + 16 P) + 56 M_idx + 48 M_acc + (8 P + the mean per-iteration M terms)
for the statistics pass, from the work counters of the records.  Writes <out>/rig_batch_timing.json.
Measurement tool, not part of the product."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from g2o_frontend_b200 import capi, synth  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        pl, sm = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit_w": float(pl), "sm_max_mhz": float(sm)}
    except Exception as e:  # the numbers stay usable without it, but say why it is missing
        return {"name": name, "power_limit_w": None, "sm_max_mhz": None, "error": str(e)}


def timed(ctx, stream, fn, reps, warmup):
    for _ in range(warmup):
        fn()
    ctx.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    ctx.synchronize()
    return e0.elapsed_time(e1) / reps, (time.perf_counter() - w0) * 1e3 / reps


def main():
    ap_ = argparse.ArgumentParser()
    ap_.add_argument("--out", required=True, help="output directory")
    ap_.add_argument("--cur", type=int, default=4)
    ap_.add_argument("--cand", type=int, default=8)
    ap_.add_argument("--prep-frames", type=int, default=8)
    ap_.add_argument("--reps", type=int, default=5)
    ap_.add_argument("--warmup", type=int, default=2)
    args = ap_.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this tool measures device time and has no CPU mode")
    os.makedirs(args.out, exist_ok=True)
    C = bench.CONF
    cams = synth.make_rig(4, 1280, 960)
    mp = capi.make_multi_projector(cams)
    rows, cols = capi.multi_image_size(mp)
    P = rows * cols
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
    # raw frames in sensor orientation (camera i: height_i x width_i), noisy, in one pinned buffer
    pinned = torch.empty((nF, len(cams), 960, 1280), dtype=torch.int16).pin_memory()
    host = pinned.numpy().view(np.uint16)
    for f, p in enumerate(poses):
        for i, c in enumerate(cams):
            host[f, i] = synth.render_depth_u16(p @ c["offset"].astype(np.float64), c["height"], c["width"], c["K"],
                                                seed=100 * f + i, zmin=c["minD"], zmax=c["maxD"])
    frames = [[host[f, i] for i in range(len(cams))] for f in range(nF)]

    ctx = capi.Context(0)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", 0))
    out = {"card": card(), "rig": "4 x 1280x960 (composite %d x %d, P = %d)" % (rows, cols, P), "reps": args.reps,
           "warmup": args.warmup}

    # ---- (a) frame preparation
    F = min(args.prep_frames, nF)
    clouds = [ctx.new_cloud(P) for _ in range(nF)]
    prep = {"frames_per_call": F, "batch": {}}
    for setting in (1, 2, 4, 8):
        os.environ["NICP_PREP_BATCH"] = str(setting)
        ms, wall = timed(ctx, stream, lambda: ctx.multi_raw_depth_to_cloud_batch(frames[:F], mp, sp, clouds=clouds[:F]),
                         args.reps, args.warmup)
        prep["batch"]["NICP_PREP_BATCH=%d" % setting] = {"device_ms_per_frame": ms / F, "frames_per_s": F / (ms * 1e-3),
                                                          "wall_ms_per_frame": wall / F}
    os.environ.pop("NICP_PREP_BATCH")
    ms, wall = timed(ctx, stream, lambda: ctx.multi_raw_depth_to_cloud_batch(frames[:F], mp, sp, clouds=clouds[:F]),
                     args.reps, args.warmup)
    prep["batch"]["default"] = {"device_ms_per_frame": ms / F, "frames_per_s": F / (ms * 1e-3), "wall_ms_per_frame": wall / F}
    n_pts = float(np.mean([c.size() for c in clouds[:F]]))

    def host_composite(fr):
        comp = np.zeros((rows, cols), np.float32)
        off = 0
        for r, c in zip(fr, cams):
            comp[:c["width"], off:off + c["height"]] = synth.u16_to_m(r).T
            off += c["height"]
        return comp

    t0 = time.perf_counter()
    comps = [host_composite(frames[f]) for f in range(F)]
    host_ms = (time.perf_counter() - t0) * 1e3 / F
    loop_clouds = [ctx.new_cloud(P) for _ in range(F)]
    ms, wall = timed(ctx, stream, lambda: [ctx.multi_depth_to_cloud(comps[f], mp, sp, cloud=loop_clouds[f]) for f in range(F)],
                     args.reps, args.warmup)
    prep["loop_multi_depth_to_cloud"] = {"device_ms_per_frame": ms / F, "frames_per_s": F / (ms * 1e-3),
                                         "wall_ms_per_frame": wall / F, "host_conversion_ms_per_frame": host_ms}
    for a, b in zip(clouds[:F], loop_clouds):  # the composites carry no scaling (step 1): the same clouds
        assert a.size() == b.size()
    byts = 88.0 * P + 76.0 * n_pts
    prep["points_per_frame"] = n_pts
    prep["algorithmic_MB_per_frame"] = byts / 1e6
    best = min(v["device_ms_per_frame"] for v in prep["batch"].values())
    prep["batch_best_GBps"] = byts / (best * 1e-3) / 1e9
    prep["speedup_default_vs_loop"] = prep["loop_multi_depth_to_cloud"]["device_ms_per_frame"] / prep["batch"]["default"]["device_ms_per_frame"]
    out["prep"] = prep

    # ---- (b) alignment: every current against every candidate, pairs that share a current adjacent
    pairs, guesses = [], []
    for ci in range(args.cur):
        for ri in range(args.cand):
            T_true = np.linalg.inv(cand_poses[ri]) @ cur_poses[ci]
            guesses.append(synth.perturbed_pose(rng, T_true, 0.05, 3.0))
            pairs.append((args.cur + ri, ci))
    guesses = np.stack(guesses).astype(np.float32)
    ctx.multi_raw_depth_to_cloud_batch(frames, mp, sp, clouds=clouds)
    refs = [clouds[r] for r, _ in pairs]
    curs = [clouds[c] for _, c in pairs]
    n = len(pairs)
    res = np.zeros(n, capi.RESULT_DTYPE)
    ms_b, wall_b = timed(ctx, stream, lambda: ctx.multi_align_batch(refs, curs, mp, ap, guesses, results=res), args.reps, args.warmup)
    loop = []
    ms_l, wall_l = timed(ctx, stream, lambda: loop.append([bytes(ctx.multi_align(r, c, mp, ap, guess=g))
                                                           for r, c, g in zip(refs, curs, guesses)]), args.reps, args.warmup)
    same = all(res[i].tobytes() == loop[-1][i] for i in range(n))
    Nr = float(np.mean([r.size() for r in refs]))
    Nc = float(np.mean([c.size() for c in curs]))
    outer = C["outerIterations"]
    midx, macc = float(res["reserved"][:, 0].sum()), float(res["reserved"][:, 1].sum())
    byts = n * ((12 * Nc + 8 * P) + outer * (12 * Nr + 16 * P) + 8 * P) + (56 * midx + 48 * macc) * (1 + 1.0 / outer)
    out["align"] = {"pairs": n, "current_frames": args.cur, "candidate_frames": args.cand,
                    "batch": {"device_ms": ms_b, "pairs_per_s": n / (ms_b * 1e-3), "wall_ms": wall_b},
                    "loop_multi_align": {"device_ms": ms_l, "pairs_per_s": n / (ms_l * 1e-3), "wall_ms": wall_l},
                    "speedup": ms_l / ms_b, "records_identical_to_loop": same,
                    "status_ok": int((res["status"] == 0).sum()), "mean_inliers": float(res["inliers"].mean()),
                    "algorithmic_MB_per_pair": byts / n / 1e6, "batch_GBps": byts / (ms_b * 1e-3) / 1e9}
    ctx.close()
    path = os.path.join(args.out, "rig_batch_timing.json")
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()

"""Kernel tuning harness (not part of the product): times the fused correspondence+linearise kernel and the
whole align step on a 64-pair batch."""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from g2o_frontend_b200 import capi, synth  # noqa: E402


def main():
    n_cur, n_cand = int(os.environ.get("TUNE_CUR", 4)), int(os.environ.get("TUNE_CAND", 16))
    reps = int(os.environ.get("TUNE_REPS", 5))
    raws_cur, raws_cand, pairs, guesses = bench.make_workload(n_cur, n_cand, 0)
    ctx = capi.Context(0)
    C = bench.CONF
    proj = capi.make_projector(synth.K_KINECT, bench.ROWS, bench.COLS, C["minD"], C["maxD"])
    sp = capi.make_stats_params(C["worldRadius"], C["minImageRadius"], C["maxImageRadius"], C["minPoints"],
                                C["curvatureThreshold"], C["omegaCurvatureThreshold"])
    ap = capi.make_align_params(C["inlierDistanceThreshold"], C["inlierNormalAngularThreshold"], C["flatCurvatureThreshold"],
                                C["inlierCurvatureRatioThreshold"], C["inlierMaxChi2"], True, 10, 1)
    clouds = [ctx.raw_depth_to_cloud(r, proj, sp)[0] for r in raws_cur + raws_cand]
    refs = [clouds[n_cur + ri] for ri, ci in pairs]
    curs = [clouds[ci] for ri, ci in pairs]
    res = ctx.align_batch(refs, curs, proj, ap, guesses)
    ctx.set_kernel_timing(True)
    t0 = time.perf_counter()
    for _ in range(reps):
        res = ctx.align_batch(refs, curs, proj, ap, guesses)
    dt = (time.perf_counter() - t0) / reps
    kt = ctx.kernel_timing()
    P = bench.ROWS * bench.COLS
    nl = max(kt["corr_lin_launches"], 1)
    byts = (8.0 * P * len(pairs) * 10 + 56.0 * res["reserved"][:, 0].sum() + 48.0 * res["reserved"][:, 1].sum()) * reps
    gbs = byts / (kt["corr_lin_ms"] * 1e-3) / 1e9
    print("slots=%s pairs=%d: step %.2f ms (%.0f align/s) | corr_lin %.1f us/launch, %.0f GB/s (%.3f of 6540) | "
          "project %.1f us/launch | checksum inliers=%d T00=%.9f" %
          (os.environ.get("NICP_BATCH_SLOTS", "64"), len(pairs), dt * 1e3,
           len(pairs) / dt, kt["corr_lin_ms"] / nl * 1e3, gbs, gbs / 6539.9, kt["project_ms"] / max(kt["project_launches"], 1) * 1e3,
           int(res["inliers"].sum()), float(res["T"][:, 0].mean())))
    ctx.close()


if __name__ == "__main__":
    main()

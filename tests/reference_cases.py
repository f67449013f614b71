"""The cases of tests/test_reference_pwn_core.py, as the oracle's outputs, for tests/golden/reference_cases.npz.

test_reference_pwn_core.py runs each case twice, once through the reference's own pwn_core sources
(oracle/_ref/libpwn_core_ref.so) and once through the oracle, and requires bit-identical results. That library is
built only where the reference sources are, so tests/test_reference_golden.py checks the same cases against stored
outputs instead. Each function below returns one case's outputs as named arrays. Names listed in TOLERANT were
compared with the reference only to rounding, and are checked with the same tolerance.

    python tests/golden/make_reference_golden.py
"""
import ctypes as C

import numpy as np

from conftest import get_scene

CLOUD_FIELDS = ("points", "normals", "statsM", "eigvals", "statsN", "curvature", "omegaP", "omegaN")
TOLERANT = {"omega": 1e-5, "ratios": 1e-4}


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def depth_conversion():
    from oracle import pwn_oracle as O
    S = get_scene(4, seed=3, dropout=0.05)
    d = O.depth_u16_to_f32(S.rawA)
    out = {"depth_f32": d}
    for step in (1, 2, 3, 4, 7):
        out["scale_%d" % step] = O.depth_scale(d, step)
    z = S.depthA.copy()
    z[z == 0] = np.finfo(np.float32).max
    z += np.float32(0.00049)
    b = np.zeros(z.shape, np.uint16)
    O.lib().orc_depth_f32_to_u16(_fp(z), z.size, C.c_float(1000.0), b.ctypes.data_as(C.POINTER(C.c_ushort)))
    out["depth_u16"] = b
    return out


def depth_to_cloud(case):
    S = {"clean": lambda: get_scene(4), "noise_dropout": lambda: get_scene(4, seed=1, dropout=0.05),
         "sensor_offset": lambda: get_scene(4, offset=True), "full_resolution": lambda: get_scene(1)}[case]()
    out = {"index": S.indexA, "interval": S.intervalA, "integral": np.asarray(S.integralA, np.float32)}
    for k in CLOUD_FIELDS:
        out["cloud_" + k] = getattr(S.cloudA, k)
    return out


PROJECTION_POSES = ([0, 0, 0, 0, 0, 0], [0.03, -0.02, 0.05, 0.01, -0.015, 0.005], [-0.2, 0.1, 0.3, -0.05, 0.08, 0.02],
                    [0.5, 0.0, -1.0, 0.0, 0.3, 0.0])


def projection():
    from oracle import pwn_oracle as O
    S = get_scene(4)
    c = S.conf
    out = {}
    for j, v in enumerate(PROJECTION_POSES):
        T = O.v2t(np.array(v, np.float32))
        out["index_%d" % j], out["depth_%d" % j] = O.project(S.cloudA.points, S.rows, S.cols, S.K, T, c["minD"], c["maxD"])
        out["unprojected_%d" % j], out["unprojected_index_%d" % j] = O.unproject(S.depthA, S.K, T, c["minD"], c["maxD"])
    return out


def finder_linearizer(threads, robust):
    from oracle import pwn_oracle as O
    S = get_scene(4, seed=2)
    c = S.conf
    T = O.v2t(np.array([0.01, -0.02, 0.015, 0.004, -0.003, 0.002], np.float32))
    ri, _ = O.project(S.cloudA.points, S.rows, S.cols, S.K, np.linalg.inv(T).astype(np.float32), c["minD"], c["maxD"])
    ci, _ = O.project(S.cloudB.points, S.rows, S.cols, S.K, np.eye(4, dtype=np.float32), c["minD"], c["maxD"])
    chi2 = 9e3 if robust else 60.0
    corr, _ = O.correspond(ri, ci, S.cloudA, S.cloudB, T, S.cp, num_threads=threads)
    H, b, err, inl = O.linearize(corr, S.cloudA, S.cloudB, T, chi2, robust, num_threads=threads)
    return {"corr": corr, "H": H, "b": b, "error": np.float32(err), "inliers": np.int64(inl)}


ALIGN_CASES = ("identity_guess", "perturbed_guess_4_threads", "inner_iterations", "sensor_offset", "one_iteration",
               "thirteen_iterations")


def align(case):
    from g2o_frontend_b200 import synth
    from oracle import pwn_oracle as O
    S = get_scene(4, offset=(case == "sensor_offset"))
    kw = {"identity_guess": dict(), "perturbed_guess_4_threads": dict(guess=synth.make_pose((0.02, 0.01, -0.03), (0.1, 1.0, 0.3), 1.5),
                                                                      threads=4),
          "inner_iterations": dict(inner=3, outer=4), "sensor_offset": dict(), "one_iteration": dict(outer=1),
          "thirteen_iterations": dict(outer=13)}[case]
    ap = S.oracle_align_params(outer=kw.get("outer"), inner=kw.get("inner"), guess=kw.get("guess"), num_threads=kw.get("threads", 1))
    o = O.align(S.cloudA, S.cloudB, ap)
    return {"T": o.T, "error": np.float32(o.error), "inliers": np.int64(o.inliers), "n": np.int64(o.numCorrespondences),
            "refIndex": o.refIndex, "curIndex": o.curIndex, "refDepth": o.refDepth, "curDepth": o.curDepth, "corr": o.corr,
            "omega": o.omega, "ratios": np.array([o.translationalRatio, o.rotationalRatio], np.float32)}


def align_with_priors():
    from g2o_frontend_b200 import synth
    from oracle import pwn_oracle as O
    S = get_scene(4)
    c = S.conf
    mean = synth.make_pose((0.03, -0.02, 0.05), (0.2, 1.0, 0.1), 2.0)
    info = np.diag([2000, 2000, 2000, 5000, 5000, 5000]).astype(np.float32)
    reference = synth.make_pose((0.5, 0.1, -0.2), (0.0, 1.0, 0.0), 10.0)
    absmean = (reference @ mean).astype(np.float32)
    out = {}
    for name, priors in (("relative", [O.make_prior(0, mean, info)]), ("absolute", [O.make_prior(1, absmean, info, reference)]),
                         ("both", [O.make_prior(0, mean, info), O.make_prior(1, absmean, info, reference)])):
        ap = O.make_align_params(S.K, S.rows, S.cols, c["minD"], c["maxD"], S.cp, max_chi2=c["inlierMaxChi2"], num_threads=1,
                                 priors=priors)
        o = O.align(S.cloudA, S.cloudB, ap)
        out[name + "_T"], out[name + "_inliers"], out[name + "_error"] = o.T, np.int64(o.inliers), np.float32(o.error)
    return out


def voxel_as_written(res):
    from test_map_ops import two_frame_map
    from oracle import pwn_oracle as O
    m, _, _ = two_frame_map(get_scene(4, 0, 0.05, True))
    return {"points": m.points[O.voxelize(m.points, res, strict=False)]}


def multi_projection(ragged):
    from g2o_frontend_b200 import synth
    from oracle import pwn_oracle as O
    cams = synth.make_rig(3 if ragged else 4, 64, 48, K=synth.scaled_K(synth.K_KINECT, 64 / 640.0))
    if ragged:
        cams[1]["width"], cams[1]["height"] = 48, 40
        cams[2]["maxD"] = 3.0
    om = O.make_multi(cams)
    rows, cols = O.multi_image_size(om)
    S = get_scene(4)
    out = {}
    for j, pose in enumerate((np.eye(4, dtype=np.float32), synth.make_pose((0.1, -0.05, 0.2), (0, 1, 0), 10.0),
                              synth.make_pose((-0.3, 0.1, 1.0), (0.2, 1.0, 0.1), 75.0))):
        out["index_%d" % j], out["depth_%d" % j] = O.multi_project(om, pose.astype(np.float32), S.cloudA.points, rows, cols)
    return out


def all_cases():
    """case id -> function returning its outputs; the ids are those of test_reference_pwn_core.py's parameters"""
    cases = {"depth_conversion": depth_conversion, "projection": projection, "align_with_priors": align_with_priors}
    for c in ("clean", "noise_dropout", "sensor_offset", "full_resolution"):
        cases["depth_to_cloud-" + c] = lambda c=c: depth_to_cloud(c)
    for robust in (True, False):
        for threads in (1, 2, 3, 4, 7, 8, 16):
            cases["finder_linearizer-%s-%d" % (robust, threads)] = lambda t=threads, r=robust: finder_linearizer(t, r)
    for c in ALIGN_CASES:
        cases["align-" + c] = lambda c=c: align(c)
    for res in (0.01, 0.05, 0.2):
        cases["voxel_as_written-%g" % res] = lambda r=res: voxel_as_written(r)
    for ragged in (False, True):
        cases["multi_projection-%s" % ragged] = lambda g=ragged: multi_projection(g)
    return cases

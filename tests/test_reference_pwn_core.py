"""The oracle against the REFERENCE'S OWN pwn_core sources.

oracle/build_ref_pwn_core.sh compiles g2o_frontend/pwn_core/*.cpp from /root/reference against the Eigen / OpenCV
stand-ins of oracle/shim/ into oracle/_ref/libpwn_core_ref.so (extern "C" face: oracle/ref_pwn_core.cpp).  Every loop,
index computation, clamp, gate, branch, accumulation order and OpenMP chunking below is therefore the reference's code
as written; what Eigen would compute inside (fixed-size products in index order, computeDirect, LDLT, ...) is supplied
by the stand-in, the numerical kernels by the oracle's own restatements -- those stay "parity unpinned" (DESIGN.md 2).

The bar is BIT-EXACT for everything up to and including H, b and the alignment result (same arithmetic, same order),
which is what makes the oracle a restatement rather than an approximation of the reference.  CPU only; runs here and
on the GPU box (the prebuilt .so travels)."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import ROOT, get_scene

REF_SO = os.path.join(ROOT, "oracle", "_ref", "libpwn_core_ref.so")


def fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


def cm(M):
    return np.ascontiguousarray(np.asarray(M, np.float32).T.reshape(-1))


@pytest.fixture(scope="module")
def R():
    # skip here rather than for the whole module: tests that run the reference's programs carry their own skip, and
    # test_host_classes_with_a_mock_backend needs no reference at all
    if not os.path.exists(REF_SO):
        pytest.skip("oracle/_ref/libpwn_core_ref.so not built (oracle/Makefile builds it where the reference sources are)")
    from oracle import pwn_oracle as O
    O.lib()  # liboracle.so (the stand-in's numerical kernels resolve against it) is loaded first
    L = C.CDLL(REF_SO)
    L.refcore_depth_to_cloud.restype = C.c_void_p
    L.refcore_set_threads(1)
    return L


class RefCloud:
    """a pwn::Cloud built by the reference's DepthImageConverterIntegralImage::compute"""

    def __init__(self, R, depth, K, conf, sensor_offset=None):
        rows, cols = depth.shape
        self.R = R
        sp = np.array([conf["worldRadius"], conf["minImageRadius"], conf["maxImageRadius"], conf["minPoints"],
                       conf["curvatureThreshold"], conf["omegaCurvatureThreshold"]], np.float32)
        self.index = np.zeros((rows, cols), np.int32)
        self.interval = np.zeros((rows, cols), np.int32)
        self.integral = np.zeros((rows, cols, 10), np.float32)
        off = cm(np.eye(4) if sensor_offset is None else sensor_offset)
        self.h = C.c_void_p(R.refcore_depth_to_cloud(fp(np.ascontiguousarray(depth, np.float32)), rows, cols, fp(cm(K)),
                                                     C.c_float(conf["minD"]), C.c_float(conf["maxD"]), fp(sp), fp(off),
                                                     ip(self.index), ip(self.interval), fp(self.integral)))
        n = self.n = R.refcore_cloud_size(self.h)
        self.points = np.zeros((n, 4), np.float32)
        self.normals = np.zeros((n, 4), np.float32)
        self.statsM = np.zeros((n, 16), np.float32)
        self.eigvals = np.zeros((n, 3), np.float32)
        self.statsN = np.zeros(n, np.int32)
        self.curvature = np.zeros(n, np.float32)
        self.omegaP = np.zeros((n, 16), np.float32)
        self.omegaN = np.zeros((n, 16), np.float32)
        self.fetch()

    def fetch(self):
        self.R.refcore_cloud_get(self.h, fp(self.points), fp(self.normals), fp(self.statsM), fp(self.eigvals), ip(self.statsN),
                                 fp(self.curvature), fp(self.omegaP), fp(self.omegaN))

    def __del__(self):
        try:
            self.R.refcore_cloud_free(self.h)
        except Exception:
            pass


def same_cloud(ref, orc):
    assert ref.n == orc.n
    for k in ("points", "normals", "statsM", "eigvals", "statsN", "curvature", "omegaP", "omegaN"):
        a, b = getattr(ref, k), getattr(orc, k)
        assert np.array_equal(a, b, equal_nan=True), (k, int((a != b).sum()))


def finder_params(conf):
    return np.array([conf["inlierDistanceThreshold"], conf["inlierNormalAngularThreshold"], conf["flatCurvatureThreshold"],
                     conf["inlierCurvatureRatioThreshold"]], np.float32)


# ---------------------------------------------------------------------------------------------------------------
def test_depth_conversion_and_scaling(R):
    """pwn_static.cpp:5-68"""
    from oracle import pwn_oracle as O
    S = get_scene(4, seed=3, dropout=0.05)
    raw = S.rawA
    d = np.zeros(raw.shape, np.float32)
    R.refcore_depth_u16_to_f32(raw.ctypes.data_as(C.POINTER(C.c_ushort)), raw.shape[0], raw.shape[1], C.c_float(0.001), fp(d))
    assert np.array_equal(d, O.depth_u16_to_f32(raw))
    for step in (1, 2, 3, 4, 7):
        out = np.zeros((raw.shape[0] // step, raw.shape[1] // step), np.float32)
        R.refcore_depth_scale(fp(d), raw.shape[0], raw.shape[1], step, C.c_float(0.01), fp(out))
        assert np.array_equal(out, O.depth_scale(d, step)), step
    # DepthImage_convert_32FC1_to_16UC1 (pwn_static.cpp:38-52), the first step of matchClouds' image statistics: a z-buffer
    # with empty pixels at FLT_MAX -> millimetres, truncated, 0 where empty
    z = S.depthA.copy()
    z[z == 0] = np.finfo(np.float32).max
    z += np.float32(0.00049)
    a = np.zeros(z.shape, np.uint16)
    b = np.zeros(z.shape, np.uint16)
    R.refcore_depth_f32_to_u16(fp(z), z.shape[0], z.shape[1], C.c_float(1000.0), a.ctypes.data_as(C.POINTER(C.c_ushort)))
    O.lib().orc_depth_f32_to_u16(fp(z), z.size, C.c_float(1000.0), b.ctypes.data_as(C.POINTER(C.c_ushort)))
    assert np.array_equal(a, b) and (a > 0).sum() > 1000 and (a == 0).sum() > 0


@pytest.mark.parametrize("case", ["clean", "noise_dropout", "sensor_offset", "full_resolution"])
def test_depth_to_cloud_is_bit_identical(R, case):
    """DepthImageConverterIntegralImage::compute: unProject, projectIntervals, PointIntegralImage (all 10 channels, every
    pixel), StatsCalculatorIntegralImage (region clamps, minPoints, eigen-decomposition, curvature, normal flip),
    Point/NormalInformationMatrixCalculator, Cloud::transformInPlace"""
    S = {"clean": lambda: get_scene(4), "noise_dropout": lambda: get_scene(4, seed=1, dropout=0.05),
         "sensor_offset": lambda: get_scene(4, offset=True), "full_resolution": lambda: get_scene(1)}[case]()
    ref = RefCloud(R, S.depthA, S.K, S.conf, S.sensor_offset)
    assert np.array_equal(ref.index, S.indexA)
    assert np.array_equal(ref.interval, S.intervalA)
    assert np.array_equal(ref.integral.reshape(-1), np.asarray(S.integralA, np.float32).reshape(-1))
    same_cloud(ref, S.cloudA)
    assert (np.abs(ref.normals[:, :3]).sum(1) > 0).mean() > 0.5  # not vacuous: most points have a normal


def test_projection_is_bit_identical(R):
    """PinholePointProjector::project (z-buffer: nearest wins, first index wins ties, empty = FLT_MAX / -1) and the
    3-argument unProject at a non-identity pose"""
    from oracle import pwn_oracle as O
    S = get_scene(4)
    c = S.conf
    ref = RefCloud(R, S.depthA, S.K, c)
    for v in ([0, 0, 0, 0, 0, 0], [0.03, -0.02, 0.05, 0.01, -0.015, 0.005], [-0.2, 0.1, 0.3, -0.05, 0.08, 0.02],
              [0.5, 0.0, -1.0, 0.0, 0.3, 0.0]):
        T = O.v2t(np.array(v, np.float32))
        ii = np.zeros((S.rows, S.cols), np.int32)
        dd = np.zeros((S.rows, S.cols), np.float32)
        R.refcore_project(ref.h, fp(cm(S.K)), fp(cm(T)), S.rows, S.cols, C.c_float(c["minD"]), C.c_float(c["maxD"]), ip(ii), fp(dd))
        oi, od = O.project(S.cloudA.points, S.rows, S.cols, S.K, T, c["minD"], c["maxD"])
        assert np.array_equal(ii, oi) and np.array_equal(dd, od), v
        pts = np.zeros((S.rows * S.cols, 4), np.float32)
        idx = np.zeros((S.rows, S.cols), np.int32)
        n = R.refcore_unproject(fp(np.ascontiguousarray(S.depthA)), S.rows, S.cols, fp(cm(S.K)), fp(cm(T)), C.c_float(c["minD"]),
                                C.c_float(c["maxD"]), fp(pts), ip(idx))
        opts, oidx = O.unproject(S.depthA, S.K, T, c["minD"], c["maxD"])
        assert n == len(opts) and np.array_equal(pts[:n], opts) and np.array_equal(idx, oidx), v


@pytest.mark.parametrize("threads", [1, 2, 3, 4, 7, 8, 16])
@pytest.mark.parametrize("robust", [True, False])
def test_finder_and_linearizer_are_bit_identical(R, threads, robust):
    """CorrespondenceFinder::compute + Linearizer::update, including what the reference's OpenMP partitioning does for
    every thread count: rows % numThreads rows are never searched (correspondencefinder.cpp:38), numCorrespondences %
    numThreads correspondences are never linearised (linearizer.cpp:32-39), per-thread float32 partial sums added in
    thread order."""
    from oracle import pwn_oracle as O
    S = get_scene(4, seed=2)
    c = S.conf
    refA, refB = RefCloud(R, S.depthA, S.K, c), RefCloud(R, S.depthB, S.K, c)
    T = O.v2t(np.array([0.01, -0.02, 0.015, 0.004, -0.003, 0.002], np.float32))
    ri, _ = O.project(S.cloudA.points, S.rows, S.cols, S.K, np.linalg.inv(T).astype(np.float32), c["minD"], c["maxD"])
    ci, _ = O.project(S.cloudB.points, S.rows, S.cols, S.K, np.eye(4, dtype=np.float32), c["minD"], c["maxD"])
    chi2 = 9e3 if robust else 60.0
    R.refcore_set_threads(threads)
    try:
        corr = np.full((S.rows * S.cols, 2), -1, np.int32)
        H = np.zeros(36, np.float32)
        b = np.zeros(6, np.float32)
        err, inl = C.c_float(0), C.c_int(0)
        n = R.refcore_correspond_linearize(refA.h, refB.h, ip(np.ascontiguousarray(ri)), ip(np.ascontiguousarray(ci)), S.rows,
                                           S.cols, fp(cm(T)), fp(finder_params(c)), C.c_float(chi2), int(robust), ip(corr),
                                           fp(H), fp(b), C.byref(err), C.byref(inl))
    finally:
        R.refcore_set_threads(1)
    ocorr, _ = O.correspond(ri, ci, S.cloudA, S.cloudB, T, S.cp, num_threads=threads)
    oH, ob, oe, oinl = O.linearize(ocorr, S.cloudA, S.cloudB, T, chi2, robust, num_threads=threads)
    assert n == len(ocorr) > 5000
    assert np.array_equal(corr[:n], ocorr)
    assert inl.value == oinl and err.value == oe
    assert np.array_equal(H.reshape(6, 6).T, oH) and np.array_equal(b, ob)


def run_ref_align(R, refA, refB, S, outer=10, inner=1, guess=None, ref_off=None, cur_off=None, priors=(), chi2=None, threads=1):
    c = S.conf
    P = S.rows * S.cols
    out = dict(T=np.zeros(16, np.float32), omega=np.zeros(36, np.float32), ratios=np.zeros(2, np.float32),
               refIndex=np.zeros((S.rows, S.cols), np.int32), refDepth=np.zeros((S.rows, S.cols), np.float32),
               curIndex=np.zeros((S.rows, S.cols), np.int32), curDepth=np.zeros((S.rows, S.cols), np.float32),
               corr=np.full((P, 2), -1, np.int32))
    err, inl = C.c_float(0), C.c_int(0)
    eye = np.eye(4, dtype=np.float32)
    pr = np.zeros(max(len(priors), 1) * 69, np.float32)
    for j, (kind, mean, info, reference) in enumerate(priors):
        pr[69 * j] = kind
        pr[69 * j + 1:69 * j + 17] = cm(mean)
        pr[69 * j + 17:69 * j + 33] = cm(eye if reference is None else reference)
        pr[69 * j + 33:69 * j + 69] = cm(info)
    R.refcore_set_threads(threads)
    try:
        n = R.refcore_align(refA.h, refB.h, fp(cm(S.K)), S.rows, S.cols, C.c_float(c["minD"]), C.c_float(c["maxD"]),
                            fp(finder_params(c)), C.c_float(c["inlierMaxChi2"] if chi2 is None else chi2), 1, outer, inner,
                            fp(cm(eye if guess is None else guess)), fp(cm(eye if ref_off is None else ref_off)),
                            fp(cm(eye if cur_off is None else cur_off)), fp(pr), len(priors), fp(out["T"]), fp(out["omega"]),
                            C.byref(err), C.byref(inl), fp(out["ratios"]), ip(out["refIndex"]), fp(out["refDepth"]),
                            ip(out["curIndex"]), fp(out["curDepth"]), ip(out["corr"]))
    finally:
        R.refcore_set_threads(1)
    out["n"] = n
    out["error"], out["inliers"] = err.value, inl.value
    out["T"] = out["T"].reshape(4, 4).T.copy()
    out["omega"] = out["omega"].reshape(6, 6).T.copy()
    return out


@pytest.mark.parametrize("case", ["identity_guess", "perturbed_guess_4_threads", "inner_iterations", "sensor_offset",
                                  "one_iteration", "thirteen_iterations"])
def test_align_is_bit_identical(R, case):
    """Aligner::align free-running: projection of the current cloud, then per outer iteration projection of the reference
    cloud, finder, lineariser, damping, LDLT step, v2t / t2v renormalisation -- T, error, inliers, the finder's index and
    depth images and the correspondence list of the last iteration all bit-identical; omega and the eigen-ratios of
    _computeStatistics to rounding."""
    from g2o_frontend_b200 import synth
    S = get_scene(4, offset=(case == "sensor_offset"))
    refA = RefCloud(R, S.depthA, S.K, S.conf, S.sensor_offset)
    refB = RefCloud(R, S.depthB, S.K, S.conf, S.sensor_offset)
    kw = {"identity_guess": dict(), "perturbed_guess_4_threads": dict(guess=synth.make_pose((0.02, 0.01, -0.03), (0.1, 1.0, 0.3), 1.5), threads=4),
          "inner_iterations": dict(inner=3, outer=4), "sensor_offset": dict(ref_off=S.sensor_offset, cur_off=S.sensor_offset),
          "one_iteration": dict(outer=1), "thirteen_iterations": dict(outer=13)}[case]
    ref = run_ref_align(R, refA, refB, S, **kw)
    from oracle import pwn_oracle as O
    ap = S.oracle_align_params(outer=kw.get("outer"), inner=kw.get("inner"), guess=kw.get("guess"), num_threads=kw.get("threads", 1))
    orc = O.align(S.cloudA, S.cloudB, ap)
    assert np.array_equal(ref["T"], orc.T), np.abs(ref["T"] - orc.T).max()
    assert ref["error"] == orc.error and ref["inliers"] == orc.inliers and ref["n"] == orc.numCorrespondences
    assert np.array_equal(ref["refIndex"], orc.refIndex) and np.array_equal(ref["curIndex"], orc.curIndex)
    assert np.array_equal(ref["refDepth"], orc.refDepth) and np.array_equal(ref["curDepth"], orc.curDepth)
    assert np.array_equal(ref["corr"][:ref["n"]], orc.corr)
    assert np.abs(ref["omega"] - orc.omega).max() <= 1e-5 * np.abs(orc.omega).max()
    assert abs(ref["ratios"][0] - orc.translationalRatio) <= 1e-4 * orc.translationalRatio
    assert abs(ref["ratios"][1] - orc.rotationalRatio) <= 1e-4 * orc.rotationalRatio
    # and the alignment is a real one: it recovers the ground-truth motion of the synthetic pair
    if kw.get("outer", 10) >= 10 and case != "sensor_offset":
        assert np.abs(ref["T"] - S.gt).max() < 5e-3


def test_align_with_priors_is_bit_identical(R):
    """SE3RelativePrior / SE3AbsolutePrior (se3_prior.cpp:8-71) inside the Gauss-Newton step (aligner.cpp:97-108)"""
    from oracle import pwn_oracle as O
    from g2o_frontend_b200 import synth
    S = get_scene(4)
    refA, refB = RefCloud(R, S.depthA, S.K, S.conf), RefCloud(R, S.depthB, S.K, S.conf)
    mean = synth.make_pose((0.03, -0.02, 0.05), (0.2, 1.0, 0.1), 2.0)
    info = np.diag([2000, 2000, 2000, 5000, 5000, 5000]).astype(np.float32)
    reference = synth.make_pose((0.5, 0.1, -0.2), (0.0, 1.0, 0.0), 10.0)
    absmean = (reference @ mean).astype(np.float32)
    for name, priors, opriors in (
            ("relative", [(0, mean, info, None)], [O.make_prior(0, mean, info)]),
            ("absolute", [(1, absmean, info, reference)], [O.make_prior(1, absmean, info, reference)]),
            ("both", [(0, mean, info, None), (1, absmean, info, reference)],
             [O.make_prior(0, mean, info), O.make_prior(1, absmean, info, reference)])):
        ref = run_ref_align(R, refA, refB, S, priors=priors)
        c = S.conf
        ap = O.make_align_params(S.K, S.rows, S.cols, c["minD"], c["maxD"], S.cp, max_chi2=c["inlierMaxChi2"], num_threads=1,
                                 priors=opriors)
        orc = O.align(S.cloudA, S.cloudB, ap)
        assert np.array_equal(ref["T"], orc.T), (name, np.abs(ref["T"] - orc.T).max())
        assert ref["inliers"] == orc.inliers and ref["error"] == orc.error, name


# ---- local-map maintenance (SURVEY.md section 8f rank 3) -------------------------------------------------------
def ref_gaussians(R, cloud):
    g = np.zeros((cloud.n, 24), np.float32)
    f = np.zeros(cloud.n, np.int32)
    n = R.refcore_cloud_gaussians(cloud.h, fp(g), ip(f))
    return g[:n], f[:n]


def ref_two_frame_map(R, S):
    A = RefCloud(R, S.depthA, S.K, S.conf, S.sensor_offset)
    B = RefCloud(R, S.depthB, S.K, S.conf, S.sensor_offset)
    R.refcore_cloud_add(A.h, B.h, fp(cm(S.gt)))  # Cloud::add (cloud.cpp:145-171)
    n = A.n = R.refcore_cloud_size(A.h)
    for k, w in (("points", 4), ("normals", 4), ("statsM", 16), ("eigvals", 3), ("omegaP", 16), ("omegaN", 16)):
        setattr(A, k, np.zeros((n, w), np.float32))
    A.statsN, A.curvature = np.zeros(n, np.int32), np.zeros(n, np.float32)
    A.fetch()
    return A


def test_gaussians_add_and_merge_are_bit_identical(R):
    """unProject with the Gaussian3f sensor model (pinholepointprojector.cpp:93-133) + Gaussian3fVector::transformInPlace,
    Cloud::add of a transformed cloud, and Merger::merge (merger.cpp:15-119) on the two-frame map"""
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_map_ops import two_frame_map, BASELINE, ALPHA
    from oracle import pwn_oracle as O
    S = get_scene(4, 0, 0.05, True)
    c = S.conf
    one = RefCloud(R, S.depthA, S.K, c, S.sensor_offset)
    g, f = ref_gaussians(R, one)
    og, of, _, _ = O.unproject_gaussians(S.depthA, S.K, c["minD"], c["maxD"], BASELINE, ALPHA, S.sensor_offset)
    assert np.array_equal(f, of)
    assert np.array_equal(g[:, :12], og[:, :12])  # moments form after the sensor offset; the info form is not valid yet
    m, mg, mf = two_frame_map(S)
    ref = ref_two_frame_map(R, S)
    for k in ("points", "normals", "statsM", "omegaP", "omegaN"):
        assert np.array_equal(getattr(ref, k), getattr(m, k)), k
    rg, rf = ref_gaussians(R, ref)
    assert np.array_equal(rf, mf) and np.array_equal(rg[:, :12], mg[:, :12])
    for T, thr in ((np.eye(4, dtype=np.float32), (0.1, float(np.cos(np.float32(10 * np.pi / 180.0))), 10.0)),
                   (S.gt, (0.05, 0.99, 3.0))):
        ref = ref_two_frame_map(R, S)
        n0 = ref.n
        col = np.zeros(n0, np.int32)
        k = R.refcore_merge(ref.h, fp(cm(S.K)), fp(cm(T)), S.rows, S.cols, C.c_float(c["minD"]), C.c_float(c["maxD"]),
                            C.c_float(thr[0]), C.c_float(thr[1]), C.c_float(thr[2]), ip(col))
        res, g2, f2, ocol = O.merge(m, mg, mf, S.rows, S.cols, S.K, T, c["minD"], c["maxD"], *thr)
        assert np.array_equal(col, ocol)
        assert k == res.n < n0
        ref.n = k
        for name, w in (("points", 4), ("normals", 4), ("statsM", 16), ("omegaP", 16), ("omegaN", 16)):
            setattr(ref, name, np.zeros((k, w), np.float32))
        ref.eigvals, ref.statsN, ref.curvature = np.zeros((k, 3), np.float32), np.zeros(k, np.int32), np.zeros(k, np.float32)
        ref.fetch()
        for name in ("points", "normals", "statsM", "omegaP", "omegaN"):
            assert np.array_equal(getattr(ref, name), getattr(res, name)), name
        # the reference forgets gaussians().resize(k) (merger.cpp:108-113): compare the first k
        rg = np.zeros((n0, 24), np.float32)
        rf = np.zeros(n0, np.int32)
        R.refcore_cloud_gaussians(ref.h, fp(rg), ip(rf))
        assert np.array_equal(rf[:k], f2)
        mom, inf = (f2 & 1) != 0, (f2 & 2) != 0
        assert np.array_equal(rg[:k][mom, :12], g2[mom, :12]) and np.array_equal(rg[:k][inf, 12:], g2[inf, 12:])


@pytest.mark.parametrize("res", [0.01, 0.05, 0.2])
def test_voxelcalculator_as_written(R, res):
    """VoxelCalculator::compute with the reference's own comparator (not a strict weak ordering, voxelcalculator.h:40-46)
    in libstdc++'s std::map: oracle/voxel_oracle.cpp in its as-written mode reproduces the reference's output exactly;
    the lexicographic order the CUDA path implements keeps a subset of it (DESIGN.md, known deviations)."""
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_map_ops import two_frame_map
    from oracle import pwn_oracle as O
    S = get_scene(4, 0, 0.05, True)
    m, _, _ = two_frame_map(S)
    ref = ref_two_frame_map(R, S)
    k = R.refcore_voxelize(ref.h, C.c_float(res))
    pts = np.zeros((k, 4), np.float32)
    R.refcore_cloud_get(ref.h, fp(pts), None, None, None, None, None, None, None)
    raw = O.voxelize(m.points, res, strict=False)
    assert k == len(raw) and np.array_equal(pts, m.points[raw])
    lex = O.voxelize(m.points, res, strict=True)
    assert set(lex.tolist()) <= set(raw.tolist())


@pytest.mark.parametrize("ragged", [False, True])
def test_multipointprojector_projection_is_bit_identical(R, ragged):
    """BASELINE config 5: the projection Aligner::align really runs for a MultiPointProjector -- the const base-class
    z-buffer PointProjector::project (pointprojector.cpp:17-40) over the per-point MultiPointProjector::project
    (multipointprojector.cpp:157-205): first camera that sees the point wins, composite pixel (u, v + column offset),
    empty depth 0."""
    from g2o_frontend_b200 import synth
    from oracle import pwn_oracle as O
    cams = synth.make_rig(3 if ragged else 4, 64, 48, K=synth.scaled_K(synth.K_KINECT, 64 / 640.0))
    if ragged:
        cams[1]["width"], cams[1]["height"] = 48, 40
        cams[2]["maxD"] = 3.0
    om = O.make_multi(cams)
    rows, cols = O.multi_image_size(om)
    S = get_scene(4)
    ref = RefCloud(R, S.depthA, S.K, S.conf)
    packed = np.zeros((len(cams), 29), np.float32)
    for i, c in enumerate(cams):
        packed[i, :9] = cm(c["K"])
        packed[i, 9:25] = cm(c["offset"])
        packed[i, 25:29] = c["width"], c["height"], c["minD"], c["maxD"]
    seen = 0
    for pose in (np.eye(4, dtype=np.float32), synth.make_pose((0.1, -0.05, 0.2), (0, 1, 0), 10.0),
                 synth.make_pose((-0.3, 0.1, 1.0), (0.2, 1.0, 0.1), 75.0)):
        ii = np.zeros((rows, cols), np.int32)
        dd = np.zeros((rows, cols), np.float32)
        R.refcore_multi_project(ref.h, fp(packed), len(cams), fp(cm(pose)), rows, cols, ip(ii), fp(dd))
        oi, od = O.multi_project(om, pose.astype(np.float32), S.cloudA.points, rows, cols)
        assert np.array_equal(ii, oi) and np.array_equal(dd, od)
        seen += int((ii >= 0).sum())
    assert seen > 1000


def test_committed_golden_fixtures_are_what_the_reference_computes(R):
    """tests/golden/small_pair.npz and map_ops_small.npz (written by the oracle, tests/golden/make_golden.py; the GPU tests
    and tests/test_oracle.py read them) certified by the reference's own sources: frame prep of both frames, the
    free-running 10-iteration alignment, Merger::merge and VoxelCalculator on the two-frame map."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "small_pair.npz"))
    conf = dict(worldRadius=0.1, minImageRadius=3, maxImageRadius=6, minPoints=10, curvatureThreshold=0.2,
                omegaCurvatureThreshold=0.02, minD=0.5, maxD=4.5, inlierDistanceThreshold=0.5, inlierNormalAngularThreshold=0.95,
                flatCurvatureThreshold=0.02, inlierCurvatureRatioThreshold=1.3, inlierMaxChi2=9e3)
    K = g["K"]
    A, B = RefCloud(R, g["depthA"], K, conf), RefCloud(R, g["depthB"], K, conf)
    sym = [0, 4, 8, 5, 9, 10]  # xx xy xz yy yz zz of a column-major 4x4
    for c, s in ((A, "A"), (B, "B")):
        assert np.array_equal(c.points, g["points" + s]) and np.array_equal(c.normals, g["normals" + s])
        assert np.array_equal(c.curvature, g["curvature" + s])
        assert np.array_equal(c.omegaP[:, sym], g["omegaP" + s]) and np.array_equal(c.omegaN[:, sym], g["omegaN" + s])
    assert np.array_equal(A.eigvals, g["eigvalsA"]) and np.array_equal(A.statsN, g["statsNA"])
    assert np.array_equal(A.index, g["indexA"]) and np.array_equal(A.interval, g["intervalA"])
    assert np.array_equal(A.integral.reshape(-1), g["integralA"].reshape(-1))

    class S:
        pass
    S.conf, S.K = conf, K
    S.rows, S.cols = g["depthA"].shape
    out = run_ref_align(R, A, B, S)
    assert np.array_equal(out["T"], g["T"]) and out["error"] == float(g["error"]) and out["inliers"] == int(g["inliers"])
    assert out["n"] == int(g["numCorr"]) and np.array_equal(out["corr"][:out["n"]], g["corr"])
    assert np.array_equal(out["refIndex"], g["refIndex"]) and np.array_equal(out["refDepth"], g["refDepth"])
    assert np.array_equal(out["curIndex"], g["curIndex"])
    assert np.abs(out["omega"] - g["omega"]).max() <= 1e-5 * np.abs(g["omega"]).max()
    # the trace of the fixture: T at the start of every outer iteration = the result of an alignment cut short there
    for k in (1, 4, 9):
        assert np.array_equal(run_ref_align(R, A, B, S, outer=k)["T"], g["trace_T"][k])

    m = np.load(os.path.join(ROOT, "tests", "golden", "map_ops_small.npz"))
    R.refcore_cloud_add(A.h, B.h, fp(cm(m["T"])))
    n = R.refcore_cloud_size(A.h)
    pts = np.zeros((n, 4), np.float32)
    nrm = np.zeros((n, 4), np.float32)
    R.refcore_cloud_get(A.h, fp(pts), fp(nrm), None, None, None, None, None, None)
    assert np.array_equal(pts, m["map_points"]) and np.array_equal(nrm, m["map_normals"])
    gg = np.zeros((n, 24), np.float32)
    ff = np.zeros(n, np.int32)
    R.refcore_cloud_gaussians(A.h, fp(gg), ip(ff))
    assert np.array_equal(ff, m["map_flags"]) and np.array_equal(gg[:, :12], m["map_gauss"][:, :12])
    # VoxelCalculator on a copy of the map (the reference's comparator as written), then Merger::merge on the map
    V = RefCloud(R, g["depthA"], K, conf)
    R.refcore_cloud_add(V.h, B.h, fp(cm(m["T"])))
    k = R.refcore_voxelize(V.h, C.c_float(0.05))
    vp = np.zeros((k, 4), np.float32)
    R.refcore_cloud_get(V.h, fp(vp), None, None, None, None, None, None, None)
    assert np.array_equal(vp, m["map_points"][m["voxel_rep_as_written"]])
    col = np.zeros(n, np.int32)
    k = R.refcore_merge(A.h, fp(cm(K)), fp(cm(np.eye(4))), S.rows, S.cols, C.c_float(0.5), C.c_float(4.5), C.c_float(0.1),
                        C.c_float(float(np.cos(np.float32(10 * np.pi / 180.0)))), C.c_float(10.0), ip(col))
    assert np.array_equal(col, m["collapsed"]) and k == len(m["merged_points"])
    mp = np.zeros((k, 4), np.float32)
    R.refcore_cloud_get(A.h, fp(mp), None, None, None, None, None, None, None)
    assert np.array_equal(mp, m["merged_points"])


@pytest.mark.parametrize("seed", [0, 1])
def test_randomised_differential(R, seed):
    """200 random small cases per seed -- ragged image sizes down to 1x1, random / planar / holed / wavy / range-boundary
    depth images, random camera, radii, minPoints, thresholds, sensor offsets, 1-8 threads, 1-4 outer and 1-2 inner
    iterations: frame prep and the whole alignment of the oracle and of the reference's own sources stay bit-identical.
    (Skipped where the reference itself is undefined: an empty cloud makes it take &points[0] of an empty vector.)"""
    from oracle import pwn_oracle as O
    rng = np.random.default_rng(seed)
    done = 0
    for it in range(200):
        rows = int(rng.choice([1, 2, 3, 5, 8, 13, 24, 37, 48]))
        cols = int(rng.choice([1, 2, 4, 7, 16, 31, 53, 64]))
        f = float(rng.uniform(20, 120))
        K = np.array([[f, 0, (cols - 1) / 2 + rng.uniform(-2, 2)], [0, f * rng.uniform(0.9, 1.1), (rows - 1) / 2 + rng.uniform(-2, 2)],
                      [0, 0, 1]], np.float32)
        kind = int(rng.integers(5))
        yy, xx = np.mgrid[0:rows, 0:cols]
        if kind == 0:
            d = rng.uniform(0.3, 5.0, (rows, cols))
        elif kind == 1:
            d = 1.5 + 0.01 * xx + 0.02 * yy + rng.normal(0, 0.002, (rows, cols))
        elif kind == 2:
            d = np.full((rows, cols), 2.0)
            d[rng.random((rows, cols)) < 0.3] = 0
        elif kind == 3:
            d = 1.0 + 0.5 * np.sin(xx / 3.0) + 0.3 * np.cos(yy / 2.0)
        else:  # values on and next to the [minDistance, maxDistance] boundaries
            d = np.where(rng.random((rows, cols)) < 0.5, 0.5, 4.5) + rng.choice([0, 1e-7, -1e-7], (rows, cols))
        if rng.random() < 0.5:
            d = np.round(d * 1000) / 1000
        d = np.ascontiguousarray(d, np.float32)
        conf = dict(worldRadius=float(rng.choice([0.05, 0.1, 0.3])), minImageRadius=int(rng.integers(1, 5)),
                    maxImageRadius=int(rng.integers(5, 12)), minPoints=int(rng.choice([1, 3, 10, 50])),
                    curvatureThreshold=float(rng.choice([0.02, 0.2, 1.0])), omegaCurvatureThreshold=float(rng.choice([0.002, 0.02, 0.5])),
                    minD=0.5, maxD=4.5, inlierDistanceThreshold=float(rng.choice([0.1, 0.5, 1.0])),
                    inlierNormalAngularThreshold=float(rng.choice([0.5, 0.95, 0.999])),
                    flatCurvatureThreshold=float(rng.choice([0.002, 0.02, 0.2])),
                    inlierCurvatureRatioThreshold=float(rng.choice([1.05, 1.3, 3.0])), inlierMaxChi2=float(rng.choice([10.0, 9e3])))
        off = None
        if rng.random() < 0.4:
            off = O.v2t(np.concatenate([rng.uniform(-0.3, 0.3, 3), rng.uniform(-0.2, 0.2, 3)]).astype(np.float32))
        sp = O.default_stats_params(minImageRadius=conf["minImageRadius"], maxImageRadius=conf["maxImageRadius"],
                                    minPoints=conf["minPoints"], curvatureThreshold=conf["curvatureThreshold"],
                                    worldRadius=conf["worldRadius"], omegaCurvatureThreshold=conf["omegaCurvatureThreshold"])
        oc, oidx, oitv, ointeg = O.depth_to_cloud(d, K, conf["minD"], conf["maxD"], sp, off, want_aux=True)
        d2 = np.roll(d, 1, axis=1).copy()
        oc2, _ = O.depth_to_cloud(d2, K, conf["minD"], conf["maxD"], sp, off)
        if oc.n == 0 or oc2.n == 0:
            continue
        rc, rc2 = RefCloud(R, d, K, conf, off), RefCloud(R, d2, K, conf, off)
        tag = (seed, it, rows, cols, kind)
        assert np.array_equal(rc.index, oidx) and np.array_equal(rc.interval, oitv), tag
        assert np.array_equal(rc.integral.reshape(-1), np.asarray(ointeg, np.float32).reshape(-1)), tag
        same_cloud(rc, oc)

        class S:
            pass
        S.conf, S.K, S.rows, S.cols = conf, K, rows, cols
        nt = int(rng.choice([1, 2, 3, 8]))
        guess = O.v2t(np.concatenate([rng.uniform(-0.02, 0.02, 3), rng.uniform(-0.01, 0.01, 3)]).astype(np.float32))
        outer, inner = int(rng.integers(1, 5)), int(rng.integers(1, 3))
        ref = run_ref_align(R, rc, rc2, S, outer=outer, inner=inner, guess=guess, ref_off=off, cur_off=off, threads=nt)
        cp = O.default_corr_params(inlierDistanceThreshold=conf["inlierDistanceThreshold"],
                                   inlierNormalAngularThreshold=conf["inlierNormalAngularThreshold"],
                                   flatCurvatureThreshold=conf["flatCurvatureThreshold"],
                                   inlierCurvatureRatioThreshold=conf["inlierCurvatureRatioThreshold"])
        ap = O.make_align_params(K, rows, cols, conf["minD"], conf["maxD"], cp, outer=outer, inner=inner, guess=guess,
                                 ref_offset=off, cur_offset=off, max_chi2=conf["inlierMaxChi2"], num_threads=nt)
        orc = O.align(oc, oc2, ap)
        assert np.array_equal(ref["T"], orc.T, equal_nan=True), tag
        assert ref["inliers"] == orc.inliers and ref["n"] == orc.numCorrespondences, tag
        assert ref["error"] == orc.error or (np.isnan(ref["error"]) and np.isnan(orc.error)), tag
        assert np.array_equal(ref["refIndex"], orc.refIndex) and np.array_equal(ref["curIndex"], orc.curIndex), tag
        assert np.array_equal(ref["refDepth"], orc.refDepth) and np.array_equal(ref["curDepth"], orc.curDepth), tag
        done += 1
    assert done > 150


# ---- the drop-in binding (INTEGRATION.md option A) ------------------------------------------------------------------
DEMO = os.path.join(ROOT, "oracle", "_ref", "drop_in_demo")


def run_drop_in_demo(S, which, tmp_path, priors=False):
    """oracle/_ref/drop_in_demo: one program on the reference's own classes, reference CPU arm and / or B200 arm"""
    import json
    import subprocess
    if not os.access(DEMO, os.X_OK):
        os.chmod(DEMO, 0o755)
    a, b = str(tmp_path / "a.f32"), str(tmp_path / "b.f32")
    np.ascontiguousarray(S.depthA, np.float32).tofile(a)
    np.ascontiguousarray(S.depthB, np.float32).tofile(b)
    c = S.conf
    args = [DEMO, a, b, str(S.rows), str(S.cols)] + [repr(float(S.K[i, j])) for i, j in ((0, 0), (1, 1), (0, 2), (1, 2))] + \
           [str(c["minImageRadius"]), str(c["maxImageRadius"]), str(c["minPoints"]), repr(float(c["inlierDistanceThreshold"])), which] + \
           (["priors"] if priors else [])
    o = subprocess.run(args, capture_output=True, text=True, timeout=600)
    return o.returncode, json.loads(o.stdout), o.stderr


@pytest.mark.skipif(not os.path.exists(DEMO), reason="oracle/_ref/drop_in_demo not built")
def test_drop_in_binding_compiles_against_the_reference_headers_and_fails_loudly_without_a_gpu(tmp_path):
    """integration/pwn_b200/b200_pwn.h (B200DepthImageConverter / B200Aligner, subclasses of the reference's own
    DepthImageConverterIntegralImage / Aligner) is compiled against the reference's headers into drop_in_demo.  Its
    reference arm reproduces the oracle bit for bit; its B200 arm has no CPU fallback."""
    import torch
    from oracle import pwn_oracle as O
    S = get_scene(4)
    rc, out, _ = run_drop_in_demo(S, "cpu", tmp_path)
    assert rc == 0
    r = out["reference_cpu"]
    orc = O.align(S.cloudA, S.cloudB, S.oracle_align_params(num_threads=1))
    assert np.array_equal(np.array(r["T"], np.float32).reshape(4, 4), orc.T)
    assert r["inliers"] == orc.inliers and r["num_correspondences"] == orc.numCorrespondences
    assert r["reference_points"] == S.cloudA.n and r["current_points"] == S.cloudB.n
    if not torch.cuda.is_available():
        rc, out, _ = run_drop_in_demo(S, "gpu", tmp_path)
        assert rc == 3 and "no CPU fallback" in out["b200_error"]


def test_library_host_helpers_match_the_reference(R):
    """The part of the PRODUCT that runs without a GPU -- libnicp_b200.so's host-side nicp_update_matrices / nicp_v2t /
    nicp_t2v, the same functions the device code is compiled from (nicp_math.cuh) -- against the reference's
    PinholePointProjector::_updateMatrices and bm_se3.h: bit-identical."""
    from g2o_frontend_b200 import capi
    rng = np.random.default_rng(5)
    for verify in (False, True):
        L = capi.load(verify)
        for _ in range(500):
            v = np.concatenate([rng.uniform(-2, 2, 3), rng.uniform(-0.55, 0.55, 3)]).astype(np.float32)
            Tr, Tl = np.zeros(16, np.float32), np.zeros(16, np.float32)
            R.refcore_v2t(fp(v), fp(Tr))
            L.nicp_v2t(fp(v), fp(Tl))
            assert np.array_equal(Tr, Tl)
            vr, vl = np.zeros(6, np.float32), np.zeros(6, np.float32)
            R.refcore_t2v(fp(Tr), fp(vr))
            L.nicp_t2v(fp(Tr), fp(vl))
            assert np.array_equal(vr, vl, equal_nan=True)
            f = float(rng.uniform(100, 1100))
            K = np.array([[f, 0, rng.uniform(100, 700)], [0, f * rng.uniform(0.95, 1.05), rng.uniform(100, 500)], [0, 0, 1]], np.float32)
            a, b, c, d = (np.zeros(16, np.float32) for _ in range(4))
            R.refcore_update_matrices(fp(cm(K)), fp(Tr), fp(a), fp(b))
            L.nicp_update_matrices(fp(cm(K)), fp(Tr), fp(c), fp(d))
            assert np.array_equal(a, c) and np.array_equal(b, d)


def test_real_kinect_frame_is_bit_identical(R):
    """real sensor data (holes, noise, 0.4-8 m range): the one Kinect frame the reference ships as data (tests/golden/
    real_depth_640x480.npz), full resolution, parameters of pwn_aligner_1_1.conf -- frame prep and the self-alignment
    from a perturbed guess, oracle vs the reference's own sources"""
    from conftest import CONF_1_1
    from g2o_frontend_b200 import synth
    from oracle import pwn_oracle as O
    raw = np.load(os.path.join(ROOT, "tests", "golden", "real_depth_640x480.npz"))["raw"]
    c = CONF_1_1
    K = synth.K_KINECT
    d = O.depth_u16_to_f32(raw)
    sp = O.default_stats_params(minImageRadius=c["minImageRadius"], maxImageRadius=c["maxImageRadius"], minPoints=c["minPoints"],
                                curvatureThreshold=c["curvatureThreshold"])
    oc, oidx, oitv, ointeg = O.depth_to_cloud(d, K, c["minD"], c["maxD"], sp, want_aux=True)
    rc = RefCloud(R, d, K, c)
    assert np.array_equal(rc.index, oidx) and np.array_equal(rc.interval, oitv)
    assert np.array_equal(rc.integral.reshape(-1), np.asarray(ointeg, np.float32).reshape(-1))
    same_cloud(rc, oc)
    assert oc.n > 0.5 * raw.size
    guess = synth.make_pose((0.02, -0.01, 0.015), (0.3, 1.0, 0.2), 1.5).astype(np.float32)

    class S:
        pass
    S.conf, S.K, S.rows, S.cols = c, K, 480, 640
    for threads in (1, 8):
        ref = run_ref_align(R, rc, rc, S, guess=guess, threads=threads)
        cp = O.default_corr_params(inlierDistanceThreshold=c["inlierDistanceThreshold"],
                                   inlierNormalAngularThreshold=c["inlierNormalAngularThreshold"])
        orc = O.align(oc, oc, O.make_align_params(K, 480, 640, c["minD"], c["maxD"], cp, guess=guess, num_threads=threads))
        assert np.array_equal(ref["T"], orc.T) and ref["inliers"] == orc.inliers and ref["error"] == orc.error
        assert np.array_equal(ref["refIndex"], orc.refIndex) and np.array_equal(ref["corr"][:ref["n"]], orc.corr)
        assert np.abs(ref["T"] - np.eye(4)).max() < 5e-3  # a frame aligned with itself: identity


# ---- the reference's own CLI driver (BASELINE config 0 / 1) -----------------------------------------------------------
REF_CLI = os.path.join(ROOT, "oracle", "_ref", "pwn_simple_aligner_ref")


def run_reference_cli(tmp_path, raws, conf, image_scale, threads=1, initial=None):
    """pwn_core/pwn_simple_aligner.cpp, compiled unmodified: config file, list of depth images, odometry file out.
    Returns the global poses (4x4) it wrote, one per frame."""
    import subprocess
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_host_cpp import write_conf, write_pgm16
    if not os.access(REF_CLI, os.X_OK):
        os.chmod(REF_CLI, 0o755)
    lst = str(tmp_path / "frames.txt")
    with open(lst, "w") as f:
        for i, r in enumerate(raws):
            p = str(tmp_path / ("ref_depth%d.pgm" % i))
            write_pgm16(p, r)
            f.write("%d.5 %s\n" % (100 + i, p))
    cfg = str(tmp_path / "ref_aligner.conf")
    write_conf(cfg, conf, image_scale, [0, 0, 0, 0, 0, 0], extra=initial)
    odo = str(tmp_path / "ref_odometry.txt")
    subprocess.run([REF_CLI, cfg, lst, odo], check=True, capture_output=True, timeout=900,
                   env=dict(os.environ, OMP_NUM_THREADS=str(threads)))
    poses = []
    for line in open(odo):
        v = [float(x) for x in line.split()[1:]]
        x, y, z, qx, qy, qz, qw = v
        Rm = np.array([[1 - 2 * (qy * qy + qz * qz), 2 * (qx * qy - qz * qw), 2 * (qx * qz + qy * qw)],
                       [2 * (qx * qy + qz * qw), 1 - 2 * (qx * qx + qz * qz), 2 * (qy * qz - qx * qw)],
                       [2 * (qx * qz - qy * qw), 2 * (qy * qz + qx * qw), 1 - 2 * (qx * qx + qy * qy)]])
        T = np.eye(4)
        T[:3, :3], T[:3, 3] = Rm, (x, y, z)
        poses.append(T)
    return poses


@pytest.mark.skipif(not os.path.exists(REF_CLI), reason="oracle/_ref/pwn_simple_aligner_ref not built")
def test_reference_cli_driver_against_the_oracle_chain(tmp_path):
    """BASELINE configs[0], "the reference's own CPU-runnable case": pwn_simple_aligner on three synthetic frames
    (16-bit PGM in, imageScale 4, parameters of pwn_aligner_1_4.conf).  The odometry it writes equals the oracle's chain
    depth_u16_to_f32 -> depth_scale -> depth_to_cloud -> align(previous, current), composed (the text file carries 6
    significant digits)."""
    from conftest import CONF_1_4
    from g2o_frontend_b200 import synth
    from oracle import pwn_oracle as O
    conf = CONF_1_4
    poses = [synth.POSE_A, synth.POSE_B, synth.POSE_B @ synth.make_pose((-0.02, 0.01, 0.03), (1.0, 0.3, 0.2), 1.5)]
    raws = [synth.render_depth_u16(p, seed=3 + i) for i, p in enumerate(poses)]
    got = run_reference_cli(tmp_path, raws, conf, 4)
    assert len(got) == 3
    K = synth.scaled_K(synth.K_KINECT, 0.25)
    sp = O.default_stats_params(minImageRadius=conf["minImageRadius"], maxImageRadius=conf["maxImageRadius"],
                                minPoints=conf["minPoints"], curvatureThreshold=conf["curvatureThreshold"],
                                worldRadius=conf["worldRadius"], omegaCurvatureThreshold=conf["omegaCurvatureThreshold"])
    cp = O.default_corr_params(inlierDistanceThreshold=conf["inlierDistanceThreshold"],
                               inlierNormalAngularThreshold=conf["inlierNormalAngularThreshold"],
                               flatCurvatureThreshold=conf["flatCurvatureThreshold"],
                               inlierCurvatureRatioThreshold=conf["inlierCurvatureRatioThreshold"])
    clouds = [O.depth_to_cloud(O.depth_scale(O.depth_u16_to_f32(r), 4), K, conf["minD"], conf["maxD"], sp)[0] for r in raws]
    G = np.eye(4, dtype=np.float32)
    assert np.abs(got[0] - np.eye(4)).max() < 1e-6
    for i in (1, 2):
        ap = O.make_align_params(K, 120, 160, conf["minD"], conf["maxD"], cp, max_chi2=conf["inlierMaxChi2"], num_threads=1)
        o = O.align(clouds[i - 1], clouds[i], ap)
        G = (G.astype(np.float64) @ o.T.astype(np.float64)).astype(np.float32)
        assert np.abs(got[i] - G).max() < 2e-5, (i, got[i], G)
    # and it is an odometry: the composed motion is the ground truth of the synthetic sequence
    assert np.abs(got[2] - poses[2]).max() < 1e-2


REF_MAP_CLI = os.path.join(ROOT, "oracle", "_ref", "pwn_aligner_ref")


def oracle_scene_odometry(raws, conf, scale, chunk_step=10):
    """pwn_core/pwn_aligner.cpp:129-222 restated over the oracle: every frame is aligned against the local map re-rendered
    at the predicted pose, added (Cloud::add) and fused (Merger::merge); after the first alignment and then every
    chunk_step frames the map is closed and a new one starts from the current frame (chunk_step 0: never).
    Returns the global pose and the map size after every frame."""
    from g2o_frontend_b200 import synth
    from oracle import pwn_oracle as O
    f32 = np.float32
    K = (synth.K_KINECT * (f32(1.0) / f32(scale))).astype(f32)
    K[2, 2] = 1.0
    rows, cols = 480 // scale, 640 // scale
    sp = O.default_stats_params(minImageRadius=conf["minImageRadius"], maxImageRadius=conf["maxImageRadius"],
                                minPoints=conf["minPoints"], curvatureThreshold=conf["curvatureThreshold"],
                                worldRadius=conf["worldRadius"], omegaCurvatureThreshold=conf["omegaCurvatureThreshold"])
    cp = O.default_corr_params(inlierDistanceThreshold=conf["inlierDistanceThreshold"],
                               inlierNormalAngularThreshold=conf["inlierNormalAngularThreshold"],
                               flatCurvatureThreshold=conf["flatCurvatureThreshold"],
                               inlierCurvatureRatioThreshold=conf["inlierCurvatureRatioThreshold"])
    def mul(A, B):  # Isometry3f * Isometry3f in float32 as Eigen does it (R = Ra Rb, t = Ra tb + ta), last row rewritten
        out = np.zeros(16, f32)
        O.lib().orc_iso_mul(fp(O.colmajor(A)), fp(O.colmajor(B)), fp(out))
        M = out.reshape(4, 4).T.copy()
        M[3] = (0, 0, 0, 1)
        return M
    globalT, sceneT = np.eye(4, dtype=f32), np.eye(4, dtype=f32)
    scene = sg = sf = None
    counter = 0
    poses, sizes = [], []
    for i, r in enumerate(raws):
        d = O.depth_scale(O.depth_u16_to_f32(r), scale)
        cloud = O.depth_to_cloud(d, K, conf["minD"], conf["maxD"], sp)[0]
        g, f, _, _ = O.unproject_gaussians(d, K, conf["minD"], conf["maxD"], 0.075, 0.1)
        if i > 0:
            _, rendered = O.project(scene.points, rows, cols, K, sceneT, conf["minD"], conf["maxD"])
            sub = O.depth_to_cloud(rendered, K, conf["minD"], conf["maxD"], sp)[0]
            o = O.align(sub, cloud, O.make_align_params(K, rows, cols, conf["minD"], conf["maxD"], cp,
                                                       max_chi2=conf["inlierMaxChi2"], num_threads=1))
            globalT, sceneT = mul(globalT, o.T), mul(sceneT, o.T)
            if chunk_step > 0:
                if counter % chunk_step == 0:
                    sceneT = np.eye(4, dtype=f32)
                    scene = sg = sf = None
                counter += 1
        pts, nrm, st, op, on = (cloud.points.copy(), cloud.normals.copy(), cloud.statsM.copy(), cloud.omegaP.copy(), cloud.omegaN.copy())
        O.lib().orc_cloud_transform(fp(O.colmajor(sceneT)), cloud.n, fp(pts), fp(nrm), fp(st), fp(op), fp(on))
        g, f = O.gaussians_transform(sceneT, g, f)
        parts = [] if scene is None else [scene]
        m = O.Cloud((0 if scene is None else scene.n) + cloud.n)
        cat = lambda name, new: np.ascontiguousarray(np.concatenate([getattr(p, name) for p in parts] + [new]))
        m.points, m.normals, m.statsM = cat("points", pts), cat("normals", nrm), cat("statsM", st)
        m.omegaP, m.omegaN = cat("omegaP", op), cat("omegaN", on)
        m.eigvals, m.statsN, m.curvature = cat("eigvals", cloud.eigvals), cat("statsN", cloud.statsN), cat("curvature", cloud.curvature)
        mg = g if scene is None else np.concatenate([sg, g])
        mf = f if scene is None else np.concatenate([sf, f])
        scene, sg, sf, _ = O.merge(m, mg, mf, rows, cols, K, sceneT, conf["minD"], conf["maxD"])
        poses.append(globalT.copy())
        sizes.append(scene.n)
    return poses, sizes


def run_reference_map_cli(tmp_path, raws, conf, image_scale, chunk_step=None, initial=None):
    """pwn_core/pwn_aligner.cpp compiled unmodified: global poses it wrote, one per frame"""
    import subprocess
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_host_cpp import write_conf, write_pgm16
    if not os.access(REF_MAP_CLI, os.X_OK):
        os.chmod(REF_MAP_CLI, 0o755)
    lst = str(tmp_path / "map_frames.txt")
    with open(lst, "w") as f:
        for i, r in enumerate(raws):
            p = str(tmp_path / ("map_depth%d.pgm" % i))
            write_pgm16(p, r)
            f.write("%d.5 %s\n" % (100 + i, p))
    cfg = str(tmp_path / "map_aligner.conf")
    extra = dict(initial or {})
    if chunk_step is not None:
        extra["chunkStep"] = chunk_step
    write_conf(cfg, conf, image_scale, [0, 0, 0, 0, 0, 0], extra=extra)
    odo = str(tmp_path / "map_odometry.txt")
    subprocess.run([REF_MAP_CLI, cfg, lst, odo], check=True, capture_output=True, timeout=900, cwd=str(tmp_path),
                   env=dict(os.environ, OMP_NUM_THREADS="1"))
    poses = []
    for line in open(odo):
        x, y, z, qx, qy, qz, qw = [float(v) for v in line.split()[1:]]
        Rm = np.array([[1 - 2 * (qy * qy + qz * qz), 2 * (qx * qy - qz * qw), 2 * (qx * qz + qy * qw)],
                       [2 * (qx * qy + qz * qw), 1 - 2 * (qx * qx + qz * qz), 2 * (qy * qz - qx * qw)],
                       [2 * (qx * qz - qy * qw), 2 * (qy * qz + qx * qw), 1 - 2 * (qx * qx + qy * qy)]])
        T = np.eye(4)
        T[:3, :3], T[:3, 3] = Rm, (x, y, z)
        poses.append(T)
    return poses


def map_sequence(n=6):
    from g2o_frontend_b200 import synth
    poses = [synth.POSE_A]
    step = synth.make_pose((0.015, -0.01, 0.02), (0.2, 1.0, 0.1), 1.0)
    for _ in range(n - 1):
        poses.append(poses[-1] @ step)
    return poses, [synth.render_depth_u16(p, seed=40 + i) for i, p in enumerate(poses)]


@pytest.mark.skipif(not os.path.exists(REF_MAP_CLI), reason="oracle/_ref/pwn_aligner_ref not built")
@pytest.mark.parametrize("chunk_step", [None, 2])
def test_reference_scene_odometry_driver_against_the_oracle_chain(tmp_path, chunk_step):
    """pwn_core/pwn_aligner.cpp (align against the re-rendered local map, Cloud::add, Merger::merge, a new map after the
    first alignment and every chunkStep frames) on six synthetic frames: its odometry equals the oracle's restatement"""
    from conftest import CONF_1_4
    gt, raws = map_sequence(6)
    got = run_reference_map_cli(tmp_path, raws, CONF_1_4, 4, chunk_step)
    want, sizes = oracle_scene_odometry(raws, CONF_1_4, 4, 10 if chunk_step is None else chunk_step)
    assert len(got) == len(want) == 6
    for i in range(6):
        assert np.abs(got[i] - want[i]).max() < 3e-5, (i, got[i], want[i])
    rel = np.linalg.inv(gt[0]) @ gt[-1]
    assert np.abs(got[-1][:3, 3] - rel[:3, 3]).max() < 2e-2


@pytest.mark.parametrize("binary", [0, 1])
def test_pwn_cloud_files_are_exchanged_with_the_reference(R, tmp_path, binary):
    """.pwn cloud files (SURVEY.md 8f rank 4): written by the reference's Cloud::save (cloud.cpp:82-133), read and written
    back by pwn::Cloud::load / save of include/pwn/pwn.h (a CPU-only program), read by the reference's Cloud::load
    (cloud.cpp:25-80).  Binary mode dumps the reference's C++ objects raw -- 32 B per Point, 32 B per Normal, 112 B per
    Stats on LP64 (vptr, padding, payload) -- which is what the header documents, reads and writes."""
    import subprocess
    sizes = (C.c_int * 3)()
    R.refcore_object_sizes(sizes)
    assert list(sizes) == [32, 32, 112]
    S = get_scene(4, seed=1, dropout=0.05)
    rc = RefCloud(R, S.depthA, S.K, S.conf)
    from g2o_frontend_b200 import synth
    T = synth.make_pose((0.3, -0.2, 0.5), (0.2, 1.0, 0.1), 12.0).astype(np.float32)
    a, b = str(tmp_path / "reference.pwn"), str(tmp_path / "ours.pwn")
    assert R.refcore_cloud_save(rc.h, a.encode(), fp(cm(T)), 1, binary) == 1
    exe = str(tmp_path / "pwn_file_roundtrip")
    lib = os.path.join(ROOT, "g2o_frontend_b200", "lib")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([cxx, "-std=c++17", "-O1", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"), "-o", exe,
                           os.path.join(ROOT, "tests", "cpp", "pwn_file_roundtrip.cpp"), "-L", lib, "-lnicp_b200",
                           "-Wl,-rpath," + lib])
    out = subprocess.run([exe, a, b, str(binary)], capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0 and int(out.stdout.split()[0]) == rc.n, out.stdout + out.stderr
    T2 = np.zeros(16, np.float32)
    R.refcore_cloud_load.restype = C.c_void_p
    h = R.refcore_cloud_load(b.encode(), fp(T2))
    assert h
    h = C.c_void_p(h)
    try:
        n = R.refcore_cloud_size(h)
        assert n == rc.n
        pts, nrm, st = np.zeros((n, 4), np.float32), np.zeros((n, 4), np.float32), np.zeros((n, 16), np.float32)
        ev, cnt = np.zeros((n, 3), np.float32), np.zeros(n, np.int32)
        R.refcore_cloud_get(h, fp(pts), fp(nrm), fp(st), fp(ev), ip(cnt), None, None, None)
        if binary:
            assert np.array_equal(pts, rc.points) and np.array_equal(nrm, rc.normals) and np.array_equal(st, rc.statsM)
            assert np.array_equal(ev, rc.eigvals) and np.array_equal(cnt, rc.statsN)
            assert np.abs(T2.reshape(4, 4).T - T).max() < 1e-5  # the pose line is text in both modes
        else:  # text with 6 significant digits
            assert np.allclose(pts, rc.points, rtol=2e-5, atol=1e-6) and np.allclose(nrm, rc.normals, rtol=2e-5, atol=1e-6)
            assert np.allclose(st, rc.statsM, rtol=2e-5, atol=1e-6)
    finally:
        # The reference's binary load reads each Point / Normal / Stats object raw, VPTR INCLUDED (cloud.cpp:72-75).  A file
        # is therefore only safe to destroy again in the process image that wrote it; our writer stores zeros there (and
        # our reader ignores those bytes), so the cloud the reference loaded from it is deliberately leaked here: its
        # element destructors are virtual calls through that pointer.
        if not binary:
            R.refcore_cloud_free(h)


def build_mock_backend(tmp_path):
    """tests/cpp/mock_nicp_backend.c (a test double of the C-ABI answered by the oracle) -> <tmp>/mock/libnicp_b200.so"""
    import subprocess
    from oracle import pwn_oracle as O
    O.lib()
    O.voxelize(np.zeros((1, 4), np.float32), 0.01)  # makes sure libvoxel_oracle.so is built
    mock = tmp_path / "mock"
    mock.mkdir()
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    build = os.path.join(ROOT, "oracle", "build")
    subprocess.check_call([cc, "-std=gnu11", "-O1", "-w", "-shared", "-fPIC", "-I", os.path.join(ROOT, "include"), "-I",
                           os.path.join(ROOT, "oracle"), "-o", str(mock / "libnicp_b200.so"),
                           os.path.join(ROOT, "tests", "cpp", "mock_nicp_backend.c"), "-L", build, "-loracle", "-lvoxel_oracle",
                           "-Wl,-rpath," + build])
    return mock


@pytest.mark.skipif(not os.path.exists(DEMO), reason="oracle/_ref/drop_in_demo not built")
def test_drop_in_binding_logic_with_a_mock_backend(tmp_path):
    """The binding's own logic (integration/pwn_b200/b200_pwn.h: buffer layouts, device-mirror bookkeeping, the state it
    publishes into the reference's finder / lineariser objects) end to end without a GPU: for this one subprocess a test
    double (tests/cpp/mock_nicp_backend.c, the dozen nicp_* calls the binding makes, answered by the oracle) is put in front
    of the real library.  The B200 arm of drop_in_demo must then reproduce its reference arm exactly.  The real library is
    what tests/test_vs_reference_gpu.py runs the same program with on a B200."""
    import json
    import subprocess
    mock = build_mock_backend(tmp_path)
    S = get_scene(4)
    a, b = str(tmp_path / "a.f32"), str(tmp_path / "b.f32")
    np.ascontiguousarray(S.depthA, np.float32).tofile(a)
    np.ascontiguousarray(S.depthB, np.float32).tofile(b)
    c = S.conf
    args = [DEMO, a, b, str(S.rows), str(S.cols)] + [repr(float(S.K[i, j])) for i, j in ((0, 0), (1, 1), (0, 2), (1, 2))] + \
           [str(c["minImageRadius"]), str(c["maxImageRadius"]), str(c["minPoints"]), repr(float(c["inlierDistanceThreshold"])), "both"]
    plain = None
    for extra in ([], ["priors"]):  # without and with SE(3) priors (Aligner::addRelativePrior / addAbsolutePrior -> nicp_prior[])
        o = subprocess.run(args + extra, capture_output=True, text=True, timeout=600, env=dict(os.environ, LD_LIBRARY_PATH=str(mock)))
        assert o.returncode == 0, o.stdout + o.stderr
        out = json.loads(o.stdout)
        cpu, dev = out["reference_cpu"], out["b200"]
        assert dev["T"] == cpu["T"], extra
        for k in ("reference_points", "current_points", "inliers", "num_correspondences", "reference_pixels", "error", "gaussians",
                  "gaussian_sum"):
            assert dev[k] == cpu[k], (k, extra)
        assert cpu["gaussians"] == cpu["reference_points"] and cpu["gaussian_sum"] > 0
        if not extra:
            plain = cpu["T"]
    assert plain != cpu["T"]  # the priors really changed the solution


@pytest.mark.skipif(not (os.path.exists(REF_CLI) and os.path.exists(REF_MAP_CLI)), reason="reference CLI drivers not built")
def test_host_drivers_against_the_reference_drivers_with_a_mock_backend(tmp_path, monkeypatch):
    """The HOST logic of this repository's CLI driver (pwn:: classes of include/pwn/pwn.h, frame-to-frame odometry and the
    scene-based odometry with its local map, Merger, chunkStep) against the reference's own drivers, without a GPU: the
    two comparisons of tests/test_vs_reference_gpu.py are run with the test double of the C-ABI in front of the real
    library, so every numerical answer is the oracle's and any disagreement is a defect of the host-side flow."""
    import test_vs_reference_gpu as TG
    mock = build_mock_backend(tmp_path)
    monkeypatch.setenv("LD_LIBRARY_PATH", str(mock))
    (tmp_path / "cli").mkdir()
    (tmp_path / "map").mkdir()
    TG.test_cli_driver_against_the_reference_cli_driver(tmp_path / "cli")
    TG.test_scene_odometry_driver_against_the_reference_driver(tmp_path / "map")


def test_host_classes_with_a_mock_backend(tmp_path, monkeypatch):
    """include/pwn/*.h and the CLI driver's other modes without a GPU: the GPU tests of tests/test_host_cpp.py -- CLI odometry
    at 160x120 and 640x480, the 3-level pyramid (pwn/pyramid.h, BASELINE config 2), the keyframe tracker (pwn/tracker.h,
    config 3), .pwn file I/O + Cloud::add, configuration through BOSS records -- run with the test double of the C-ABI in
    front of the real library.  Every numerical answer is then the oracle's, so these check the host-side flow (what is
    called, in which order, with which matrices) and nothing else."""
    import test_host_cpp as TH
    if not os.path.exists(TH.BIN):
        pytest.skip("host driver not built")
    mock = build_mock_backend(tmp_path)
    monkeypatch.setenv("LD_LIBRARY_PATH", str(mock))
    for i, (fn, args) in enumerate([(TH.test_cli_driver_matches_oracle, (4,)), (TH.test_cli_driver_matches_oracle, (1,)),
                                    (TH.test_pyramid_matches_oracle_composition, ()),
                                    (TH.test_sequential_tracker_matches_oracle_loop, ()),
                                    (TH.test_cloud_file_io_and_add, ()),
                                    (TH.test_cloud_value_semantics_and_host_mirror, ()),
                                    (TH.test_cli_driver_accepts_boss_configuration, ())]):
        d = tmp_path / ("case%d" % i)
        d.mkdir()
        fn(d, *args)


def run_both_drivers_with_the_reference_command_line(tmp_path, image_scale=4, initial=None):
    """`driver config list odometry` -- the reference's own three-argument command line -- once with the reference's
    pwn_simple_aligner (oracle/_ref) and once with this repository's driver.  Returns the two odometry texts and, per frame,
    the two .pwn files they left next to the depth images."""
    import subprocess
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from conftest import CONF_1_1, CONF_1_4
    from g2o_frontend_b200 import synth
    from test_host_cpp import BIN, write_conf, write_pgm16
    conf = CONF_1_1 if image_scale == 1 else CONF_1_4
    poses = [synth.POSE_A, synth.POSE_B, synth.POSE_B @ synth.make_pose((-0.02, 0.01, 0.03), (1.0, 0.3, 0.2), 1.5)]
    raws = [synth.render_depth_u16(p, seed=3 + i) for i, p in enumerate(poses)]
    out = {}
    for who, exe in (("reference", REF_CLI), ("ours", BIN)):
        d = tmp_path / who
        d.mkdir()
        lst = str(d / "frames.txt")
        with open(lst, "w") as f:
            f.write("# timestamp depthFilename\n")
            for i, r in enumerate(raws):
                p = str(d / ("depth%d.pgm" % i))
                write_pgm16(p, r)
                f.write("%d.25 %s\n" % (1000 + i, p))
        cfg = str(d / "aligner.conf")
        write_conf(cfg, conf, image_scale, [0, 0, 0, 0, 0, 0], extra=initial)
        odo = str(d / "odometry.txt")
        if not os.access(exe, os.X_OK):
            os.chmod(exe, 0o755)
        subprocess.run([exe, cfg, lst, odo], check=True, capture_output=True, timeout=900, env=dict(os.environ, OMP_NUM_THREADS="1"))
        out[who] = (open(odo).read(), [str(d / ("depth%d.pgm.pwn" % i)) for i in range(len(raws))])
    return out


def pwn_payload(path):
    """points, normals, Stats matrix, n, eigenvalues of a binary .pwn file (the vptr / padding bytes of the raw object dump
    are skipped: cloud.cpp:116-124, 32 + 32 + 112 bytes per point)"""
    data = open(path, "rb").read()
    head_end = data.index(b"\n", data.index(b"\n") + 1) + 1
    n = int(data.split()[1])
    rec = np.frombuffer(data, np.uint8, n * 176, head_end).reshape(n, 176)
    f = lambda a, b: np.ascontiguousarray(rec[:, a:b]).view(np.float32)
    return f(16, 32), f(48, 64), f(80, 144), np.ascontiguousarray(rec[:, 144:148]).view(np.int32)[:, 0], f(148, 160)


@pytest.mark.skipif(not os.path.exists(REF_CLI), reason="oracle/_ref/pwn_simple_aligner_ref not built")
def test_same_command_line_same_files_as_the_reference_driver(tmp_path, monkeypatch):
    """Drop-in at the command line: `pwn_simple_aligner config list odometry` with the reference's binary and with this
    repository's driver (behind the test double of the C-ABI, so that every number is the oracle's): the odometry files
    are identical BYTE FOR BYTE and the .pwn clouds left next to the frames carry identical payloads."""
    mock = build_mock_backend(tmp_path)
    monkeypatch.setenv("LD_LIBRARY_PATH", str(mock))
    start = dict(tx=0.4, ty=-0.1, tz=0.25, qx=0.05, qy=-0.1, qz=0.02, qw=0.9935290634701167)
    for k, initial in enumerate((None, start)):
        d = tmp_path / ("run%d" % k)
        d.mkdir()
        out = run_both_drivers_with_the_reference_command_line(d, 4, initial)
        assert out["ours"][0] == out["reference"][0] and len(out["ours"][0].splitlines()) == 3
        for a, b in zip(out["ours"][1], out["reference"][1]):
            pa, pb = pwn_payload(a), pwn_payload(b)
            assert open(a, "rb").read().split(b"\n")[:2] == open(b, "rb").read().split(b"\n")[:2]  # header + pose line
            for x, y in zip(pa, pb):
                assert np.array_equal(x, y, equal_nan=True)


@pytest.mark.skipif(not os.path.exists(REF_MAP_CLI), reason="oracle/_ref/pwn_aligner_ref not built")
def test_same_command_line_same_odometry_as_the_reference_scene_driver(tmp_path, monkeypatch):
    """`pwn_aligner config list odometry` (the reference's scene-based odometry driver: local map, Merger, chunkStep) and
    this repository's driver with the same three arguments and `localmap 1` in the configuration, behind the test double
    of the C-ABI: byte-identical odometry files, identical per-frame .pwn payloads."""
    import subprocess
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from conftest import CONF_1_4
    from test_host_cpp import BIN, write_conf, write_pgm16
    mock = build_mock_backend(tmp_path)
    monkeypatch.setenv("LD_LIBRARY_PATH", str(mock))
    gt, raws = map_sequence(6)
    start = dict(tx=0.4, ty=-0.1, tz=0.25, qx=0.05, qy=-0.1, qz=0.02, qw=0.9935290634701167)
    for k, extra in enumerate((dict(), dict(start, chunkStep=2))):
        texts, clouds = {}, {}
        for who, exe in (("reference", REF_MAP_CLI), ("ours", BIN)):
            d = tmp_path / ("%s%d" % (who, k))
            d.mkdir()
            lst = str(d / "frames.txt")
            with open(lst, "w") as f:
                for i, r in enumerate(raws):
                    p = str(d / ("depth%d.pgm" % i))
                    write_pgm16(p, r)
                    f.write("%d.5 %s\n" % (100 + i, p))
            cfg = str(d / "aligner.conf")
            write_conf(cfg, CONF_1_4, 4, [0, 0, 0, 0, 0, 0], extra=dict(extra, localmap=1))
            odo = str(d / "odometry.txt")
            if not os.access(exe, os.X_OK):
                os.chmod(exe, 0o755)
            subprocess.run([exe, cfg, lst, odo], check=True, capture_output=True, timeout=900, cwd=str(d),
                           env=dict(os.environ, OMP_NUM_THREADS="1"))
            texts[who] = open(odo).read()
            clouds[who] = [str(d / ("depth%d.pgm.pwn" % i)) for i in range(len(raws))]
        assert texts["ours"] == texts["reference"] and len(texts["ours"].splitlines()) == 6, k
        for a, b in zip(clouds["ours"], clouds["reference"]):
            for x, y in zip(pwn_payload(a), pwn_payload(b)):
                assert np.array_equal(x, y, equal_nan=True)

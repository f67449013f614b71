"""ctypes wrapper around oracle/pwn_oracle.c (CPU restatement of pwn_core).

TEST INFRASTRUCTURE ONLY -- see oracle/pwn_oracle.h.  May be imported from tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs, nowhere else.
Pinned against the reference's own sources except for Eigen's numerical kernels (oracle/_ref, DESIGN.md section 2).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBS = {}


def build(force=False):
    """(Re)build the oracle shared objects with `make` (gcc is in the image)."""
    so = os.path.join(_HERE, "build", "liboracle.so")
    so2 = os.path.join(_HERE, "build", "liboracle_fast.so")
    src = os.path.join(_HERE, "pwn_oracle.c")
    so3 = os.path.join(_HERE, "build", "libvoxel_oracle.so")
    src3 = os.path.join(_HERE, "voxel_oracle.cpp")
    stale = (not os.path.exists(so) or not os.path.exists(so2) or not os.path.exists(so3)
             or os.path.getmtime(so) < os.path.getmtime(src) or os.path.getmtime(so3) < os.path.getmtime(src3))
    if force or stale:
        subprocess.check_call(["make", "-C", _HERE, "-B" if force else "-s"], stdout=subprocess.DEVNULL)
    return so


class StatsParams(C.Structure):
    _fields_ = [("worldRadius", C.c_float), ("minImageRadius", C.c_int), ("maxImageRadius", C.c_int),
                ("minPoints", C.c_int), ("curvatureThreshold", C.c_float),
                ("omegaCurvatureThreshold", C.c_float),
                ("flatOmegaP", C.c_float * 3), ("nonFlatOmegaP", C.c_float * 3),
                ("flatOmegaN", C.c_float * 3), ("nonFlatOmegaN", C.c_float * 3)]


class CorrParams(C.Structure):
    _fields_ = [("inlierDistanceThreshold", C.c_float), ("inlierNormalAngularThreshold", C.c_float),
                ("flatCurvatureThreshold", C.c_float), ("inlierCurvatureRatioThreshold", C.c_float)]


class Prior(C.Structure):
    _fields_ = [("kind", C.c_int), ("mean", C.c_float * 16), ("refInv", C.c_float * 16),
                ("info", C.c_float * 36)]


MAX_CAMERAS = 8


class Multi(C.Structure):
    _fields_ = [("n", C.c_int), ("width", C.c_int * MAX_CAMERAS), ("height", C.c_int * MAX_CAMERAS),
                ("minD", C.c_float * MAX_CAMERAS), ("maxD", C.c_float * MAX_CAMERAS),
                ("K", (C.c_float * 9) * MAX_CAMERAS), ("offset", (C.c_float * 16) * MAX_CAMERAS)]


def make_multi(cameras):
    """cameras: list of dicts {K, width, height, minD, maxD, offset}"""
    m = Multi()
    m.n = len(cameras)
    for i, c in enumerate(cameras):
        m.width[i], m.height[i] = int(c["width"]), int(c["height"])
        m.minD[i], m.maxD[i] = c["minD"], c["maxD"]
        m.K[i][:] = colmajor(c["K"]).tolist()
        m.offset[i][:] = colmajor(c["offset"]).tolist()
    return m


def multi_image_size(m):
    r, c = C.c_int(0), C.c_int(0)
    lib().orc_multi_image_size(C.byref(m), C.byref(r), C.byref(c))
    return r.value, c.value


def multi_project(m, T, points, rows, cols):
    pts, pp = _f(points)
    Tc, tp = _f(colmajor(T))
    idx = np.zeros((rows, cols), np.int32)
    dep = np.zeros((rows, cols), np.float32)
    lib().orc_multi_project(C.byref(m), tp, pp, pts.shape[0], rows, cols, _ip(idx), _fp(dep))
    return idx, dep


def multi_depth_to_cloud(m, depth, sp, sensor_offset=None, want_aux=False):
    depth, dp = _f(depth)
    rows, cols = depth.shape
    so, sop = _f(colmajor(np.eye(4) if sensor_offset is None else sensor_offset))
    cl = Cloud(rows * cols)
    idx = np.zeros((rows, cols), np.int32)
    itv = np.zeros((rows, cols), np.int32)
    integ = np.zeros((rows, cols, 10), np.float32)
    n = lib().orc_multi_depth_to_cloud(C.byref(m), dp, rows, cols, C.byref(sp), sop, _fp(cl.points), _fp(cl.normals),
                                       _fp(cl.statsM), _fp(cl.eigvals), _ip(cl.statsN), _fp(cl.curvature),
                                       _fp(cl.omegaP), _fp(cl.omegaN), _ip(idx), _ip(itv), _fp(integ))
    cl = cl.truncated(n)
    if want_aux:
        return cl, idx, itv, integ
    return cl, idx


class AlignParams(C.Structure):
    _fields_ = [("outerIterations", C.c_int), ("innerIterations", C.c_int), ("K", C.c_float * 9),
                ("rows", C.c_int), ("cols", C.c_int), ("minD", C.c_float), ("maxD", C.c_float),
                ("refSensorOffset", C.c_float * 16), ("curSensorOffset", C.c_float * 16),
                ("initialGuess", C.c_float * 16), ("corr", CorrParams), ("inlierMaxChi2", C.c_float),
                ("robustKernel", C.c_int), ("numThreads", C.c_int), ("numPriors", C.c_int),
                ("priors", C.POINTER(Prior)), ("multi", C.POINTER(Multi))]


class AlignResult(C.Structure):
    _fields_ = [("T", C.c_float * 16), ("H", C.c_float * 36), ("b", C.c_float * 6), ("error", C.c_float),
                ("inliers", C.c_int), ("numCorrespondences", C.c_int), ("omega", C.c_float * 36),
                ("mean", C.c_float * 6), ("translationalRatio", C.c_float), ("rotationalRatio", C.c_float)]


TRACE_STRIDE = 61


def lib(fast=False):
    key = "fast" if fast else "verify"
    if key not in _LIBS:
        build()
        name = "liboracle_fast.so" if fast else "liboracle.so"
        _LIBS[key] = C.CDLL(os.path.join(_HERE, "build", name))
    return _LIBS[key]


def _f(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a, a.ctypes.data_as(C.POINTER(C.c_float))


def _i(a):
    a = np.ascontiguousarray(a, dtype=np.int32)
    return a, a.ctypes.data_as(C.POINTER(C.c_int))


def _fp(a):
    assert a.dtype == np.float32 and a.flags.c_contiguous
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _ip(a):
    assert a.dtype == np.int32 and a.flags.c_contiguous
    return a.ctypes.data_as(C.POINTER(C.c_int))


def colmajor(M):
    """numpy (r,c) matrix -> flat column-major float32 (the ABI's matrix convention)."""
    return np.ascontiguousarray(np.asarray(M, dtype=np.float32).T).reshape(-1)


def from_colmajor(v, n):
    return np.asarray(v, dtype=np.float32).reshape(n, n).T.copy()


def default_stats_params(**kw):
    """ctor defaults: statscalculatorintegralimage.cpp:6-12, informationmatrixcalculator.h:107-109,142-144"""
    p = StatsParams()
    p.worldRadius = 0.1
    p.minImageRadius = 10
    p.maxImageRadius = 30
    p.minPoints = 50
    p.curvatureThreshold = 0.02
    p.omegaCurvatureThreshold = 0.02
    p.flatOmegaP[:] = [1000.0, 1.0, 1.0]
    p.nonFlatOmegaP[:] = [1.0, 1.0, 1.0]
    p.flatOmegaN[:] = [100.0, 100.0, 100.0]
    p.nonFlatOmegaN[:] = [1.0, 1.0, 1.0]
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def default_corr_params(**kw):
    """ctor defaults: correspondencefinder.cpp:9-18"""
    p = CorrParams()
    p.inlierDistanceThreshold = 0.5
    p.inlierNormalAngularThreshold = float(np.cos(np.pi / 6))
    p.flatCurvatureThreshold = 0.02
    p.inlierCurvatureRatioThreshold = 1.3
    for k, v in kw.items():
        setattr(p, k, v)
    return p


class Cloud:
    """Host cloud in the oracle's layout (full 4x4 stats / information matrices)."""

    def __init__(self, n):
        self.n = n
        self.points = np.zeros((n, 4), np.float32)
        self.normals = np.zeros((n, 4), np.float32)
        self.statsM = np.zeros((n, 16), np.float32)
        self.eigvals = np.zeros((n, 3), np.float32)
        self.statsN = np.zeros(n, np.int32)
        self.curvature = np.zeros(n, np.float32)
        self.omegaP = np.zeros((n, 16), np.float32)
        self.omegaN = np.zeros((n, 16), np.float32)

    def truncated(self, n):
        c = Cloud(0)
        c.n = n
        for k in ("points", "normals", "statsM", "eigvals", "statsN", "curvature", "omegaP", "omegaN"):
            setattr(c, k, np.ascontiguousarray(getattr(self, k)[:n]))
        return c

    def omegaP6(self):
        return sym6(self.omegaP)

    def omegaN6(self):
        return sym6(self.omegaN)


def sym6(om16):
    """(n,16) column-major 4x4 -> (n,6) upper triangle xx,xy,xz,yy,yz,zz (row<=col entries)."""
    o = om16.reshape(-1, 4, 4)  # o[i, c, r]
    return np.ascontiguousarray(np.stack([o[:, 0, 0], o[:, 1, 0], o[:, 2, 0], o[:, 1, 1], o[:, 2, 1], o[:, 2, 2]], axis=1))


def depth_u16_to_f32(raw, scale=0.001, fast=False):
    raw = np.ascontiguousarray(raw, dtype=np.uint16)
    out = np.empty(raw.shape, np.float32)
    lib(fast).orc_depth_u16_to_f32(raw.ctypes.data_as(C.POINTER(C.c_uint16)), raw.size, C.c_float(scale), _fp(out))
    return out


def depth_scale(depth, step, max_depth_cov=0.01, fast=False):
    depth, dp = _f(depth)
    rows, cols = depth.shape
    out = np.zeros((rows // step, cols // step), np.float32)
    lib(fast).orc_depth_scale(dp, rows, cols, step, C.c_float(max_depth_cov), _fp(out))
    return out


def v2t(v):
    v, vp = _f(v)
    T = np.zeros(16, np.float32)
    lib().orc_v2t(vp, _fp(T))
    return from_colmajor(T, 4)


def t2v(T):
    Tc, tp = _f(colmajor(T))
    v = np.zeros(6, np.float32)
    lib().orc_t2v(tp, _fp(v))
    return v


def update_matrices(K, T):
    Kc, kp = _f(colmajor(K))
    Tc, tp = _f(colmajor(T))
    KRt = np.zeros(16, np.float32)
    iKRt = np.zeros(16, np.float32)
    lib().orc_update_matrices(kp, tp, _fp(KRt), _fp(iKRt))
    return from_colmajor(KRt, 4), from_colmajor(iKRt, 4)


def unproject(depth, K, T, minD, maxD, fast=False):
    depth, dp = _f(depth)
    rows, cols = depth.shape
    _, iKRt = update_matrices(K, T)
    ik, ikp = _f(colmajor(iKRt))
    pts = np.zeros((rows * cols, 4), np.float32)
    idx = np.zeros((rows, cols), np.int32)
    n = lib(fast).orc_unproject(dp, rows, cols, ikp, C.c_float(minD), C.c_float(maxD), _fp(pts), _ip(idx))
    return np.ascontiguousarray(pts[:n]), idx


def project_intervals(depth, K, minD, maxD, world_radius, fast=False):
    depth, dp = _f(depth)
    rows, cols = depth.shape
    Kc, kp = _f(colmajor(K))
    out = np.zeros((rows, cols), np.int32)
    lib(fast).orc_project_intervals(dp, rows, cols, kp, C.c_float(minD), C.c_float(maxD), C.c_float(world_radius), _ip(out))
    return out


def project(points, rows, cols, K, T, minD, maxD, fast=False):
    """PinholePointProjector::project with projector transform T (sensor pose)."""
    KRt, _ = update_matrices(K, T)
    return project_KRt(points, rows, cols, KRt, minD, maxD, fast)


def project_KRt(points, rows, cols, KRt, minD, maxD, fast=False):
    pts, pp = _f(points)
    kr, krp = _f(colmajor(KRt))
    idx = np.zeros((rows, cols), np.int32)
    dep = np.zeros((rows, cols), np.float32)
    lib(fast).orc_project(pp, pts.shape[0], rows, cols, krp, C.c_float(minD), C.c_float(maxD), _ip(idx), _fp(dep))
    return idx, dep


def integral_image(index, points, fast=False):
    index, ip = _i(index)
    pts, pp = _f(points)
    rows, cols = index.shape
    out = np.zeros((rows, cols, 10), np.float32)
    lib(fast).orc_integral_image(ip, pp, rows, cols, _fp(out))
    return out


def eigen3(Cm):
    c, cp = _f(colmajor(Cm))
    ev = np.zeros(3, np.float32)
    U = np.zeros(9, np.float32)
    lib().orc_eigen3(cp, _fp(ev), _fp(U))
    return ev, from_colmajor(U, 3)


def depth_to_cloud(depth, K, minD, maxD, sp, sensor_offset=None, fast=False, want_aux=False):
    """DepthImageConverterIntegralImage::compute -> (Cloud, index image[, interval, integral])."""
    depth, dp = _f(depth)
    rows, cols = depth.shape
    Kc, kp = _f(colmajor(K))
    so, sop = _f(colmajor(np.eye(4) if sensor_offset is None else sensor_offset))
    cl = Cloud(rows * cols)
    idx = np.zeros((rows, cols), np.int32)
    itv = np.zeros((rows, cols), np.int32)
    integ = np.zeros((rows, cols, 10), np.float32)
    n = lib(fast).orc_depth_to_cloud(dp, rows, cols, kp, C.c_float(minD), C.c_float(maxD), C.byref(sp), sop,
                                     _fp(cl.points), _fp(cl.normals), _fp(cl.statsM), _fp(cl.eigvals),
                                     _ip(cl.statsN), _fp(cl.curvature), _fp(cl.omegaP), _fp(cl.omegaN),
                                     _ip(idx), _ip(itv), _fp(integ))
    cl = cl.truncated(n)
    if want_aux:
        return cl, idx, itv, integ
    return cl, idx


def correspond(ref_index, cur_index, ref, cur, T, cp, num_threads=8, fast=False):
    """CorrespondenceFinder::compute(ref, cur, T) -> (corr (n,2), corr image of ref indices)."""
    ri, rip = _i(ref_index)
    ci, cip = _i(cur_index)
    rows, cols = ri.shape
    Tc, tp = _f(colmajor(T))
    corr = np.full((rows * cols, 2), -1, np.int32)
    cimg = np.full((rows, cols), -1, np.int32)
    n = lib(fast).orc_correspond(rip, cip, rows, cols, _fp(ref.points), _fp(ref.normals), _fp(ref.curvature),
                                 _fp(cur.points), _fp(cur.normals), _fp(cur.curvature), tp, C.byref(cp),
                                 num_threads, _ip(corr), _ip(cimg))
    return np.ascontiguousarray(corr[:n]), cimg


def linearize(corr, ref, cur, T, max_chi2=9e3, robust=True, num_threads=8, fast=False):
    corr, cp = _i(corr)
    Tc, tp = _f(colmajor(T))
    H = np.zeros(36, np.float32)
    b = np.zeros(6, np.float32)
    err = C.c_float(0)
    inl = C.c_int(0)
    lib(fast).orc_linearize(cp, corr.shape[0], _fp(ref.points), _fp(ref.normals), _fp(cur.points), _fp(cur.normals),
                            _fp(cur.omegaP), _fp(cur.omegaN), tp, C.c_float(max_chi2), int(robust), num_threads,
                            _fp(H), _fp(b), C.byref(err), C.byref(inl))
    return from_colmajor(H, 6), b, err.value, inl.value


def linearize_f64(corr, ref, cur, T, max_chi2=9e3, robust=True):
    corr, cp = _i(corr)
    Tc, tp = _f(colmajor(T))
    H = np.zeros(36, np.float64)
    b = np.zeros(6, np.float64)
    err = C.c_double(0)
    inl = C.c_int(0)
    dptr = C.POINTER(C.c_double)
    lib().orc_linearize_f64(cp, corr.shape[0], _fp(ref.points), _fp(ref.normals), _fp(cur.points), _fp(cur.normals),
                            _fp(cur.omegaP), _fp(cur.omegaN), tp, C.c_float(max_chi2), int(robust),
                            H.ctypes.data_as(dptr), b.ctypes.data_as(dptr), C.byref(err), C.byref(inl))
    return H.reshape(6, 6).T.copy(), b, err.value, inl.value


def ldlt_solve6(H, b):
    Hc, hp = _f(colmajor(H))
    bb, bp = _f(b)
    x = np.zeros(6, np.float32)
    lib().orc_ldlt_solve6(hp, bp, _fp(x))
    return x


def compute_statistics(H, T):
    """_computeStatistics' dense tail (orc_compute_statistics) on the linearisation H (6, 6) at the pose T (4, 4) ->
    (mean (6,), Omega (6, 6), translational ratio, rotational ratio)"""
    Hc, hp = _f(colmajor(H))
    Tc, tp = _f(colmajor(T))
    mean = np.zeros(6, np.float32)
    om = np.zeros(36, np.float32)
    tr, rr = C.c_float(0), C.c_float(0)
    lib().orc_compute_statistics(hp, tp, _fp(mean), _fp(om), C.byref(tr), C.byref(rr))
    return mean, from_colmajor(om, 6), np.float32(tr.value), np.float32(rr.value)


def gn_step(H, b, T, priors=()):
    """one outer iteration of align() with inner = 1 after its linearisation (orc_gn_step): H (6, 6), b (6,) at T (4, 4),
    priors a sequence of Prior (make_prior) -> the next T (4, 4)"""
    Hc, hp = _f(colmajor(H))
    bb, bp = _f(b)
    Tc, tp = _f(colmajor(T))
    out = np.zeros(16, np.float32)
    parr = (Prior * len(priors))(*priors) if len(priors) else None
    lib().orc_gn_step(hp, bp, tp, parr, len(priors), _fp(out))
    return from_colmajor(out, 4)


def make_prior(kind, mean, info, reference=None):
    p = Prior()
    p.kind = kind
    p.mean[:] = colmajor(mean).tolist()
    ri = np.eye(4, dtype=np.float32)
    if reference is not None:
        ref = np.asarray(reference, np.float32)
        ri = np.eye(4, dtype=np.float32)
        ri[:3, :3] = ref[:3, :3].T
        ri[:3, 3] = -(ref[:3, :3].T @ ref[:3, 3])
    p.refInv[:] = colmajor(ri).tolist()
    p.info[:] = colmajor(info).tolist()
    return p


def make_align_params(K, rows, cols, minD, maxD, cp, outer=10, inner=1, guess=None, ref_offset=None,
                      cur_offset=None, max_chi2=9e3, robust=True, num_threads=8, priors=(), multi=None):
    p = AlignParams()
    p.outerIterations = outer
    p.innerIterations = inner
    p.K[:] = colmajor(K).tolist()
    p.rows, p.cols = rows, cols
    p.minD, p.maxD = minD, maxD
    eye = np.eye(4, dtype=np.float32)
    p.refSensorOffset[:] = colmajor(eye if ref_offset is None else ref_offset).tolist()
    p.curSensorOffset[:] = colmajor(eye if cur_offset is None else cur_offset).tolist()
    p.initialGuess[:] = colmajor(eye if guess is None else guess).tolist()
    p.corr = cp
    p.inlierMaxChi2 = max_chi2
    p.robustKernel = int(robust)
    p.numThreads = num_threads
    p.numPriors = len(priors)
    if priors:
        arr = (Prior * len(priors))(*priors)
        p._keep = arr
        p.priors = C.cast(arr, C.POINTER(Prior))
    if multi is not None:
        p._keep_multi = multi
        p.multi = C.pointer(multi)
    return p


class AlignOutput:
    pass


def align(ref, cur, ap, fast=False, want_trace=True, accumulate_f64=False):
    """Aligner::align() on two oracle clouds.  accumulate_f64: sum the Linearizer terms exactly
    (float64) instead of the reference's float32 partial sums -- a yardstick, not the reference."""
    lib(fast).orc_set_accumulate_f64(int(accumulate_f64))
    rows, cols = ap.rows, ap.cols
    res = AlignResult()
    out = AlignOutput()
    out.refIndex = np.zeros((rows, cols), np.int32)
    out.refDepth = np.zeros((rows, cols), np.float32)
    out.curIndex = np.zeros((rows, cols), np.int32)
    out.curDepth = np.zeros((rows, cols), np.float32)
    corr = np.full((rows * cols, 2), -1, np.int32)
    trace = np.zeros((max(ap.outerIterations, 1), TRACE_STRIDE), np.float32)
    lib(fast).orc_align(ref.n, _fp(ref.points), _fp(ref.normals), _fp(ref.curvature),
                        cur.n, _fp(cur.points), _fp(cur.normals), _fp(cur.curvature),
                        _fp(cur.omegaP), _fp(cur.omegaN), C.byref(ap), C.byref(res),
                        _ip(out.refIndex), _fp(out.refDepth), _ip(out.curIndex), _fp(out.curDepth), _ip(corr),
                        _fp(trace) if want_trace else None)
    out.T = from_colmajor(np.array(res.T[:], np.float32), 4)
    out.H = from_colmajor(np.array(res.H[:], np.float32), 6)
    out.b = np.array(res.b[:], np.float32)
    out.error = res.error
    out.inliers = res.inliers
    out.numCorrespondences = res.numCorrespondences
    out.corr = np.ascontiguousarray(corr[:res.numCorrespondences])
    out.omega = from_colmajor(np.array(res.omega[:], np.float32), 6)
    out.mean = np.array(res.mean[:], np.float32)
    out.translationalRatio = res.translationalRatio
    out.rotationalRatio = res.rotationalRatio
    out.trace_T = [from_colmajor(trace[i, :16], 4) for i in range(ap.outerIterations)]
    out.trace_H = [from_colmajor(trace[i, 16:52], 6) for i in range(ap.outerIterations)]
    out.trace_b = [trace[i, 52:58].copy() for i in range(ap.outerIterations)]
    out.trace_err = trace[:, 58].copy()
    out.trace_inliers = trace[:, 59].astype(np.int64)
    out.trace_ncorr = trace[:, 60].astype(np.int64)
    return out


def image_stats(cur_depth, ref_depth, thr=50.0):
    c, cp = _f(cur_depth)
    r, rp = _f(ref_depth)
    nz, inl, outl = C.c_int(0), C.c_int(0), C.c_int(0)
    rd = C.c_float(0)
    lib().orc_image_stats(cp, rp, c.size, C.c_float(thr), C.byref(nz), C.byref(inl), C.byref(outl), C.byref(rd))
    return nz.value, inl.value, outl.value, rd.value


# ---- local-map maintenance: Gaussian3f sensor model, Merger, VoxelCalculator ----
GAUSS_FLOATS = 24
GAUSS_MOMENTS, GAUSS_INFO = 1, 2


def unproject_gaussians(depth, K, minD, maxD, baseline=0.075, alpha=0.1, sensor_offset=None):
    """PinholePointProjector::unProject with gaussians (projector transform = identity, as in
    DepthImageConverterIntegralImage::compute) followed by Gaussian3fVector::transformInPlace(sensor_offset).
    Returns (gauss (n,24), flags (n,), points (n,4) before the sensor offset, index image)."""
    depth, dp = _f(depth)
    rows, cols = depth.shape
    Kc, kp = _f(colmajor(K))
    _, iKRt = update_matrices(K, np.eye(4, dtype=np.float32))
    ik, ikp = _f(colmajor(iKRt))
    pts = np.zeros((rows * cols, 4), np.float32)
    idx = np.zeros((rows, cols), np.int32)
    g = np.zeros((rows * cols, GAUSS_FLOATS), np.float32)
    fl = np.zeros(rows * cols, np.int32)
    n = lib().orc_unproject_gaussians(dp, rows, cols, kp, ikp, C.c_float(minD), C.c_float(maxD), C.c_float(baseline),
                                      C.c_float(alpha), _fp(pts), _ip(idx), _fp(g), _ip(fl))
    g, fl, pts = np.ascontiguousarray(g[:n]), np.ascontiguousarray(fl[:n]), np.ascontiguousarray(pts[:n])
    if sensor_offset is not None:
        so, sop = _f(colmajor(sensor_offset))
        lib().orc_gaussians_transform(sop, n, _fp(g), _ip(fl))
    return g, fl, pts, idx


def gaussians_transform(T, gauss, flags):
    g = np.ascontiguousarray(gauss, np.float32).copy()
    fl = np.ascontiguousarray(flags, np.int32).copy()
    Tc, tp = _f(colmajor(T))
    lib().orc_gaussians_transform(tp, g.shape[0], _fp(g), _ip(fl))
    return g, fl


def merge(cloud, gauss, flags, rows, cols, K, T, minD, maxD, distance_threshold=0.1,
          normal_threshold=float(np.cos(np.float32(10 * np.pi / 180.0))), max_point_depth=10.0):
    """Merger::merge on copies.  Returns (Cloud, gauss, flags, collapsed indices of the input points)."""
    n = cloud.n
    out = cloud.truncated(n)
    for k in ("points", "normals", "statsM", "omegaP", "omegaN"):
        setattr(out, k, np.ascontiguousarray(getattr(out, k)).copy())
    g = np.ascontiguousarray(gauss, np.float32).copy()
    fl = np.ascontiguousarray(flags, np.int32).copy()
    collapsed = np.zeros(max(n, 1), np.int32)
    Kc, kp = _f(colmajor(K))
    Tc, tp = _f(colmajor(T))
    k = lib().orc_merge(n, _fp(out.points), _fp(out.normals), _fp(out.statsM), _fp(out.omegaP), _fp(out.omegaN),
                        _fp(g), _ip(fl), rows, cols, kp, tp, C.c_float(minD), C.c_float(maxD),
                        C.c_float(distance_threshold), C.c_float(normal_threshold), C.c_float(max_point_depth),
                        _ip(collapsed))
    keep = (collapsed[:n] < 0) | (collapsed[:n] == np.arange(n))
    res = out.truncated(k)
    # the per-point arrays orc_merge does not carry are compacted with the same keep mask
    res.eigvals = np.ascontiguousarray(cloud.eigvals[keep])
    res.statsN = np.ascontiguousarray(cloud.statsN[keep])
    res.curvature = np.ascontiguousarray(cloud.curvature[keep])
    return res, np.ascontiguousarray(g[:k]), np.ascontiguousarray(fl[:k]), collapsed[:n].copy()


def _voxel_lib():
    if "voxel" not in _LIBS:
        build()
        so = os.path.join(_HERE, "build", "libvoxel_oracle.so")
        if not os.path.exists(so):
            subprocess.check_call(["make", "-C", _HERE, "-s"], stdout=subprocess.DEVNULL)
        _LIBS["voxel"] = C.CDLL(so)
        _LIBS["voxel"].orc_voxelize.restype = C.c_int
    return _LIBS["voxel"]


def voxelize(points, resolution=0.01, strict=True):
    """VoxelCalculator::compute -> indices of the representative points in output order.
    strict=False: the reference's comparator exactly as written (not a strict weak order);
    strict=True: lexicographic order (what the CUDA path implements)."""
    pts, pp = _f(points)
    rep = np.zeros(max(pts.shape[0], 1), np.int32)
    m = _voxel_lib().orc_voxelize(pp, pts.shape[0], C.c_float(resolution), 1 if strict else 0, _ip(rep))
    return rep[:m].copy()


def stats_stage(integral, index, interval, points, sp):
    """StatsCalculatorIntegralImage::compute given the integral image (orc_stats): normals, statsM, eigvals, statsN, curvature"""
    rows, cols = index.shape
    pts, pp = _f(points)
    n = pts.shape[0]
    integ, ip_ = _f(integral)
    idx = np.ascontiguousarray(index, np.int32)
    itv = np.ascontiguousarray(interval, np.int32)
    normals = np.zeros((n, 4), np.float32)
    statsM = np.zeros((n, 16), np.float32)
    eig = np.zeros((n, 3), np.float32)
    cnt = np.zeros(n, np.int32)
    curv = np.zeros(n, np.float32)
    f = lib().orc_stats
    f.restype = None
    f(ip_, _ip(idx), _ip(itv), pp, rows, cols, n, C.byref(sp), _fp(normals), _fp(statsM), _fp(eig), _ip(cnt), _fp(curv))
    return normals, statsM, eig, cnt, curv


def information_stage(normals, statsM, eigvals, curvature, sp):
    """Point / NormalInformationMatrixCalculator::compute (orc_information): full 4x4 per point"""
    n = normals.shape[0]
    oP = np.zeros((n, 16), np.float32)
    oN = np.zeros((n, 16), np.float32)
    f = lib().orc_information
    f.restype = None
    f(_fp(np.ascontiguousarray(normals, np.float32)), _fp(np.ascontiguousarray(statsM, np.float32)),
      _fp(np.ascontiguousarray(eigvals, np.float32)), _fp(np.ascontiguousarray(curvature, np.float32)), n, C.byref(sp),
      _fp(oP), _fp(oN))
    return oP, oN


def set_eigen_variant(v, fast=False):
    """0: Eigen 3.2.x computeDirect (default; what the CUDA path follows), 1: the Eigen >= 3.3 implementation,
    2: Eigen 3.2.x with atan2 / cos / sin evaluated in float64 and rounded, as the CUDA path evaluates them.
    The variant is global state of the library: callers that change it restore 0 afterwards."""
    f = lib(fast).orc_set_eigen_variant
    f.restype = None
    f(int(v))


def eigen3_devtrig(Cm):
    """Eigen 3.2.x computeDirect with the CUDA path's float64 trig (eigen variant 2)"""
    Cm, cp = _f(colmajor(Cm))
    ev = np.zeros(3, np.float32)
    U = np.zeros(9, np.float32)
    f = lib().orc_eigen3_devtrig
    f.restype = None
    f(cp, _fp(ev), _fp(U))
    return ev, from_colmajor(U, 3)


def eigen3_v33(Cm):
    Cm, cp = _f(colmajor(Cm))
    ev = np.zeros(3, np.float32)
    U = np.zeros(9, np.float32)
    f = lib().orc_eigen3_v33
    f.restype = None
    f(cp, _fp(ev), _fp(U))
    return ev, from_colmajor(U, 3)


def set_threads(n, fast=False):
    """omp_set_num_threads(n) inside the oracle library (OMP_NUM_THREADS is only read when libgomp initialises);
    returns the OpenMP team size actually in force"""
    f = lib(fast).orc_set_threads
    f.restype = C.c_int
    return int(f(int(n)))


# restype declarations that are not int
def _declare():
    for fast in (False, True):
        l = lib(fast)
        for name in ("orc_unproject", "orc_depth_to_cloud", "orc_correspond", "orc_multi_unproject",
                     "orc_multi_depth_to_cloud", "orc_unproject_gaussians", "orc_merge"):
            getattr(l, name).restype = C.c_int
        for name in ("orc_depth_u16_to_f32", "orc_depth_scale", "orc_v2t", "orc_t2v", "orc_update_matrices",
                     "orc_project_intervals", "orc_project", "orc_integral_image", "orc_eigen3", "orc_linearize",
                     "orc_linearize_f64", "orc_ldlt_solve6", "orc_align", "orc_image_stats", "orc_multi_image_size",
                     "orc_multi_intervals", "orc_multi_project", "orc_set_accumulate_f64", "orc_cloud_transform", "orc_gaussians_transform",
                     "orc_compute_statistics", "orc_gn_step"):
            getattr(l, name).restype = None


_declare()

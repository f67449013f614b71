"""Frame preparation statistics (k_stats, k_stats_stage, k_information_stage) bit for bit against the oracle.

The oracle's default eigen-solver (variant 0) calls libm atan2f / cosf / sinf; the CUDA path evaluates atan2 / cos / sin in
float64 and rounds (DESIGN.md section 5), which is why test_gpu_parity holds normals to a statistical bar.  Oracle variant 2
is the same closed form with the CUDA path's trig, so every other operation -- region sums, covariance, the eigen-solver's
branches, curvature, the gates, orientation, information matrices, sensor offset -- must agree with it in every bit of every
point.  The one admitted exception is a pixel where a float64 trig value lies within a few double ulps of a float32 rounding
midpoint (the two float64 implementations may then round to different floats); such pixels are printed.

Covered here, beside the realistic scenes: hand-built windows that take every reachable branch of the closed-form solver
(a float32 restatement of it below reports the branch), every gate exactly on its threshold and one ulp to either side,
windows clipped by the image borders, the three column-pass kernels at their switch points, and the size limits of frame
preparation (NICP_MAX_PREP_COLS, NICP_MAX_PREP_PIXELS).
"""
import math

import numpy as np
import pytest

from conftest import get_scene, CONF_1_1, CONF_1_4
from oracle import pwn_oracle as O

f32 = np.float32
EPS = f32(np.finfo(np.float32).eps)


# ---- float32 restatement of eigen3 (frame_prep.cu) / orc_eigen3_devtrig, reporting the branches it takes ---------------
def _cross(a, b):
    return [f32(a[1] * b[2]) - f32(a[2] * b[1]), f32(a[2] * b[0]) - f32(a[0] * b[2]), f32(a[0] * b[1]) - f32(a[1] * b[0])]


def _sq(a):
    return f32(f32(a[0] * a[0]) + f32(a[1] * a[1])) + f32(a[2] * a[2])


def _unit(v, n):
    sn = np.sqrt(n)
    return [f32(v[0] / sn), f32(v[1] / sn), f32(v[2] / sn)]


def _unit_orthogonal(s, branches):
    prec = f32(1e-5)
    if not (abs(s[0]) <= f32(abs(s[2]) * prec)) or not (abs(s[1]) <= f32(abs(s[2]) * prec)):
        branches.add("unit_orthogonal_xy")
        inv = f32(1) / np.sqrt(f32(f32(s[0] * s[0]) + f32(s[1] * s[1])))
        return [f32(-s[1] * inv), f32(s[0] * inv), f32(0)]
    branches.add("unit_orthogonal_yz")
    inv = f32(1) / np.sqrt(f32(f32(s[1] * s[1]) + f32(s[2] * s[2])))
    return [f32(0), f32(-s[2] * inv), f32(s[1] * inv)]


def eigen3(c6):
    """c6 = (c00, c10, c20, c11, c21, c22) float32 -> (eigenvalues, U (columns = eigenvectors), branches, float64 trig values
    (theta before the division by 3, cos, sin)), every operation rounded to float32 in the CUDA path's order"""
    with np.errstate(all="ignore"):
        c00, c10, c20, c11, c21, c22 = [f32(v) for v in c6]
        br = set()
        scale = max(max(max(abs(c00), abs(c10)), max(abs(c20), abs(c11))), max(abs(c21), abs(c22)))
        if scale == 0:
            br.add("zero_scale")
        m00, m10, m20, m11, m21, m22 = [f32(v / scale) for v in (c00, c10, c20, c11, c21, c22)]
        inv3, sqrt3 = f32(1) / f32(3), np.sqrt(f32(3))
        c0 = f32(f32(f32(f32(f32(m00 * m11) * m22) + f32(f32(f32(f32(2) * m10) * m20) * m21)) - f32(f32(m00 * m21) * m21))
                 - f32(f32(m11 * m20) * m20)) - f32(f32(m22 * m10) * m10)
        c1 = f32(f32(f32(f32(f32(m00 * m11) - f32(m10 * m10)) + f32(m00 * m22)) - f32(m20 * m20)) + f32(m11 * m22)) - f32(m21 * m21)
        c2 = f32(m00 + m11) + m22
        c2o3 = f32(c2 * inv3)
        ao3 = f32(f32(c1 - f32(c2 * c2o3)) * inv3)
        if ao3 > 0:
            ao3 = f32(0)
        hb = f32(f32(0.5) * f32(c0 + f32(c2o3 * f32(f32(f32(f32(2) * c2o3) * c2o3) - c1))))
        q = f32(f32(hb * hb) + f32(f32(ao3 * ao3) * ao3))
        if q > 0:
            q = f32(0)
        rho = np.sqrt(f32(-ao3))
        th64 = math.atan2(float(np.sqrt(f32(-q))), float(hb))
        theta = f32(f32(th64) * inv3)
        co64, si64 = math.cos(float(theta)), math.sin(float(theta))
        ct, st = f32(co64), f32(si64)
        r0 = f32(c2o3 + f32(f32(f32(2) * rho) * ct))
        r1 = f32(c2o3 - f32(rho * f32(ct + f32(sqrt3 * st))))
        r2 = f32(c2o3 - f32(rho * f32(ct - f32(sqrt3 * st))))
        if r0 >= r1:
            r0, r1 = r1, r0
        if r1 >= r2:
            r1, r2 = r2, r1
            if r0 >= r1:
                r0, r1 = r1, r0
        ev = np.array([r0 * scale, r1 * scale, r2 * scale], np.float32)
        U = np.eye(3, dtype=np.float32)
        trig = (th64, co64, si64)
        safe = f32(EPS * EPS)
        if f32(r2 - r0) <= EPS:
            br.add("identity")
            return ev, U, br, trig
        d0, d1 = f32(r2 - r1), f32(r1 - r0)
        k = 2 if d0 > d1 else 0
        evk = r2 if d0 > d1 else r0
        d0 = d1 if d0 > d1 else d0
        row0, row1, row2 = [f32(m00 - evk), m10, m20], [m10, f32(m11 - evk), m21], [m20, m21, f32(m22 - evk)]
        for tag, a, b in (("uk_row01", row0, row1), ("uk_row02", row0, row2), ("uk_row12", row1, row2)):
            cr = _cross(a, b)
            n = _sq(cr)
            if n > safe:
                break
        else:
            br.add("numerical_issue")
            return ev, U, br, trig
        br.add(tag)
        uk = _unit(cr, n)
        if d0 <= EPS:
            br.add("d0_small")
            u1 = _unit_orthogonal(uk, br)
        else:
            r0v, r1v, r2v = [f32(m00 - r1), m10, m20], [m10, f32(m11 - r1), m21], [m20, m21, f32(m22 - r1)]
            nr0 = np.sqrt(_sq(r0v))
            r0n = [f32(r0v[0] / nr0), f32(r0v[1] / nr0), f32(r0v[2] / nr0)]
            for tag, v in (("u1_r0", r0n), ("u1_r1", r1v), ("u1_r2", r2v)):
                cr = _cross(uk, v)
                n = _sq(cr)
                if n > safe:
                    br.add(tag)
                    u1 = _unit(cr, n)
                    break
            else:
                br.add("u1_unit_orthogonal")
                u1 = _unit_orthogonal(uk, br)
            t2 = _cross(uk, _cross(u1, uk))
            u1 = _unit(t2, _sq(t2))
        t = _cross(uk, u1)
        ul = _unit(t, _sq(t))
        U[:, k], U[:, 1], U[:, 0 if k == 2 else 2] = uk, u1, ul
        return ev, U, br, trig


# Every branch of the solver a window reaches.  Not listed: the unit_orthogonal fallback after the three u1 cross products
# (it needs r1 isolated by more than FLT_EPSILON while all three rows of M - r1 I lie within FLT_EPSILON of uk's direction),
# and a scaled spread r2 - r0 or gap d0 just above FLT_EPSILON: near a double root the closed form resolves eigenvalue
# differences only to ~sqrt(FLT_EPSILON) of the scale, so computed spreads are 0, eps/2, eps or >= ~2e-4 (the cases
# "spread_zero", "d0_half_eps" and "d0_tiny" below sit on the <= side of both comparisons, the tetrahedra on the other).
BRANCHES = {"zero_scale", "numerical_issue", "identity", "uk_row01", "uk_row02", "uk_row12", "d0_small", "unit_orthogonal_xy",
            "unit_orthogonal_yz", "u1_r0", "u1_r1", "u1_r2"}


def near_f32_midpoint(x, ulps=4):
    """whether float64 x lies within `ulps` double ulps of a point halfway between two float32 values (checked in long
    double): there two float64 implementations of one function may round to different float32 values"""
    if not math.isfinite(x):
        return False
    f = f32(x)
    other = np.nextafter(f, f32(np.inf) if float(f) < x else f32(-np.inf))
    mid = (np.longdouble(f) + np.longdouble(other)) / 2
    return abs(np.longdouble(x) - mid) <= ulps * np.longdouble(np.spacing(abs(x)))


def canon(a):
    """float32 bit patterns with every NaN as one pattern: a NaN matches a NaN (the device's default NaN is 0x7fffffff,
    x86's 0xffc00000), every other value matches only itself, signed zeros included"""
    b = np.ascontiguousarray(a, np.float32).view(np.uint32).copy()
    b[np.isnan(np.ascontiguousarray(a, np.float32))] = 0x7FC00000
    return b


# ---- windows -----------------------------------------------------------------------------------------------------------
ROWS = COLS = 8
CENTER = (4, 4)      # window of radius 3: rows and columns 1..6 (getRegion sums (c - k - 1, c + k - 1])
WIN = [CENTER] + [(r, c) for r in range(1, 7) for c in range(1, 7) if (r, c) != CENTER]


def layout(pts, pixels=None):
    """points -> (points4, index image): point 0 at the window's centre pixel, the others over the window in raster order"""
    pixels = WIN if pixels is None else pixels
    idx = np.full((ROWS, COLS), -1, np.int32)
    P = np.zeros((len(pts), 4), np.float32)
    for i, p in enumerate(pts):
        P[i, :3] = p
        P[i, 3] = 1
        idx[pixels[i]] = i
    return P, idx


def clampi(v, lo, hi):
    return lo if v < lo else (hi if v > hi else v)


def region(I, r, c, k):
    """PointIntegralImage::getRegion(c - k, c + k, r - k, r + k) in float32 (the kernels' order)"""
    rows, cols = I.shape[:2]
    x0, x1 = clampi(c - k - 1, 0, cols - 1), clampi(c + k - 1, 0, cols - 1)
    y0, y1 = clampi(r - k - 1, 0, rows - 1), clampi(r + k - 1, 0, rows - 1)
    return ((I[y1, x1] + I[y0, x0]) - I[y1, x0]) - I[y0, x1]


def cov6(acc):
    """PointAccumulator mean / covariance of region sums, float32 in the kernels' order"""
    dd = f32(1) / acc[0]
    mu = [f32(acc[1] * dd), f32(acc[2] * dd), f32(acc[3] * dd)]
    v = lambda a, i, j: f32(f32(acc[a] * dd) - f32(mu[i] * mu[j]))
    return [v(4, 0, 0), v(5, 0, 1), v(6, 0, 2), v(7, 1, 1), v(8, 1, 2), v(9, 2, 2)]


def pixel_cov(I, interval, r, c, sp):
    k = clampi(int(interval[r, c]), sp.minImageRadius, sp.maxImageRadius)
    return cov6(region(I, r, c, k))


def tetra(a, b, g, o=(0.0, 0.0, 0.0)):
    """four points whose covariance is exactly diag(a^2, b^2, g^2) for dyadic a, b, g"""
    return [(o[0] + a, o[1] + b, o[2] + g), (o[0] + a, o[1] - b, o[2] - g), (o[0] - a, o[1] + b, o[2] - g),
            (o[0] - a, o[1] - b, o[2] + g)]


def grid(fn, n=3, h=0.25):
    return [fn(h * (a - n // 2), h * (b - n // 2)) for a in range(n) for b in range(n)]


# name -> (points, min_points); point 0 sits at the centre pixel
CASES = {
    "repeated_point": ([(0.5, -0.25, 2.0)] * 4, 1),
    "single_point": ([(0.5, -0.25, 2.0)], 1),
    "line_z": ([(0.25, -0.5, z) for z in (1.0, 1.5, 2.0, 2.5)], 1),
    "line_generic": ([(0.5 * t, 0.25 * t, 1.0 + t) for t in (0, 1, 2, 3)], 1),
    "cube_corners": ([(0.5 * a, 0.5 * b, 2 + 0.5 * c) for a in (-1, 1) for b in (-1, 1) for c in (-1, 1)], 1),
    "plane_fronto": (grid(lambda x, y: (x, y, 2.0)), 1),
    "plane_oblique": (grid(lambda x, y: (x, y, 2.0 + 0.5 * x + 0.25 * y)), 1),
    "plane_through_origin": (grid(lambda y, z: (0.0, y, 1.5 + 2 * z)), 1),
    "diag_0_q_1": (tetra(0.0, 0.5, 1.0), 1),        # covariance diag(0, 1/4, 1)
    "diag_q_1_0": (tetra(0.5, 1.0, 0.0), 1),
    "diag_1_q_0": (tetra(1.0, 0.5, 0.0), 1),
    "diag_1_s_0": (tetra(1.0, 0.25, 0.0), 1),     # covariance diag(1, 1/16, 0)
    "diag_1_h_q": (tetra(1.0, 0.75, 0.5), 1),
    "diag_h_1_q": (tetra(0.75, 1.0, 0.5), 1),
    "spread_zero": (tetra(1.0, 1.0, float(np.nextafter(f32(1), f32(0)) * np.nextafter(f32(1), f32(0)))), 1),
    "d0_half_eps": (tetra(1.0, float(np.nextafter(f32(1), f32(0))), 0.0), 1),
    "d0_tiny": (tetra(1.0, float(f32(0.9999996)), 0.0), 1),
    "curved": ([(0.0, 0.0, 2.0)] + [(0.25 * a, 0.25 * b, 2.0 + 0.5 * (0.25 * a) ** 2 + 0.125 * (0.25 * b))
                                    for a in range(-2, 3) for b in range(-2, 3) if (a, b) != (0, 0)], 1),
}


def case_inputs(name):
    """(points4, index image, interval image (3 at every point, radius 1..3), window covariance at the centre pixel)"""
    pts, _ = CASES[name]
    P, idx = layout(pts)
    itv = np.where(idx >= 0, 3, -1).astype(np.int32)
    I = O.integral_image(idx, P)
    return P, idx, itv, cov6(region(I, CENTER[0], CENTER[1], 3))


def case_params(name, **kw):
    base = dict(minImageRadius=1, maxImageRadius=3, minPoints=CASES[name][1], curvatureThreshold=0.5)
    base.update(kw)
    return base


def oracle_sp(p):
    return O.default_stats_params(**p)


def gpu_sp(p):
    from g2o_frontend_b200 import capi
    o = O.default_stats_params(**p)
    return capi.make_stats_params(o.worldRadius, o.minImageRadius, o.maxImageRadius, o.minPoints, o.curvatureThreshold,
                                  o.omegaCurvatureThreshold, tuple(o.flatOmegaP), tuple(o.flatOmegaN), tuple(o.nonFlatOmegaN))


def sym_mat(c6):
    c00, c10, c20, c11, c21, c22 = c6
    return np.array([[c00, c10, c20], [c10, c11, c21], [c20, c21, c22]], np.float32)


@pytest.fixture
def variant2():
    """oracle eigen variant 2 for the duration of a test (the variant is global state of the oracle library)"""
    O.set_eigen_variant(2)
    try:
        yield
    finally:
        O.set_eigen_variant(0)


# ---- CPU: the yardstick itself -----------------------------------------------------------------------------------------
def test_variant2_is_an_eigendecomposition():
    """orc_eigen3_devtrig against numpy.linalg.eigh in float64, with the bars test_oracle holds variant 0 to (the closed
    form loses ~sqrt(eps) when eigenvalues cluster)"""
    rng = np.random.default_rng(0)
    for i in range(400):
        Q, _ = np.linalg.qr(rng.standard_normal((3, 3)))
        lam = np.sort(rng.uniform(0.01, 1.0, 3)) * 10.0 ** rng.integers(-5, 1)
        if i % 3 == 0:
            lam[0] *= 1e-3  # planar patch
        Cm = (Q @ np.diag(lam) @ Q.T)
        Cm = ((Cm + Cm.T) / 2).astype(np.float32)
        ev, U = O.eigen3_devtrig(Cm)
        w, V = np.linalg.eigh(Cm.astype(np.float64))
        assert np.all(np.diff(ev) >= 0)
        sep = min(w[1] - w[0], w[2] - w[1]) / w[2]
        assert np.allclose(ev, w, atol=(2e-5 if sep > 0.1 else 1e-3) * w[-1])
        assert np.allclose(U.T @ U, np.eye(3), atol=1e-4)
        if (w[1] - w[0]) > 1e-2 * w[2]:
            assert abs(float(U[:, 0] @ V[:, 0])) > 1 - 1e-4


def test_restatement_matches_oracle_variant2():
    """the numpy float32 restatement equals orc_eigen3_devtrig bit for bit on every hand-built window and on random
    covariances of every scale, and the case list takes every branch of BRANCHES"""
    taken = {}
    inputs = [(name, case_inputs(name)[3]) for name in CASES]
    rng = np.random.default_rng(3)
    for i in range(400):
        A = rng.normal(size=(3, 3)) * 10.0 ** rng.uniform(-6, 3)
        if i % 4 == 0:
            A[:, 0] = 0  # rank deficient
        C = (A @ A.T).astype(np.float32)
        inputs.append(("random%d" % i, [C[0, 0], C[1, 0], C[2, 0], C[1, 1], C[2, 1], C[2, 2]]))
    for name, c6 in inputs:
        ev, U, br, _ = eigen3(c6)
        evo, Uo = O.eigen3_devtrig(sym_mat(c6))
        assert np.array_equal(canon(ev), canon(evo)), (name, ev, evo)
        assert np.array_equal(canon(U), canon(Uo)), (name, U, Uo)
        if name in CASES:
            for b in br:
                taken.setdefault(b, name)
    missing = BRANCHES - set(taken)
    assert not missing, missing
    print("branches and the first case taking them:", sorted(taken.items()))


def test_midpoint_detector():
    f = f32(1.5)
    mid = float((np.longdouble(f) + np.longdouble(np.nextafter(f, f32(2)))) / 2)
    assert near_f32_midpoint(mid) and near_f32_midpoint(np.nextafter(mid, 2.0))
    assert not near_f32_midpoint(1.5) and not near_f32_midpoint(float(f32(1.5)) + 1e-9)


# ---- GPU -----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", params=["verify", "default"])
def ctx(request):
    from g2o_frontend_b200 import capi
    c = capi.Context(0, verify=(request.param == "verify"))
    assert bool(c.L.nicp_is_verification_build()) == (request.param == "verify")
    yield c
    c.close()


def mismatched_rows(got, ref):
    g, r = canon(got).reshape(len(got), -1), canon(ref).reshape(len(ref), -1)
    assert g.shape == r.shape
    return np.nonzero((g != r).any(axis=1))[0]


def check_cloud(what, got, ref, cov_of_point):
    """every array of the GPU cloud (dict: points, normals, curvature, omega_p, omega_n, stats16, eigvals, n) bit-identical
    to the oracle's cloud; cov_of_point(i) -> the window covariance of point i (None: no window), for the double-rounding
    exception"""
    assert got["n"].shape == ref.statsN.shape, what
    assert np.array_equal(got["n"], ref.statsN), what
    pairs = (("points", got["points"], ref.points), ("normals", got["normals"][:, :3], ref.normals[:, :3]),
             ("curvature", got["curvature"], ref.curvature), ("omega_p", got["omega_p"], ref.omegaP6()),
             ("omega_n", got["omega_n"], ref.omegaN6()), ("stats16", got["stats16"], ref.statsM),
             ("eigvals", got["eigvals"], ref.eigvals))
    bad = set()
    for key, g, r in pairs:
        bad |= set(mismatched_rows(g, r).tolist())
    for i in sorted(bad):
        c6 = cov_of_point(i)
        assert c6 is not None, (what, i, "no window, yet outputs differ")
        trig = eigen3(c6)[3]
        assert any(near_f32_midpoint(t) for t in trig), (what, i, "differs without a double-rounding case", trig,
                                                         {k: (g[i], r[i]) for k, g, r in pairs})
        print("%s: point %d differs at a float64 trig value next to a float32 midpoint: %r" % (what, i, trig))
    print("%s: %d of %d points bit-identical to oracle variant 2" % (what, len(ref.points) - len(bad), len(ref.points)))


def gpu_cloud(cl):
    d = cl.download()
    s16, ev, cnt = cl.download_stats()
    d.update(stats16=s16, eigvals=ev, n=cnt)
    return d


def cov_lookup(index, interval, integral, sp):
    """point -> covariance of its window, from the oracle's aux images (integral (rows, cols, 10))"""
    pix = {}
    rr, cc = np.nonzero(index >= 0)
    for r, c in zip(rr, cc):
        pix[int(index[r, c])] = (r, c)

    def f(i):
        r, c = pix[i]
        if interval[r, c] < 0:
            return None
        return pixel_cov(integral, interval, r, c, sp)
    return f


@pytest.mark.gpu
@pytest.mark.parametrize("step,seed,dropout,offset", [(4, None, 0.0, False), (4, 0, 0.05, True), (1, None, 0.0, False),
                                                       (1, 2, 0.05, True), (4, 0, 0.05, False), (1, 1, 0.05, False)])
def test_converter_scenes_bit_identical(ctx, variant2, step, seed, dropout, offset):
    """the scenes of test_depth_to_cloud and test_stage_level_stats_and_information through the fused converter"""
    s = get_scene(step, seed, dropout, offset)
    oc, oidx, oitv, ointeg = O.depth_to_cloud(s.depthA, s.K, s.conf["minD"], s.conf["maxD"], s.sp, s.sensor_offset,
                                              want_aux=True)
    cl, idx = ctx.depth_to_cloud(s.depthA, s.projector(), s.stats_params(), s.sensor_offset, keep_stats=True)
    assert np.array_equal(idx, oidx) and cl.size() == oc.n
    check_cloud("scene %r" % ((step, seed, dropout, offset),), gpu_cloud(cl), oc, cov_lookup(oidx, oitv, ointeg, s.sp))


@pytest.mark.gpu
@pytest.mark.parametrize("step,seed,dropout", [(4, 0, 0.05), (1, 1, 0.05)])
def test_stage_scenes_bit_identical(ctx, variant2, step, seed, dropout):
    """the stage entries on the scenes of test_stage_level_stats_and_information, shuffled point order"""
    s = get_scene(step, seed, dropout)
    n = s.cloudA.n
    perm = np.random.default_rng(5).permutation(n).astype(np.int32)
    points = np.zeros_like(s.cloudA.points)
    points[perm] = s.cloudA.points
    index = np.where(s.indexA >= 0, perm[np.maximum(s.indexA, 0)], -1).astype(np.int32)
    stage_compare("stage %r" % ((step, seed, dropout),), ctx, points, index, s.intervalA, s.sp, s.stats_params())


def stage_compare(what, ctx, points, index, interval, osp, gsp):
    """nicp_stats_compute + nicp_information_compute against orc_stats + orc_information, every output bit for bit;
    returns the oracle's (normals, statsM, eigvals, n, curvature)"""
    integral = O.integral_image(index, points)
    on, oS, oe, ocnt, ocurv = O.stats_stage(integral, index, interval, points, osp)
    g = ctx.stats_compute(points, index, interval, gsp)
    assert np.array_equal(g["n"], ocnt), what
    look = cov_lookup(index, interval, integral, osp)
    bad = set()
    for key, a, b in (("normals", g["normals"], on), ("stats16", g["stats16"], oS), ("eigenvalues", g["eigenvalues"], oe),
                      ("curvature", g["curvature"], ocurv)):
        bad |= set(mismatched_rows(a, b).tolist())
    for i in sorted(bad):
        c6 = look(i)
        assert c6 is not None and any(near_f32_midpoint(t) for t in eigen3(c6)[3]), (what, i, g["normals"][i], on[i])
        print("%s: point %d differs at a float64 trig value next to a float32 midpoint" % (what, i))
    # information matrices from the oracle's statistics (stage isolated)
    oP, oN = O.information_stage(on, oS, oe, ocurv, osp)
    gp, gn = ctx.information_compute(on, oS, oe, ocurv, gsp)
    assert np.array_equal(canon(gp), canon(O.sym6(oP))), what
    assert np.array_equal(canon(gn), canon(O.sym6(oN))), what
    print("%s: %d of %d points bit-identical to oracle variant 2" % (what, len(points) - len(bad), len(points)))
    return on, oS, oe, ocnt, ocurv


@pytest.mark.gpu
def test_real_kinect_frame_bit_identical(ctx, variant2):
    import os
    from conftest import ROOT
    from g2o_frontend_b200 import capi, synth
    raw = np.load(os.path.join(ROOT, "tests", "golden", "real_depth_640x480.npz"))["raw"]
    c = CONF_1_1
    sp = O.default_stats_params(minImageRadius=c["minImageRadius"], maxImageRadius=c["maxImageRadius"],
                                minPoints=c["minPoints"], curvatureThreshold=c["curvatureThreshold"])
    oc, oidx, oitv, ointeg = O.depth_to_cloud(O.depth_u16_to_f32(raw), synth.K_KINECT, c["minD"], c["maxD"], sp, want_aux=True)
    proj = capi.make_projector(synth.K_KINECT, 480, 640, c["minD"], c["maxD"])
    gsp = capi.make_stats_params(c["worldRadius"], c["minImageRadius"], c["maxImageRadius"], c["minPoints"],
                                 c["curvatureThreshold"], c["omegaCurvatureThreshold"])
    cl, idx = ctx.raw_depth_to_cloud(raw, proj, gsp, keep_stats=True, want_index=True)
    assert np.array_equal(idx, oidx)
    check_cloud("real Kinect frame", gpu_cloud(cl), oc, cov_lookup(oidx, oitv, ointeg, sp))


@pytest.mark.gpu
def test_ragged_and_tiny_images_bit_identical(ctx, variant2):
    from g2o_frontend_b200 import capi
    s = get_scene(4)
    for rows, cols in ((37, 53), (1, 160), (120, 1), (1, 1), (2, 2)):
        d = np.ascontiguousarray(s.depthA[:rows, :cols])
        oc, oi, oitv, ointeg = O.depth_to_cloud(d, s.K, 0.5, 4.5, s.sp, want_aux=True)
        cl, idx = ctx.depth_to_cloud(d, capi.make_projector(s.K, rows, cols, 0.5, 4.5), s.stats_params(), keep_stats=True)
        assert np.array_equal(idx, oi) and cl.size() == oc.n
        check_cloud("%dx%d" % (rows, cols), gpu_cloud(cl), oc, cov_lookup(oi, oitv, ointeg, s.sp))


def rig_composite(raws, cams, step):
    """the oracle's composite depth image of one raw rig frame"""
    rows, cols = max(c["width"] for c in cams), sum(c["height"] for c in cams)
    out = np.zeros((rows, cols), np.float32)
    off = 0
    for r, c in zip(raws, cams):
        d = O.depth_u16_to_f32(r)
        if step > 1:
            d = O.depth_scale(d, step)
        out[:c["width"], off:off + c["height"]] = d.T
        off += c["height"]
    return out


def rig_compare(what, ctx, cams, frames, step, osp, gsp, so):
    from g2o_frontend_b200 import capi
    om, gm = O.make_multi(cams), capi.make_multi_projector(cams)
    clouds = ctx.multi_raw_depth_to_cloud_batch(frames, gm, gsp, step=step, sensor_offset=so, keep_stats=True)
    ctx.synchronize()
    for f, (raws, cl) in enumerate(zip(frames, clouds)):
        oc, oidx, oitv, ointeg = O.multi_depth_to_cloud(om, rig_composite(raws, cams, step), osp, so, want_aux=True)
        assert cl.size() == oc.n, (what, f)
        check_cloud("%s frame %d" % (what, f), gpu_cloud(cl), oc, cov_lookup(oidx, oitv, ointeg, osp))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["4cam", "ragged"])
def test_rigs_bit_identical(ctx, variant2, kind):
    """both test rigs through nicp_multi_raw_depth_to_cloud_batch: windows straddle the seams between the cameras' column
    blocks, and the ragged rig has zero rows past its narrower camera"""
    from g2o_frontend_b200 import capi, synth
    from test_rig_batch import make_cams, render_raw_frame, rig_poses
    cams = make_cams(kind)
    frames = [render_raw_frame(p, cams, 1, 40 + 3 * i) for i, p in enumerate(rig_poses(3, 9))]
    so = synth.make_pose((0.05, 0.0, 0.1), (1.0, 0.2, 0.0), 3.0).astype(np.float32)
    osp = O.default_stats_params(minImageRadius=3, maxImageRadius=6, minPoints=10, curvatureThreshold=0.2)
    gsp = capi.make_stats_params(0.1, 3, 6, 10, 0.2, 0.02)
    rig_compare(kind, ctx, cams, frames, 1, osp, gsp, so)


# ---- hand-built windows through the stage entry -------------------------------------------------------------------------
# Windows whose covariance is exactly diagonal with the middle eigenvalue's row of M - r1 I zero up to rounding: Eigen 3.2's
# computeDirect (which the reference builds against, and the oracle and the CUDA path restate) normalises that noise
# (r0n) or accepts an unnormalised noise row (r1v, r2v) above its eps^2 threshold, and so returns the middle and the
# smallest eigenvectors swapped.  The kernel reproduces this bit for bit; the float64 bar on the normal does not apply.
SWAPPED_BY_THE_REFERENCE = {"diag_1_s_0", "diag_h_1_q", "diag_q_1_0"}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_hand_built_windows(ctx, variant2, name):
    """bit identity to variant 2, and the eigen step against numpy.linalg.eigh (float64) of the covariance the kernel forms
    from the bit-exact region sums: eigenvalues within 8 eps scale where they are apart (the closed form's documented
    sqrt(eps) loss, 1e-3 scale, where they cluster); the normal within 8 eps scale / gap where the gap is resolved"""
    p = case_params(name)
    P, idx, itv, c6 = case_inputs(name)
    on, oS, oe, ocnt, ocurv = stage_compare(name, ctx, P, idx, itv, oracle_sp(p), gpu_sp(p))
    ev, U, br, _ = eigen3(c6)
    print(name, sorted(br))
    assert ocnt[0] == len(CASES[name][0])
    ev[0] = max(ev[0], f32(0))   # the kernel clamps the smallest eigenvalue at 0
    assert np.array_equal(canon(oe[0]), canon(ev)) and np.array_equal(canon(oS[0].reshape(4, 4)[:3, :3].T), canon(U))
    if "zero_scale" in br:
        assert np.isnan(oe[0]).all() and not on[0, :3].any()
        return
    C = sym_mat(c6).astype(np.float64)
    w, V = np.linalg.eigh(C)
    scale = np.abs(C).max()
    w[0] = max(w[0], 0.0)
    apart = np.diff(w).min() > 0.1 * scale
    assert np.abs(oe[0].astype(np.float64) - w).max() <= (8 * EPS if apart else 1e-3) * scale, (name, oe[0], w)
    gap = w[1] - w[0]
    if gap > 64 * EPS * scale and on[0, :3].any() and name not in SWAPPED_BY_THE_REFERENCE:
        n = oS[0].reshape(4, 4)[0, :3].astype(np.float64)   # first eigenvector (column 0 of the Stats matrix)
        ang = np.arcsin(min(1.0, np.linalg.norm(np.cross(n, V[:, 0]))))
        assert ang <= 8 * EPS * scale / gap, (name, ang, gap)


# ---- gates on their thresholds ----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_min_points_gate(ctx, variant2):
    P, idx, itv, _ = case_inputs("curved")
    n = len(CASES["curved"][0])
    for mp, computed in ((n, True), (n + 1, False), (n - 1, True)):
        p = case_params("curved", minPoints=mp)
        on, oS, oe, ocnt, _ = stage_compare("min_points=%d" % mp, ctx, P, idx, itv, oracle_sp(p), gpu_sp(p))
        assert (ocnt[0] == n) == computed


@pytest.mark.gpu
def test_interval_gate_stage(ctx, variant2):
    """interval k at -1, minR - 1, minR, maxR, maxR + 1 (minR = 1, maxR = 3): the window radius the kernels use is clamp(k),
    and -1 skips the pixel; the counts are checked against the getRegion rule in integers"""
    P, idx, _, _ = case_inputs("curved")
    valid = (idx >= 0).astype(np.int64)
    for k in (-1, 0, 1, 3, 4, 7):
        itv = np.where(idx >= 0, k, -1).astype(np.int32)
        p = case_params("curved")
        _, _, _, ocnt, _ = stage_compare("interval %d" % k, ctx, P, idx, itv, oracle_sp(p), gpu_sp(p))
        kk = clampi(k, 1, 3)
        r, c = CENTER
        y0, y1, x0, x1 = clampi(r - kk - 1, 0, ROWS - 1), clampi(r + kk - 1, 0, ROWS - 1), clampi(c - kk - 1, 0, COLS - 1), \
            clampi(c + kk - 1, 0, COLS - 1)
        want = 0 if k < 0 else int(valid[y0 + 1:y1 + 1, x0 + 1:x1 + 1].sum())
        assert ocnt[0] == want, (k, ocnt[0], want)


def depth_crossing(ivx, m):
    """float32 depths (d_lo, d_hi), adjacent floats, with (int)(ivx * (1 / d)) >= m at d_lo and < m at d_hi (float32)"""
    d = f32(ivx / m)
    k = lambda x: int(f32(ivx) * (f32(1) / f32(x)))
    while k(d) < m:
        d = np.nextafter(d, f32(0))
    while k(np.nextafter(d, f32(np.inf))) >= m:
        d = np.nextafter(d, f32(np.inf))
    return d, np.nextafter(d, f32(np.inf))


@pytest.mark.gpu
def test_interval_gate_converter(ctx, variant2):
    """the converter's interval (int)(ivx / d): depths on both sides of the crossings of minR - 1, minR, maxR, maxR + 1"""
    from g2o_frontend_b200 import capi
    K = np.array([[100.0, 0, 12], [0, 100.0, 9], [0, 0, 1]], np.float32)
    wr = 0.1
    ivx = f32(f32(K[0, 0] * f32(wr)) + f32(K[0, 1] * f32(wr)))
    minR, maxR = 2, 5
    ds, want = [], set()
    for m in (minR - 1, minR, maxR, maxR + 1):
        lo, hi = depth_crossing(ivx, m)
        ds += [lo, hi]
        want |= {m, m - 1}
    rows, cols = 18, 24
    yy, xx = np.mgrid[0:rows, 0:cols]
    depth = np.array(ds, np.float32)[(yy + 3 * xx) % len(ds)]
    depth[::7, ::5] = 0  # holes
    sp = O.default_stats_params(worldRadius=wr, minImageRadius=minR, maxImageRadius=maxR, minPoints=3, curvatureThreshold=0.5)
    oc, oidx, oitv, ointeg = O.depth_to_cloud(depth, K, 0.5, 20.0, sp, want_aux=True)
    assert want <= set(np.unique(oitv).tolist()), (want, np.unique(oitv))
    gsp = capi.make_stats_params(wr, minR, maxR, 3, 0.5, 0.02)
    cl, idx = ctx.depth_to_cloud(depth, capi.make_projector(K, rows, cols, 0.5, 20.0), gsp, keep_stats=True)
    assert np.array_equal(idx, oidx) and np.array_equal(ctx.last_interval_image(rows, cols), oitv)
    check_cloud("interval crossings", gpu_cloud(cl), oc, cov_lookup(oidx, oitv, ointeg, sp))


@pytest.mark.gpu
def test_curvature_thresholds(ctx, variant2):
    """curvature_threshold and omega_curvature_threshold set to the exact curvature of a window, and one ulp to either side:
    the normal is kept / the window is flat exactly when curvature < threshold"""
    P, idx, itv, _ = case_inputs("curved")
    p = case_params("curved", curvatureThreshold=1.0)
    _, _, _, _, ocurv = O.stats_stage(O.integral_image(idx, P), idx, itv, P, oracle_sp(p))
    c = f32(ocurv[0])
    assert 0 < c < 0.5
    for thr in (np.nextafter(c, f32(0)), c, np.nextafter(c, f32(1))):
        p = case_params("curved", curvatureThreshold=float(thr))
        on, oS, oe, ocnt, curv = stage_compare("curvature_threshold %r" % thr, ctx, P, idx, itv, oracle_sp(p), gpu_sp(p))
        assert bool(on[0, :3].any()) == bool(c < thr)
    for thr in (np.nextafter(c, f32(0)), c, np.nextafter(c, f32(1))):
        p = case_params("curved", curvatureThreshold=1.0, omegaCurvatureThreshold=float(thr))
        on, oS, oe, ocnt, curv = stage_compare("omega_curvature_threshold %r" % thr, ctx, P, idx, itv, oracle_sp(p), gpu_sp(p))
        oP, oN = O.information_stage(on, oS, oe, curv, oracle_sp(p))
        assert O.sym6(oN)[0, 0] == (100.0 if c < thr else 1.0)


@pytest.mark.gpu
def test_orientation_on_a_plane_through_the_origin(ctx, variant2):
    """dot(n, p) == 0 exactly: no flip (the comparison is > 0)"""
    P, idx, itv, _ = case_inputs("plane_through_origin")
    p = case_params("plane_through_origin")
    on, *_ = stage_compare("plane through the origin", ctx, P, idx, itv, oracle_sp(p), gpu_sp(p))
    dots = [f32(f32(f32(on[i, 0] * P[i, 0]) + f32(on[i, 1] * P[i, 1])) + f32(on[i, 2] * P[i, 2])) for i in range(len(P))
            if on[i, :3].any()]
    assert dots and all(d == 0 for d in dots), dots


@pytest.mark.gpu
def test_windows_clipped_by_the_borders(ctx, variant2):
    """every pixel valid, radius 3 everywhere: windows clipped by all four borders, including the getRegion clamp that
    leaves out row and column 0; the counts against the rule in integers"""
    rows, cols = 9, 11
    yy, xx = np.mgrid[0:rows, 0:cols].astype(np.float32)
    P = np.stack([0.05 * xx, 0.05 * yy, 2.0 + 0.01 * xx * xx - 0.02 * yy, np.ones_like(xx)], -1).reshape(-1, 4).astype(np.float32)
    idx = np.arange(rows * cols, dtype=np.int32).reshape(rows, cols)
    itv = np.full((rows, cols), 3, np.int32)
    p = dict(minImageRadius=1, maxImageRadius=3, minPoints=1, curvatureThreshold=0.5)
    _, _, _, ocnt, _ = stage_compare("borders", ctx, P, idx, itv, oracle_sp(p), gpu_sp(p))
    for r in range(rows):
        for c in range(cols):
            y0, y1 = clampi(r - 4, 0, rows - 1), clampi(r + 2, 0, rows - 1)
            x0, x1 = clampi(c - 4, 0, cols - 1), clampi(c + 2, 0, cols - 1)
            assert ocnt[idx[r, c]] == (y1 - y0) * (x1 - x0), (r, c)


@pytest.mark.gpu
def test_zero_omega_curvature_threshold_on_flat_windows(ctx, variant2):
    """omega_curvature_threshold = 0: every window, flat ones included, takes the non-flat Omega_P = U diag(1 / eigenvalues)
    U^T.  Where the solver's smallest eigenvalue is exactly 0 (a plane through the origin, a line, a flat tetrahedron) that
    is inf / NaN, as in the reference; where rounding leaves it a few ulps above 0 (the fronto-parallel and oblique 3x3
    planes, 2.5e-9 and 1.2e-7) it is finite and huge.  The bar is the oracle's bits either way."""
    zero = finite = 0
    for name in ("plane_fronto", "plane_oblique", "plane_through_origin", "line_z", "d0_half_eps", "diag_1_q_0"):
        P, idx, itv, _ = case_inputs(name)
        p = case_params(name, omegaCurvatureThreshold=0.0)
        on, oS, oe, ocnt, curv = stage_compare("omega threshold 0, %s" % name, ctx, P, idx, itv, oracle_sp(p), gpu_sp(p))
        oP, _ = O.information_stage(on, oS, oe, curv, oracle_sp(p))
        assert on[0, :3].any() and curv[0] >= 0, name
        assert np.isfinite(O.sym6(oP)[0]).all() == (oe[0, 0] != 0), (name, oe[0], O.sym6(oP)[0])
        zero += oe[0, 0] == 0
        finite += oe[0, 0] != 0
    assert zero >= 3 and finite >= 3


# ---- the column-pass kernels at their switch points ---------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("rows", [1600, 1601])
@pytest.mark.parametrize("frames", [1, 3, 4, 5])
def test_column_pass_switch_points(ctx, variant2, rows, frames):
    """a launch set of F frames: F >= 4 streams the columns (k_integral_cols_stream), fewer frames stage 32-column strips in
    shared memory up to 1600 rows (k_integral_cols_smem) and walk them in registers above (k_integral_cols)"""
    from g2o_frontend_b200 import capi, synth
    cols = 48
    K = np.array([[300.0, 0, cols / 2], [0, 300.0, rows / 2], [0, 0, 1]], np.float32)
    rng = np.random.default_rng(rows + frames)
    raws = [synth.render_depth_u16(synth.perturbed_pose(rng, np.eye(4), 0.2, 5.0), rows, cols, K, seed=70 + i, dropout=0.03)
            for i in range(frames)]
    c = CONF_1_4
    osp = O.default_stats_params(minImageRadius=c["minImageRadius"], maxImageRadius=c["maxImageRadius"],
                                 minPoints=c["minPoints"], curvatureThreshold=c["curvatureThreshold"])
    gsp = capi.make_stats_params(c["worldRadius"], c["minImageRadius"], c["maxImageRadius"], c["minPoints"],
                                 c["curvatureThreshold"], c["omegaCurvatureThreshold"])
    clouds = ctx.raw_depth_to_cloud_batch(raws, capi.make_projector(K, rows, cols, c["minD"], c["maxD"]), gsp, keep_stats=True)
    ctx.synchronize()
    for f, (raw, cl) in enumerate(zip(raws, clouds)):
        oc, oidx, oitv, ointeg = O.depth_to_cloud(O.depth_u16_to_f32(raw), K, c["minD"], c["maxD"], osp, want_aux=True)
        assert cl.size() == oc.n > 0
        check_cloud("%d rows, frame %d of %d" % (rows, f, frames), gpu_cloud(cl), oc, cov_lookup(oidx, oitv, ointeg, osp))


@pytest.mark.gpu
@pytest.mark.parametrize("step", [1, 2])
def test_1080p_rig_column_pass(ctx, variant2, step):
    """a 4-camera 1920x1080 rig (composite 1920 x 4320 at step 1): one frame per launch set, so step 1 takes the register
    fallback of the column pass (1920 rows) and step 2 the shared-memory strips (960 rows)"""
    from g2o_frontend_b200 import capi, synth
    from test_rig_batch import render_raw_frame, rig_poses
    cams = synth.make_rig(4, 1920 // step, 1080 // step, K=synth.scaled_K(synth.K_KINECT, 1920 / 640.0 / step))
    frames = [render_raw_frame(rig_poses(1, 21)[0], cams, step, 90)]
    osp = O.default_stats_params(curvatureThreshold=0.2)
    gsp = capi.make_stats_params(0.1, 10, 30, 50, 0.2, 0.02)
    rig_compare("1080p rig, step %d" % step, ctx, cams, frames, step, osp, gsp, None)


# ---- size limits --------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_size_limits_are_rejected_up_front(ctx):
    """a row pass wider than NICP_MAX_PREP_COLS and more than NICP_MAX_PREP_PIXELS pixels: NICP_ERR_INVALID naming the size,
    before anything is launched; the same context then prepares a valid frame"""
    from g2o_frontend_b200 import capi, synth
    L = ctx.L
    cams = synth.make_rig(6, 1920, 1080)
    mp = capi.make_multi_projector(cams)
    assert capi.multi_image_size(mp, ctx.verify) == (1920, 6480)
    frame = [np.zeros((1080, 1920), np.uint16)] * 6
    sp = capi.make_stats_params()
    small = ctx.new_cloud(1)

    def rejected(fn, needle):
        before = ctx.launch_count()
        with pytest.raises(capi.NicpError) as e:
            fn()
        assert "nicp error 1:" in str(e.value) and needle in str(e.value), str(e.value)
        assert ctx.launch_count() == before
        s = get_scene(4)
        cl, idx = ctx.depth_to_cloud(s.depthA, s.projector(), s.stats_params())
        assert np.array_equal(idx, s.indexA) and np.array_equal(canon(cl.download()["points"]), canon(s.cloudA.points))

    rejected(lambda: ctx.multi_raw_depth_to_cloud_batch([frame], mp, sp, clouds=[small]), "6480 columns")
    rejected(lambda: ctx.stats_compute(np.zeros((1, 4), np.float32), np.full((1, 6480), -1, np.int32),
                                       np.full((1, 6480), -1, np.int32), sp), "6480 columns")
    rows, cols = 4097, 4096
    K = np.array([[1000.0, 0, cols / 2], [0, 1000.0, rows / 2], [0, 0, 1]], np.float32)
    proj = capi.make_projector(K, rows, cols, 0.5, 4.5)
    raw = np.zeros((rows, cols), np.uint16)
    needle = "4097 x 4096 = 16781312 pixels"
    rejected(lambda: ctx.raw_depth_to_cloud(raw, proj, sp, cloud=small), needle)
    rejected(lambda: ctx.raw_depth_to_cloud_batch([raw], proj, sp, clouds=[small]), needle)
    rejected(lambda: ctx.depth_to_cloud(np.zeros((rows, cols), np.float32), proj, sp, cloud=small, want_index=False), needle)
    rejected(lambda: ctx.stats_compute(np.zeros((1, 4), np.float32), np.full((rows, cols), -1, np.int32),
                                       np.full((rows, cols), -1, np.int32), sp), needle)


@pytest.mark.gpu
def test_largest_image_every_pixel_valid(ctx):
    """4096 x 4096 = 2^24 valid pixels, the most the float32 pixel counts hold exactly: the index image is the raster
    order and the cloud has 2^24 points"""
    from g2o_frontend_b200 import capi
    n = 4096
    K = np.array([[1000.0, 0, n / 2], [0, 1000.0, n / 2], [0, 0, 1]], np.float32)
    depth = np.full((n, n), 1.5, np.float32)
    sp = capi.make_stats_params(0.1, 1, 3, 4, 0.02, 0.02)
    cl, idx = ctx.depth_to_cloud(depth, capi.make_projector(K, n, n, 0.5, 4.5), sp)
    assert cl.size() == 1 << 24
    want = np.cumsum(np.ones(n * n, np.int64)) - 1
    assert np.array_equal(idx.reshape(-1), want)
    cl.close()

"""The fused correspondence + linearise kernels (corr_lin.cuh: k_corr_lin_group and k_corr_lin_tiled) at the edges where the
realistic scenes of test_gpu_parity.py never go, in both builds and through both kernels:

- every correspondence gate exactly on its threshold and one ulp to either side, hand-built in numpy with the float32
  operation order of dot3 / xform_point / xform_normal, including the float32 pre-test band of the curvature ratio and a
  ratio threshold below 1;
- the chi2 cut of the Linearizer with the robust kernel on and off, at thresholds that cut a quarter to all but a tenth of
  the terms (the parity scenes keep every term at inlierMaxChi2 = 9000);
- whole teacher-forced iterations with the cut engaged, single and batched;
- NICP_GROUP_MIN_AVG, which must only choose the kernel, never change a result.

The hand-built cases are checked on the CPU, through the oracle alone, to land where they are meant to."""
import ctypes as C

import numpy as np
import pytest

from conftest import get_scene

F = np.float32
H_RTOL = 1e-4
T_TOL = 1e-4
NORMAL_THR = 0.95
DIST_THR = 0.3
GATE_THRS = (1.3, 1.0, 0.5)    # inlierCurvatureRatioThreshold
FLATS = (0.02, 0.0)            # flatCurvatureThreshold
SIZES = ((1, 1), (1, 95), (1, 97), (3, 65), (37, 53))
TILE = 96                      # pixels per warp tile of both kernels (kTilePixels)


def frob_rel(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def rot_angle(Ra, Rb):
    R = Ra.astype(np.float64).T @ Rb.astype(np.float64)
    w = np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]]) / 2
    return float(np.arcsin(min(1.0, np.linalg.norm(w))))


def ulp_step(x, k):
    """x moved by k float32 ulps (x > 0 or the steps do not cross zero)"""
    return (np.asarray(x, F).reshape(1).view(np.int32) + np.int32(k)).view(F)[0]


# ---- float32 arithmetic in the order of nicp_math.cuh (numpy rounds every float32 operation) ----
def dot3(a, b):
    return (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]


def xform(T, v, point):
    """rows 0..2 of T (v, 1) (xform_point) or T (v, 0) (xform_normal); v: (3,) or (n, 3) float32"""
    T = np.asarray(T, F)
    v = np.asarray(v, F)
    out = np.empty_like(v)
    for i in range(3):
        r = (T[i, 0] * v[..., 0] + T[i, 1] * v[..., 1]) + T[i, 2] * v[..., 2]
        out[..., i] = r + T[i, 3] if point else r
    return out


def iso_inverse(T):
    """Isometry3f::inverse() as the aligner forms state->invT from a guess"""
    T = np.asarray(T, F)
    o = np.eye(4, dtype=F)
    o[:3, :3] = T[:3, :3].T
    for r in range(3):
        o[r, 3] = -((o[r, 0] * T[0, 3] + o[r, 1] * T[1, 3]) + o[r, 2] * T[2, 3])
    return o


def ratio(rc, cc):
    """(rc + 1e-5) / (cc + 1e-5) in float64, rounded to float (correspondencefinder.cpp:87-99)"""
    return F((np.float64(rc) + 1e-5) / (np.float64(cc) + 1e-5))


def gate_consts(thr, flat):
    return dict(nt=F(NORMAL_THR), sq=F(DIST_THR) * F(DIST_THR), flat=F(flat), lo=F(1.0) / F(thr), hi=F(thr))


def emulate_gates(case, T, g):
    """correspondencefinder.cpp:64-99 for one hand-built case, in numpy: the verdict the oracle must reach"""
    rn0, cn = case["rn0"], case["cn"]
    if dot3(cn, cn) == 0 or dot3(rn0, rn0) == 0:
        return False
    rn, rp = xform(T, rn0, False), xform(T, case["rp0"], True)
    if dot3(cn, rn) < g["nt"]:
        return False
    d = case["cp"] - rp
    if dot3(d, d) > g["sq"]:
        return False
    rc, cc = max(case["rc"], g["flat"]), max(case["cc"], g["flat"])
    r = ratio(rc, cc)
    return not (r < g["lo"] or r > g["hi"])


# ---- hand-built gate cases -----------------------------------------------------------------------------------------
def _solve_dot(rn, target, rng):
    """a current normal cn (about unit length) with dot3(cn, rn) == target exactly"""
    u = rn.astype(np.float64) / np.linalg.norm(rn.astype(np.float64))
    steps = np.arange(-4096, 4097, dtype=np.int32)
    for _ in range(64):
        w = np.cross(u, rng.normal(size=3))
        w /= np.linalg.norm(w)
        c = (float(target) * u + np.sqrt(max(0.0, 1.0 - float(target) ** 2)) * w).astype(F)
        if np.abs(c).min() < 0.05:
            continue
        X = (c[0:1].view(np.int32) + steps).view(F)
        for dy in range(-16, 17):
            Y = ulp_step(c[1], dy)
            d = (X * rn[0] + Y * rn[1]) + c[2] * rn[2]
            hit = np.flatnonzero(d == target)
            if hit.size:
                return np.array([X[hit[0]], Y, c[2]], F)
    raise AssertionError("no normal with dot3 == %r" % target)


def _solve_sq(rp, target, rng):
    """a current point cp with dot3(cp - rp, cp - rp) == target exactly"""
    steps = np.arange(-4096, 4097, dtype=np.int32)
    for _ in range(64):
        u = rng.normal(size=3)
        u /= np.linalg.norm(u)
        c = (rp.astype(np.float64) + np.sqrt(float(target)) * u).astype(F)
        if np.abs(c - rp).min() < 0.05:
            continue
        X = (c[0:1].view(np.int32) + steps).view(F)
        dz = c[2] - rp[2]
        for dy in range(-16, 17):
            Y = ulp_step(c[1], dy)
            dx, dyv = X - rp[0], Y - rp[1]
            s = (dx * dx + dyv * dyv) + dz * dz
            hit = np.flatnonzero(s == target)
            if hit.size:
                return np.array([X[hit[0]], Y, c[2]], F)
    raise AssertionError("no point with squared distance == %r" % target)


def _solve_ratio(target, cc_list):
    """(rc, cc) with ratio(rc, cc) == target exactly, both above every flat threshold used here"""
    steps = np.arange(-1024, 1025, dtype=np.int32)
    for cc in cc_list:
        cc = F(cc)
        rc0 = F(np.float64(target) * (np.float64(cc) + 1e-5) - 1e-5)
        R = (np.array([rc0], F).view(np.int32) + steps).view(F)
        r = ((R.astype(np.float64) + 1e-5) / (np.float64(cc) + 1e-5)).astype(F)
        hit = np.flatnonzero((r == target) & (R != cc) & (R > 0.021))
        if hit.size:
            return R[hit[0]], cc
    raise AssertionError("no curvature pair with ratio == %r" % target)


_CASES = {}


def gate_cases(thr, flat, rigid):
    """list of cases, each one reference point / normal / curvature and one current point / normal / curvature, plus
    `probe`: what the case pins (checked by test_gate_cases_land_on_their_thresholds)"""
    key = (thr, flat, rigid)
    if key in _CASES:
        return _CASES[key]
    T = gate_transform(rigid)
    g = gate_consts(thr, flat)
    rng = np.random.default_rng(7)
    cases = []

    def base(probe):
        rp0 = rng.uniform((-1.0, -1.0, 1.0), (1.0, 1.0, 3.0)).astype(F)
        rn0 = rng.normal(size=3)
        rn0 = (rn0 / np.linalg.norm(rn0)).astype(F)
        rp, rn = xform(T, rp0, True), xform(T, rn0, False)
        off = rng.normal(size=3)
        cp = (rp.astype(np.float64) + 0.05 * off / np.linalg.norm(off)).astype(F)
        c = dict(rp0=rp0, rn0=rn0, rc=F(0.05), cp=cp, cn=rn.copy(), cc=F(0.05), probe=probe)
        cases.append(c)
        return c, rp, rn

    for _ in range(3):
        base(("plain",))
    # normal angle (correspondencefinder.cpp:78): kept at == threshold, rejected one ulp below
    for k in (0, -1, 1):
        c, rp, rn = base(("dot", k))
        c["cn"] = _solve_dot(rn, ulp_step(g["nt"], k), rng)
    c, _, _ = base(("zero_ref_normal",))
    c["rn0"] = np.zeros(3, F)
    c, _, _ = base(("zero_cur_normal",))
    c["cn"] = np.zeros(3, F)
    # distance (:84): kept at == squared threshold, rejected one ulp above
    for k in (0, 1, -1):
        c, rp, rn = base(("sq", k))
        c["cp"] = _solve_sq(rp, ulp_step(g["sq"], k), rng)
    # curvature ratio (:87-99): equal curvatures -- unclamped, both clamped, one clamped onto the other
    for rc, cc in ((0.05, 0.05), (0.001, 0.005), (0.01, 0.02), (0.02, 0.01)):
        c, _, _ = base(("equal", rc, cc))
        c["rc"], c["cc"] = F(rc), F(cc)
    # float(ratio) exactly at the thresholds and one ulp either side of each
    # (a quotient that rounds to exactly 1 from rc != cc needs cc one ulp under a power of two and rc on it)
    cc_list = (0.05, 0.0503, 0.0611, 0.0717, 0.083, 0.0947, ulp_step(F(0.0625), -1), ulp_step(F(0.125), -1))
    for side in ("lo", "hi"):
        for k in (0, -1, 1):
            c, _, _ = base(("ratio", side, k))
            c["rc"], c["cc"] = _solve_ratio(ulp_step(g[side], k), cc_list)
    # quotients just inside the 1e-4 band around a threshold (the float64 quotient decides) and just outside it (the
    # float32 pre-test decides), on both sides of both thresholds
    for side in ("lo", "hi"):
        for rel in (-1.1e-4, -0.9e-4, 0.9e-4, 1.1e-4):
            c, _, _ = base(("band", side, rel))
            cc = F(0.05)
            c["rc"], c["cc"] = F(np.float64(g[side]) * (1.0 + rel) * (np.float64(cc) + 1e-5) - 1e-5), cc
    # curvature exactly at the flat threshold and one ulp under it (clamped onto it)
    under = np.nextafter(g["flat"], F(-1))
    for rc, cc in ((g["flat"], under), (under, g["flat"]), (under, under), (g["flat"], g["flat"])):
        c, _, _ = base(("flat", float(rc), float(cc)))
        c["rc"], c["cc"] = F(rc), F(cc)
    _CASES[key] = cases
    return cases


def gate_transform(rigid):
    from g2o_frontend_b200 import synth
    if not rigid:
        return np.eye(4, dtype=F)
    T = synth.make_pose((0.2, -0.1, 0.15), (0.4, 1.0, -0.3), 23.0).astype(F)
    T[3] = (0, 0, 0, 1)
    return T


def gate_clouds(cases):
    """two oracle clouds: case i is reference point i and current point i"""
    from oracle import pwn_oracle as O
    n = len(cases)
    R, Cc = O.Cloud(n), O.Cloud(n)
    omP = np.array([[60.0, 5.0, -3.0], [5.0, 90.0, 7.0], [-3.0, 7.0, 140.0]])
    omN = np.array([[8.0, 1.0, 0.0], [1.0, 12.0, -2.0], [0.0, -2.0, 10.0]])
    for i, c in enumerate(cases):
        R.points[i] = (*c["rp0"], 1.0)
        R.normals[i, :3] = c["rn0"]
        R.curvature[i] = c["rc"]
        Cc.points[i] = (*c["cp"], 1.0)
        Cc.normals[i, :3] = c["cn"]
        Cc.curvature[i] = c["cc"]
        s = 1.0 + 0.25 * (i % 5)
        P4, N4 = np.eye(4), np.eye(4)
        P4[:3, :3], N4[:3, :3] = s * omP, omN / s
        Cc.omegaP[i] = P4.T.reshape(16)
        Cc.omegaN[i] = N4.T.reshape(16)
        R.omegaP[i], R.omegaN[i] = Cc.omegaP[i], Cc.omegaN[i]
    return R, Cc


def gate_layout(rows, cols, n):
    """index images: every pixel shows a case drawn at random (seeded; over the tiles every lane and pixel slot of a tile
    sees accepted and rejected cases), with scattered pixels that lack one side, and -- where the image is large enough --
    a tile without any current pixel and a tile without any reference pixel"""
    P = rows * cols
    p = np.arange(P)
    ri = np.random.default_rng(0).integers(0, n, P)
    ci = ri.copy()
    ri[p % 11 == 10] = -1
    ci[p % 13 == 12] = -1
    if P > 5 * TILE:
        ci[4 * TILE:5 * TILE] = -1
    if P > 10 * TILE:
        ri[9 * TILE:10 * TILE] = -1
    return ri.reshape(rows, cols).astype(np.int32), ci.reshape(rows, cols).astype(np.int32)


def corr_params(thr, flat):
    from oracle import pwn_oracle as O
    return O.default_corr_params(inlierDistanceThreshold=DIST_THR, inlierNormalAngularThreshold=NORMAL_THR,
                                 flatCurvatureThreshold=flat, inlierCurvatureRatioThreshold=thr)


def gpu_align_params(thr, flat, max_chi2=9000.0, robust=True, outer=10, inner=1, dist=DIST_THR, normal=NORMAL_THR):
    from g2o_frontend_b200 import capi
    return capi.make_align_params(dist, normal, flat, thr, max_chi2, robust, outer, inner)


# ---- CPU: the constructed cases pin what they are meant to ---------------------------------------------------------
@pytest.mark.parametrize("thr", GATE_THRS)
@pytest.mark.parametrize("flat", FLATS)
@pytest.mark.parametrize("rigid", [False, True])
def test_gate_cases_land_on_their_thresholds(thr, flat, rigid):
    from oracle import pwn_oracle as O
    cases = gate_cases(thr, flat, rigid)
    T = gate_transform(rigid)
    g = gate_consts(thr, flat)
    in_band = 0
    for c in cases:
        kind = c["probe"][0]
        rn, rp = xform(T, c["rn0"], False), xform(T, c["rp0"], True)
        if kind == "dot":
            assert dot3(c["cn"], rn) == ulp_step(g["nt"], c["probe"][1]), c["probe"]
        elif kind == "sq":
            d = c["cp"] - rp
            assert dot3(d, d) == ulp_step(g["sq"], c["probe"][1]), c["probe"]
        elif kind == "ratio":
            _, side, k = c["probe"]
            assert c["rc"] != c["cc"] and min(c["rc"], c["cc"]) > g["flat"]
            assert ratio(c["rc"], c["cc"]) == ulp_step(g[side], k), c["probe"]
        elif kind == "band":
            _, side, rel = c["probe"]
            q = (np.float64(c["rc"]) + 1e-5) / (np.float64(c["cc"]) + 1e-5)
            off = q / np.float64(g[side]) - 1.0
            assert np.sign(off) == np.sign(rel) and abs(abs(off) - abs(rel)) < 2e-6, (c["probe"], off)
            in_band += abs(off) < 1e-4
        elif kind == "flat":
            _, rc, cc = c["probe"]
            assert {c["rc"], c["cc"]} <= {g["flat"], np.nextafter(g["flat"], F(-1))}
    assert in_band == 4
    # the neighbours fall on the other side: verdicts of the oracle on a 1 x n image, and of the numpy emulation
    R, Cc = gate_clouds(cases)
    n = len(cases)
    ri = np.arange(n, dtype=np.int32).reshape(1, n)
    corr, cimg = O.correspond(ri, ri, R, Cc, T, corr_params(thr, flat), num_threads=1)
    got = cimg[0] >= 0
    want = np.array([emulate_gates(c, T, g) for c in cases])
    assert np.array_equal(got, want), [c["probe"] for c, a, b in zip(cases, got, want) if a != b]
    verdict = {c["probe"]: bool(v) for c, v in zip(cases, got)}
    # what each neighbour pins, independent of the ratio threshold
    if thr >= 1.0:
        assert verdict[("dot", 0)] and not verdict[("dot", -1)] and verdict[("dot", 1)]
        assert verdict[("sq", 0)] and not verdict[("sq", 1)] and verdict[("sq", -1)]
        assert not verdict[("zero_ref_normal",)] and not verdict[("zero_cur_normal",)]
        assert verdict[("ratio", "hi", 0)] and not verdict[("ratio", "hi", 1)]
        assert verdict[("ratio", "lo", 0)] and not verdict[("ratio", "lo", -1)]
        assert verdict[("equal", 0.05, 0.05)]
    if thr > 1.0:
        assert verdict[("ratio", "hi", -1)] and verdict[("ratio", "lo", 1)]
        assert [verdict[("band", "hi", r)] for r in (-1.1e-4, -0.9e-4, 0.9e-4, 1.1e-4)] == [True, True, False, False]
        assert [verdict[("band", "lo", r)] for r in (-1.1e-4, -0.9e-4, 0.9e-4, 1.1e-4)] == [False, False, True, True]
    if thr == 1.0:
        # a quotient one ulp off 1 is rejected, so the clamp onto the flat threshold decides these
        assert not verdict[("ratio", "hi", -1)] and not verdict[("ratio", "lo", 1)]
        assert all(verdict[p] for p in verdict if p[0] == "flat")
    if thr < 1.0:  # 1 lies outside [1 / thr, thr]: the reference rejects every pair
        assert not got.any()
    # every lane and pixel slot of a tile sees both verdicts on the largest image
    if thr > 1.0 and flat > 0:
        ri2, ci2 = gate_layout(37, 53, n)
        _, cimg2 = O.correspond(ri2, ci2, R, Cc, T, corr_params(thr, flat), num_threads=1)
        acc = (cimg2.reshape(-1) >= 0)
        rej = (ri2.reshape(-1) >= 0) & (ci2.reshape(-1) >= 0) & ~acc
        P = acc.size
        pos = np.arange(P) % TILE
        for m in (acc, rej):
            assert np.array_equal(np.unique(pos[m]), np.arange(TILE))


# ---- GPU contexts: both builds x both kernels ----------------------------------------------------------------------
KERNELS = {"grouped": "0", "per_pair": "1000"}


@pytest.fixture(scope="module")
def contexts():
    from g2o_frontend_b200 import capi
    out = {}
    for verify in (True, False):
        for kernel, avg in KERNELS.items():
            with pytest.MonkeyPatch.context() as mp:
                mp.setenv("NICP_GROUP_MIN_AVG", avg)
                out[(verify, kernel)] = capi.Context(0, verify=verify)
            assert bool(out[(verify, kernel)].L.nicp_is_verification_build()) == verify
    yield out
    for c in out.values():
        c.close()


def upload(ctx, oc):
    cl = ctx.new_cloud(max(oc.n, 1))
    cl.upload(oc.points, oc.normals, oc.curvature, oc.omegaP6(), oc.omegaN6())
    return cl


def check_stage(got, corr_o, cimg_o, R, Cc, T, max_chi2, robust):
    """correspond_linearize output against the oracle: correspondence image bit-exact, count and inliers exact, H / b /
    error within 1e-4 of the float64-accumulated sums of the same terms"""
    from oracle import pwn_oracle as O
    H, b, err, inl, nc, cimg = got
    assert np.array_equal(cimg, cimg_o)
    assert nc == corr_o.shape[0]
    check_lin((H, b, err, inl), O.linearize_f64(corr_o, R, Cc, T, max_chi2, robust))


def check_lin(got, want):
    H, b, err, inl = got
    H64, b64, err64, inl64 = want
    assert inl == inl64, (inl, inl64)
    assert frob_rel(H, H64) <= H_RTOL, frob_rel(H, H64)
    assert frob_rel(b, b64) <= H_RTOL, frob_rel(b, b64)
    assert abs(err - err64) <= H_RTOL * abs(err64), (err, err64)


@pytest.mark.gpu
@pytest.mark.parametrize("verify", [True, False])
@pytest.mark.parametrize("kernel", list(KERNELS))
@pytest.mark.parametrize("thr", GATE_THRS)
@pytest.mark.parametrize("flat", FLATS)
def test_gates_at_their_thresholds(contexts, verify, kernel, thr, flat):
    """every hand-built gate case on images whose last tile is partial or that have tiles without a pixel, at T = I and a
    general rigid T: the correspondence image bit for bit, the sums within 1e-4"""
    from oracle import pwn_oracle as O
    ctx = contexts[(verify, kernel)]
    ap = gpu_align_params(thr, flat)
    for rigid in (False, True):
        cases = gate_cases(thr, flat, rigid)
        T = gate_transform(rigid)
        R, Cc = gate_clouds(cases)
        ref, cur = upload(ctx, R), upload(ctx, Cc)
        for rows, cols in SIZES:
            ri, ci = gate_layout(rows, cols, len(cases))
            corr_o, cimg_o = O.correspond(ri, ci, R, Cc, T, corr_params(thr, flat), num_threads=1)
            got = ctx.correspond_linearize(ref, cur, ri, ci, T, ap)
            check_stage(got, corr_o, cimg_o, R, Cc, T, 9000.0, True)
            if thr < 1.0:
                assert got[4] == 0
            elif rows * cols > 1:
                assert 0 < got[4] < ((ri >= 0) & (ci >= 0)).sum()


# ---- the chi2 cut ---------------------------------------------------------------------------------------------------
def chi2_of(corr, R, Cc, T):
    """per-correspondence chi2 of the Linearizer: errors in float32 exactly as the kernels form them (so the only
    difference to a kernel's chi2 is the order of the quadratic form's sum), the form in float64"""
    r, q = corr[:, 0], corr[:, 1]
    ep = (xform(T, R.points[r, :3], True) - Cc.points[q, :3]).astype(np.float64)
    en = (xform(T, R.normals[r, :3], False) - Cc.normals[q, :3]).astype(np.float64)
    OP = Cc.omegaP.reshape(-1, 4, 4)[q, :3, :3].astype(np.float64)
    ON = Cc.omegaN.reshape(-1, 4, 4)[q, :3, :3].astype(np.float64)
    return np.einsum("ni,nij,nj->n", ep, OP, ep) + np.einsum("ni,nij,nj->n", en, ON, en)


def pick_gap(chi, lo_q, hi_q):
    """inlierMaxChi2 in the widest relative gap of the chi2 distribution between two quantiles, no chi2 within 1e-5
    (relative) of it: the kernels' float32 chi2 and the oracle's then reach the same verdict on every term"""
    s = np.sort(chi)
    n = s.size
    i0, i1 = int(lo_q * n), int(hi_q * n)
    g = (s[i0 + 1:i1 + 1] - s[i0:i1]) / s[i0 + 1:i1 + 1]
    k = i0 + int(np.argmax(g))
    m = F(np.sqrt(s[k] * s[k + 1]))
    assert np.abs(chi - np.float64(m)).min() > 1e-5 * m, (lo_q, hi_q, g.max())
    return float(m)


CUTS = ((0.23, 0.27), (0.48, 0.52), (0.86, 0.89))  # near the 25th, 50th and 90th percentiles

_STAGE = {}


def stage_inputs(step, at_gt):
    """the oracle's index images, correspondences and the chi2 thresholds of one scene and pose"""
    key = (step, at_gt)
    if key not in _STAGE:
        from oracle import pwn_oracle as O
        s = get_scene(step)
        c = s.conf
        guess = s.gt if at_gt else np.eye(4, dtype=F)
        KRt, _ = O.update_matrices(s.K, guess)
        ri, _ = O.project_KRt(s.cloudA.points, s.rows, s.cols, KRt, c["minD"], c["maxD"])
        KRtc, _ = O.update_matrices(s.K, np.eye(4, dtype=F))
        ci, _ = O.project_KRt(s.cloudB.points, s.rows, s.cols, KRtc, c["minD"], c["maxD"])
        invT = np.linalg.inv(guess.astype(np.float64)).astype(F)
        corr, cimg = O.correspond(ri, ci, s.cloudA, s.cloudB, invT, s.cp, num_threads=8)
        chi = chi2_of(corr, s.cloudA, s.cloudB, invT)
        _STAGE[key] = (s, ri, ci, invT, corr, cimg, chi, [pick_gap(chi, a, b) for a, b in CUTS])
    return _STAGE[key]


@pytest.mark.gpu
@pytest.mark.parametrize("verify", [True, False])
@pytest.mark.parametrize("kernel", list(KERNELS))
@pytest.mark.parametrize("step", [4, 1])
def test_chi2_cut_robust_on_and_off(contexts, verify, kernel, step):
    """inlierMaxChi2 that cuts 11-77 % of the terms, robust kernel on (the term scaled by sqrt(maxChi2 / chi2)) and off
    (the term dropped): through correspond_linearize (MODE 0) and linearize over the oracle's list (MODE 1, also 0, 1 and
    97 terms), inliers exact, H / b / error within 1e-4 of the float64-accumulated oracle"""
    from oracle import pwn_oracle as O
    ctx = contexts[(verify, kernel)]
    for at_gt in (False, True):
        s, ri, ci, invT, corr, cimg, chi, cuts = stage_inputs(step, at_gt)
        c = s.conf
        ref, cur = upload(ctx, s.cloudA), upload(ctx, s.cloudB)
        for m in cuts:
            cut = int((chi > m).sum())
            assert cut >= 0.1 * chi.size
            for robust in (False, True):
                ap = gpu_align_params(c["inlierCurvatureRatioThreshold"], c["flatCurvatureThreshold"], m, robust,
                                      dist=c["inlierDistanceThreshold"], normal=c["inlierNormalAngularThreshold"])
                got = ctx.correspond_linearize(ref, cur, ri, ci, invT, ap)
                check_stage(got, corr, cimg, s.cloudA, s.cloudB, invT, m, robust)
                assert got[3] == (chi.size if robust else chi.size - cut)
                for k in (0, 1, 97, corr.shape[0]):
                    check_lin(ctx.linearize(ref, cur, corr[:k], invT, ap),
                              O.linearize_f64(corr[:k], s.cloudA, s.cloudB, invT, m, robust))


@pytest.mark.gpu
@pytest.mark.parametrize("verify", [True, False])
@pytest.mark.parametrize("kernel", list(KERNELS))
def test_chi2_cut_exact_at_the_threshold(contexts, verify, kernel):
    """Two terms with dyadic values, so every chi2 has the same bits however it is summed: e_p = (1/2, 0, 0) (chi2 1/4)
    and e_p = (2, 0, 0) (chi2 4), Omega_P = Omega_N = I, e_n = 0.  maxChi2 == 4 keeps the large term unscaled; one ulp
    below 4 without the robust kernel drops it; maxChi2 = 1 with the robust kernel scales it by exactly 1/2 (a power of
    two, which the approximate reciprocal and reciprocal square root return exactly)."""
    from oracle import pwn_oracle as O
    ctx = contexts[(verify, kernel)]
    R, Cc = O.Cloud(2), O.Cloud(2)
    for i, (ex, p) in enumerate(((0.5, (0.25, -0.5, 2.0)), (2.0, (1.0, 0.75, 3.0)))):
        R.points[i] = (p[0] + ex, p[1], p[2], 1.0)
        Cc.points[i] = (*p, 1.0)
        R.normals[i, :3] = Cc.normals[i, :3] = (0.0, 0.0, -1.0)
        R.curvature[i] = Cc.curvature[i] = 0.05
        Cc.omegaP[i] = Cc.omegaN[i] = np.eye(4, dtype=F).reshape(16)
    ref, cur = upload(ctx, R), upload(ctx, Cc)
    T = np.eye(4, dtype=F)
    corr = np.array([[0, 0], [1, 1]], np.int32)
    ri = np.array([[0, 1]], np.int32)
    full = O.linearize(corr, R, Cc, T, 4.0, True, num_threads=1)
    small = O.linearize(corr[:1], R, Cc, T, 4.0, True, num_threads=1)
    assert full[2] == F(4.25) and small[2] == F(0.25)
    cases = ((4.0, False, full, 2), (4.0, True, full, 2), (float(np.nextafter(F(4), F(0))), False, small, 1))
    for m, robust, want, inl in cases:
        ap = gpu_align_params(1.3, 0.02, m, robust, dist=3.0, normal=0.5)
        for H, b, err, n in (ctx.linearize(ref, cur, corr, T, ap), ctx.correspond_linearize(ref, cur, ri, ri, T, ap)[:4]):
            assert n == inl
            assert err == want[2] and np.array_equal(b, want[1]) and np.array_equal(H, want[0]), (m, robust, err, b)
    # robust, maxChi2 = chi2 / 4: the large term's error and b are halved, H is not scaled
    ap = gpu_align_params(1.3, 0.02, 1.0, True, dist=3.0, normal=0.5)
    big_b = full[1] - small[1]
    for H, b, err, n in (ctx.linearize(ref, cur, corr, T, ap), ctx.correspond_linearize(ref, cur, ri, ri, T, ap)[:4]):
        assert n == 2
        assert err == F(0.25) + F(2.0), err
        assert np.array_equal(b, small[1] + big_b / 2), (b, small[1], big_b)
        assert np.array_equal(H, full[0])


# ---- whole iterations with the cut engaged -----------------------------------------------------------------------------
_ITER = {}


def iteration_inputs(step, seed, dropout):
    """the oracle's pose at the start of iterations 0, 3 and 9 and one inlierMaxChi2 in a gap of the chi2 of all three
    iterations' correspondences (near their median)"""
    key = (step, seed, dropout)
    if key not in _ITER:
        from oracle import pwn_oracle as O
        s = get_scene(step, seed, dropout)
        out = O.align(s.cloudA, s.cloudB, s.oracle_align_params(num_threads=8))
        Ts = [out.trace_T[i] for i in (0, 3, 9)]
        chis = []
        for Ti in Ts:
            o = O.align(s.cloudA, s.cloudB, s.oracle_align_params(outer=1, guess=Ti, num_threads=8), want_trace=False)
            chis.append(chi2_of(o.corr, s.cloudA, s.cloudB, iso_inverse(Ti)))
        _ITER[key] = (s, Ts, pick_gap(np.concatenate(chis), 0.45, 0.55))
    return _ITER[key]


_ORACLE_ITER = {}


def oracle_iteration(s, Ti, m, robust, inner):
    from oracle import pwn_oracle as O
    key = (id(s), Ti.tobytes(), m, robust, inner)
    if key not in _ORACLE_ITER:
        p = O.make_align_params(s.K, s.rows, s.cols, s.conf["minD"], s.conf["maxD"], s.cp, outer=1, inner=inner, guess=Ti,
                                max_chi2=m, robust=robust, num_threads=1)
        _ORACLE_ITER[key] = O.align(s.cloudA, s.cloudB, p, accumulate_f64=True)
    return _ORACLE_ITER[key]


def check_record(rec, o, m, robust, inner):
    """one teacher-forced iteration's record.  The record's inliers and error come from _computeStatistics at the pose
    AFTER the step, where the chi2 gap no longer separates the two sides' verdicts (their poses differ by ~1e-6):
    without the robust kernel a term within that distance of maxChi2 may fall on either side (at most 2, as in the
    teacher-forced sweep of test_gpu_parity.py; each moves the error by maxChi2).  With the robust kernel the error is
    continuous in chi2 and every term is an inlier."""
    from g2o_frontend_b200 import capi
    assert int(rec["status"]) == 0
    assert int(rec["num_correspondences"]) == o.numCorrespondences
    dinl = abs(int(rec["inliers"]) - o.inliers)
    assert dinl == 0 if robust else dinl <= 2, (int(rec["inliers"]), o.inliers)
    assert abs(float(rec["error"]) - o.error) <= H_RTOL * abs(o.error) + dinl * m, (float(rec["error"]), o.error)
    T = capi.from_colmajor(np.asarray(rec["T"], F), 4)
    assert rot_angle(T[:3, :3], o.T[:3, :3]) <= T_TOL
    assert np.abs(T[:3, 3] - o.T[:3, 3]).max() <= T_TOL


def as_record(res):
    from g2o_frontend_b200 import capi
    return np.frombuffer(C.string_at(C.addressof(res), C.sizeof(res)), capi.RESULT_DTYPE)[0]


@pytest.mark.gpu
@pytest.mark.parametrize("verify", [True, False])
@pytest.mark.parametrize("step,seed,dropout", [(4, 0, 0.05), (1, None, 0.0)])
def test_teacher_forced_iterations_with_the_chi2_cut(contexts, verify, step, seed, dropout):
    """one iteration restarted from the oracle's T at iterations 0, 3 and 9, with an inlierMaxChi2 near the median of the
    three iterations' chi2 taken together (it cuts at least a tenth of every iteration's terms), robust kernel off and on: as a single align (per-pair kernel, CUDA graph) with the iteration's correspondences
    bit-exact, its count and inliers exact, its H / b / error within 1e-4; and as one batch of the three pairs sharing
    the current cloud (grouped kernel).  inner = 3 runs MODE 1 over the stored correspondences."""
    from g2o_frontend_b200 import capi
    s, Ts, m = iteration_inputs(step, seed, dropout)
    c = s.conf
    single, batch = contexts[(verify, "per_pair")], contexts[(verify, "grouped")]
    refS, curS = upload(single, s.cloudA), upload(single, s.cloudB)
    refB, curB = upload(batch, s.cloudA), upload(batch, s.cloudB)
    for robust in (False, True):
        for inner in (1, 3):
            ap = gpu_align_params(c["inlierCurvatureRatioThreshold"], c["flatCurvatureThreshold"], m, robust, outer=1,
                                  inner=inner, dist=c["inlierDistanceThreshold"], normal=c["inlierNormalAngularThreshold"])
            oracle = [oracle_iteration(s, Ti, m, robust, inner) for Ti in Ts]
            for Ti, o in zip(Ts, oracle):
                res = single.align(refS, curS, s.projector(), ap, guess=Ti)
                check_record(as_record(res), o, m, robust, inner)
                st = single.align_state(s.rows, s.cols)
                assert np.array_equal(st["corr"], o.corr)
                if inner > 1:
                    continue
                tr = single.align_trace(1)
                assert int(tr[0, 60]) == o.trace_ncorr[0]
                assert int(tr[0, 59]) == o.trace_inliers[0]
                assert frob_rel(capi.from_colmajor(tr[0, 16:52], 6), o.trace_H[0]) <= H_RTOL
                assert frob_rel(tr[0, 52:58], o.trace_b[0]) <= H_RTOL
                assert abs(tr[0, 58] - o.trace_err[0]) <= H_RTOL * abs(o.trace_err[0])
                if not robust:  # the cut is engaged in every iteration
                    assert o.trace_inliers[0] <= 0.9 * o.trace_ncorr[0]
            recs = batch.align_batch([refB] * 3, [curB] * 3, s.projector(), ap, np.stack(Ts).astype(F))
            for rec, o in zip(recs, oracle):
                check_record(rec, o, m, robust, inner)


# ---- NICP_GROUP_MIN_AVG chooses the kernel and nothing else ----------------------------------------------------------
def knob_sequence(verify, avg):
    """every entry that stages pairs, each on clouds it sees first, in a context created with NICP_GROUP_MIN_AVG = avg;
    returns the bytes of every result"""
    from g2o_frontend_b200 import capi, synth
    with pytest.MonkeyPatch.context() as mp:
        mp.setenv("NICP_GROUP_MIN_AVG", avg)
        ctx = capi.Context(0, verify=verify)
    s, s2 = get_scene(4, 0, 0.05), get_scene(4, 1, 0.05)
    proj, ap = s.projector(), s.align_params(outer=3)
    rng = np.random.default_rng(5)
    guesses = np.stack([synth.perturbed_pose(rng, s.gt.astype(np.float64), 0.03, 2.0) for _ in range(3)]).astype(F)
    out = {}

    def fresh(oc, capacity=None):
        cl = ctx.new_cloud(max(capacity or oc.n, 1))
        cl.upload(oc.points, oc.normals, oc.curvature, oc.omegaP6(), oc.omegaN6())
        return cl

    out["single"] = bytes(as_record(ctx.align(fresh(s.cloudA), fresh(s.cloudB), proj, ap, guess=guesses[0])).tobytes())
    out["batch1"] = ctx.align_batch([fresh(s.cloudA)], [fresh(s.cloudB)], proj, ap, guesses[:1]).tobytes()
    A, B = fresh(s.cloudA), fresh(s.cloudB)
    out["batch2_shared"] = ctx.align_batch([A, fresh(s2.cloudA)], [B, B], proj, ap, guesses[:2]).tobytes()
    out["batch2_apart"] = ctx.align_batch([fresh(s.cloudA), fresh(s2.cloudA)], [fresh(s.cloudB), fresh(s2.cloudB)], proj,
                                          ap, guesses[:2]).tobytes()
    s0, ri, ci, invT, corr = stage_inputs(4, True)[:5]
    got = ctx.correspond_linearize(fresh(s0.cloudA), fresh(s0.cloudB), ri, ci, invT, s0.align_params())
    out["correspond_linearize"] = b"".join(np.asarray(v).tobytes() for v in got)
    got = ctx.linearize(fresh(s0.cloudA), fresh(s0.cloudB), corr, invT, s0.align_params())
    out["linearize"] = b"".join(np.asarray(v).tobytes() for v in got)
    # a batch packs the interleaved caches of its clouds; the reference is then uploaded anew and aligned alone
    A, B = fresh(s.cloudA, max(s.cloudA.n, s2.cloudA.n)), fresh(s.cloudB)
    out["stale_batch"] = ctx.align_batch([A] * 3, [B] * 3, proj, ap, guesses).tobytes()
    A.upload(s2.cloudA.points, s2.cloudA.normals, s2.cloudA.curvature, s2.cloudA.omegaP6(), s2.cloudA.omegaN6())
    out["stale_single"] = as_record(ctx.align(A, B, proj, ap, guess=guesses[1])).tobytes()
    ctx.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("verify", [True, False])
def test_group_min_avg_changes_no_result(verify):
    """NICP_GROUP_MIN_AVG = 0, 1, 2 against 1000 (never the grouped kernel): a single align, batches of 1 and 2 pairs,
    both stage entries, and an align after the reference cloud was re-uploaded, byte for byte"""
    want = knob_sequence(verify, "1000")
    for avg in ("0", "1", "2"):
        got = knob_sequence(verify, avg)
        for k in want:
            assert got[k] == want[k], (avg, k)

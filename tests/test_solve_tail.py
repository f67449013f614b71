"""The dense end of every alignment at the edges where the synthetic scenes of the other files never go: the Gauss-Newton
step of k_reduce_solve (solve_step in align.cu: damping, SE(3) priors, ldlt_solve6, the v2t / t2v pose update) and the
_computeStatistics tail (nicp_stats_tail.cuh: pseudo-inverse, float32 Cholesky, 13 sigma points, 6x6 inverse, eigen-ratios)
with both of its callers, the host (a single nicp_align finishes its record there) and k_statistics (a batch).

CPU: the tail through its host hook (nicp_statistics_tail_host) on hand-chosen H -- zero, weak and strong multiples of I, a
plane, pseudo-inverse threshold ties in the axis basis and a rotated one, inf / NaN entries, an indefinite H, translational-
or rotational-only degeneracy -- and ~2000 random symmetric H, each at poses that reach both branches of t2v and its
diagonal ties.  It must equal the oracle's _computeStatistics (orc_compute_statistics) bit for bit where finite and be NaN
at the same entries, every NaN being the quiet NaN 0x7fc00000; where the float64 restatement below is finite and not near
one of its edges (a sigma point at |q| = 1, an eigenvalue at the pseudo-inverse threshold, a quaternion sign flip) the
float32 tail is within a condition-scaled bar of it (OMEGA_RTOL, RATIO_RTOL below).

GPU: the device hook (nicp_statistics_tail, k_statistics) byte-identical to the host hook on the whole CPU set; and hand-built
pinhole pairs (no overlap, one point, one to three planes, a sphere; Omega_P = Omega_N = s I over nine decades of s; small
motions and rotations near and exactly at pi; relative and absolute priors, also without any correspondence), where every
traced Gauss-Newton step equals orc_gn_step bit for bit, the record's pose follows a float64 solve, the record's Omega and
ratios equal the oracle's tail at the final state and the host hook's bytes, the state's H follows the float64
linearisation, and the batched entries -- lone pairs (k_corr_lin_tiled) and pairs sharing a current cloud (k_corr_lin_group),
weak and strong pairs in one chunk -- give every pair the record of its single call, twice."""
import numpy as np
import pytest

from test_corr_lin_edges import iso_inverse

F = np.float32
EPS = float(np.finfo(F).eps)
QNAN = np.uint32(0x7FC00000)
# float32 tail against the float64 restatement: relative Frobenius norm of Omega, relative eigen-ratios.  The float32
# Cholesky of Sigma loses about cond(H + I) eps in its weak directions, which are Omega's strong ones, and the sigma points'
# differences lose a few eps of the pose against their spread.  Measured on the random set: below cond 100 at most 8.1e-5
# (Omega) and 8.9e-5 (ratios); above it at most 0.94 cond eps (Omega) and 0.91 cond eps (ratios), 1.32 cond eps for the
# ratios of the rotated threshold tie.  The bars leave a margin of 2 to 5x.  (The teacher-forced end-to-end bar of
# test_gpu_parity, on well-conditioned scenes, is 2e-3.)
OMEGA_RTOL, OMEGA_COND = 4e-4, 2.0
RATIO_RTOL, RATIO_COND = 4e-4, 3.0
EDGE = 1e-3          # relative distance from |q| = 1, from the pseudo-inverse threshold and of |q_w| from 0 that is excluded
LAMBDA = 1e-6 * 6    # alpha^2 * dim of unscented.h
H_RTOL = 1e-5        # the state's H against orc_linearize_f64
T_ROT_TOL = T_TRA_TOL = 1e-4   # test_gpu_parity's bar for a free-running alignment against orc_align


# ---- column-major helpers ----------------------------------------------------------------------------------------------
def cm(M):
    return np.ascontiguousarray(np.asarray(M, F).T).reshape(-1)


def unc(v, n):
    return np.asarray(v, F).reshape(n, n).T.copy()


def axis_rot(axis, angle):
    a = np.asarray(axis, np.float64)
    a = a / np.linalg.norm(a)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * K @ K


def pose(R=np.eye(3), t=(0, 0, 0)):
    T = np.eye(4)
    T[:3, :3] = R
    T[:3, 3] = t
    return T.astype(F)


# poses of the tail: identity, small, and rotations by pi (trace -1: t2v's else branch, with diagonal ties about x and z)
POSES = {
    "identity": np.eye(4, dtype=F),
    "small": pose(axis_rot((0.3, 1.0, 0.2), 0.05), (0.02, -0.01, 0.03)),
    "pi_x": pose(np.diag([1.0, -1.0, -1.0]), (0.1, 0.0, 0.0)),
    "pi_z": pose(np.diag([-1.0, -1.0, 1.0]), (0.0, 0.2, -0.1)),
    "pi_111": pose(axis_rot((1, 1, 1), np.pi), (0.0, 0.0, 0.5)),
}


def rand_rot(rng):
    Q, R = np.linalg.qr(rng.normal(size=(6, 6)))
    return Q * np.sign(np.diag(R))


def sym32(M):
    M = np.asarray(M, np.float64)
    return ((M + M.T) / 2).astype(F)


def handmade_H():
    """(name, H (6, 6) float32): the inputs where the tail turns NaN or sits on one of its edges"""
    rng = np.random.default_rng(7)
    out = [("zero", np.zeros((6, 6), F))]
    for s in (4, 5, 6, 10, 1e3, 1e8):
        out.append(("%g I" % s, (np.eye(6) * s).astype(F)))
    out.append(("plane", np.diag([0, 0, 1e8, 1e8, 1e8, 0]).astype(F)))
    Q = rand_rot(rng)
    for w in (94, 95, 96):  # H + I = diag(w + 1, 2^27, ...): the pseudo-inverse threshold 6 eps 2^27 is 96
        D = np.diag([w] + [2.0 ** 27] * 5)
        out.append(("tie w=%d" % w, D.astype(F)))
        out.append(("tie w=%d rotated" % w, sym32(Q @ D @ Q.T)))
    H = np.eye(6, dtype=F) * 1e3
    for name, (r, c, v) in {"inf diag": (2, 2, np.inf), "-inf diag": (4, 4, -np.inf), "inf off": (1, 3, np.inf),
                            "nan diag": (0, 0, np.nan), "nan off": (2, 5, np.nan)}.items():
        M = H.copy()
        M[r, c] = v
        M[c, r] = v
        out.append((name, M))
    for ev in (-0.5, -2.0):  # H + I positive / indefinite
        D = np.diag([ev, 10, 100, 1e3, 1e4, 1e5])
        out.append(("eigenvalue %g" % ev, sym32(Q @ D @ Q.T)))
    out.append(("translation only", np.diag([1e4, 2e4, 3e4, 0, 0, 0]).astype(F)))
    out.append(("rotation only", np.diag([0, 0, 0, 1e4, 2e4, 3e4]).astype(F)))
    out.append(("weak rotation", np.diag([1e4, 1e4, 1e4, 1e4, 1e4, 3]).astype(F)))
    return out


def random_H(n, seed=1):
    """n random symmetric H with eigenvalues log-uniform in a random sub-range of [1e-2, 1e10]"""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        lo, hi = np.sort(rng.uniform(-2, 10, size=2))
        ev = 10.0 ** rng.uniform(lo, hi, size=6)
        Q = rand_rot(rng)
        out.append(sym32(Q @ np.diag(ev) @ Q.T))
    return out


def tail_cases(n_random=2000):
    """(names, H (n, 36) column-major, T (n, 16) column-major): every hand-made H at every pose, the random H cycling
    through the poses"""
    names, Hs, Ts = [], [], []
    for name, H in handmade_H():
        for pn, T in POSES.items():
            names.append("%s @ %s" % (name, pn))
            Hs.append(cm(H))
            Ts.append(cm(T))
    pnames = list(POSES)
    for i, H in enumerate(random_H(n_random)):
        pn = pnames[i % len(pnames)]
        names.append("random %d @ %s" % (i, pn))
        Hs.append(cm(H))
        Ts.append(cm(POSES[pn]))
    return names, np.array(Hs, F), np.array(Ts, F)


_CASES = {}


def cases():
    if not _CASES:
        _CASES["all"] = tail_cases()
    return _CASES["all"]


# ---- float64 restatement of the tail (aligner.cpp:172-198, unscented.h:23-65) ---------------------------------------
def v2t64(v):
    qx, qy, qz = v[3:]
    qw = np.sqrt(1.0 - (qx * qx + qy * qy + qz * qz))
    T = np.eye(4)
    T[:3, :3] = [[qw * qw + qx * qx - qy * qy - qz * qz, 2 * (qx * qy - qw * qz), 2 * (qx * qz + qw * qy)],
                 [2 * (qx * qy + qz * qw), qw * qw - qx * qx + qy * qy - qz * qz, 2 * (qy * qz - qx * qw)],
                 [2 * (qx * qz - qy * qw), 2 * (qy * qz + qx * qw), qw * qw - qx * qx - qy * qy + qz * qz]]
    T[:3, 3] = v[:3]
    return T


def t2v64(T):
    """-> (v, |q_w| after normalisation): the sign rule of mat2quat flips at q_w = 0"""
    R = T[:3, :3]
    tr = np.trace(R)
    q = np.zeros(4)  # x y z w
    if tr > 0:
        t = np.sqrt(tr + 1)
        q[3] = 0.5 * t
        t = 0.5 / t
        q[:3] = [(R[2, 1] - R[1, 2]) * t, (R[0, 2] - R[2, 0]) * t, (R[1, 0] - R[0, 1]) * t]
    else:
        i = 0
        if R[1, 1] > R[0, 0]:
            i = 1
        if R[2, 2] > R[i, i]:
            i = 2
        j, k = (i + 1) % 3, (i + 2) % 3
        t = np.sqrt(R[i, i] - R[j, j] - R[k, k] + 1)
        q[i] = 0.5 * t
        t = 0.5 / t
        q[3] = (R[k, j] - R[j, k]) * t
        q[j] = (R[j, i] + R[i, j]) * t
        q[k] = (R[k, i] + R[i, k]) * t
    q /= np.linalg.norm(q)
    v = np.concatenate([T[:3, 3], -q[:3] if q[3] < 0 else q[:3]])
    return v, abs(q[3])


def tail_f64(H32, T32):
    """-> (Omega, tr, rr) in float64, or None where the float64 tail is not finite or the case sits within EDGE of an edge
    where float32 rounding decides the outcome"""
    A = H32.astype(np.float64) + np.eye(6)
    A = (A + A.T) / 2
    if not np.isfinite(A).all():
        return None
    w, V = np.linalg.eigh(A)
    thr = np.abs(w).max() * 6 * EPS
    if np.any(np.abs(np.abs(w) - thr) <= EDGE * thr):
        return None
    keep = np.abs(w) > thr
    if not keep.all() or (w <= 0).any():
        return None  # a dropped direction or a negative one: the Cholesky of Sigma does not exist
    Sigma = (V / w) @ V.T
    L = np.linalg.cholesky((6 + LAMBDA) * Sigma)
    samples = [np.zeros(6)] + [s * L[:, i] for i in range(6) for s in (1, -1)]
    T = T32.astype(np.float64)
    out = []
    for s in samples:
        qq = s[3:] @ s[3:]
        if qq >= 1 - EDGE:
            return None
        X = v2t64(s)
        v, qw = t2v64(T @ np.linalg.inv(X))
        if qw < EDGE:
            return None
        out.append(v)
    out = np.array(out)
    wm = np.full(13, 1 / (2 * (6 + LAMBDA)))
    wc = wm.copy()
    wm[0] = LAMBDA / (6 + LAMBDA)
    wc[0] = wm[0] + (1 - 1e-6 + 2)
    mean = wm @ out
    d = out - mean
    cov = (d.T * wc) @ d
    Om = np.linalg.inv(cov)

    def ratio(B):
        e = np.abs(np.linalg.eigvalsh((B + B.T) / 2))
        return e.max() / e.min()
    return Om, ratio(Om[:3, :3]), ratio(Om[3:, 3:])


# ---- comparisons -------------------------------------------------------------------------------------------------------
def same_or_both_nan(a, b):
    """bit-equal where a is finite, NaN where a is NaN (the oracle's NaN bits are x86's)"""
    a, b = np.asarray(a, F), np.asarray(b, F)
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint32), b[~nb].view(np.uint32)))


def oracle_tail(H36, T16):
    from oracle import pwn_oracle as O
    _, Om, tr, rr = O.compute_statistics(unc(H36, 6), unc(T16, 4))
    return cm(Om), np.array([tr, rr], F)


def frob_rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


# ---- CPU ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("verify", [False, True])
def test_host_tail_equals_oracle_bit_for_bit(verify):
    from g2o_frontend_b200 import capi
    names, H, T = cases()
    om, ra = capi.statistics_tail_host(H, T, verify)
    nan_cases = 0
    for i, name in enumerate(names):
        o_om, o_ra = oracle_tail(H[i], T[i])
        assert same_or_both_nan(om[i], o_om), (name, om[i], o_om)
        assert same_or_both_nan(ra[i], o_ra), (name, ra[i], o_ra)
        nan_cases += bool(np.isnan(om[i]).any())
    # every NaN the tail writes is the one quiet NaN
    for a in (om, ra):
        assert (a.view(np.uint32)[np.isnan(a)] == QNAN).all()
    # the table of the hand-made cases: which of them are NaN (T = I)
    want_nan = {"zero": True, "4 I": True, "5 I": True, "6 I": False, "10 I": False, "1000 I": False, "1e+08 I": False,
                "plane": True, "tie w=94": True, "tie w=95": True, "tie w=96": False}
    for name, nan in want_nan.items():
        i = names.index(name + " @ identity")
        assert bool(np.isnan(om[i]).all()) == nan and bool(np.isfinite(om[i]).all()) == (not nan), (name, om[i])
    assert 100 < nan_cases < len(names) - 1000, nan_cases


def test_nan_omega_reports_zero_ratios():
    """the current rule: a 3x3 block of Omega with a NaN has an eigen-ratio of 0 (every comparison with NaN is false), on
    the host and in the oracle alike -- so a `ratio > min` rejection test lets such a pair through"""
    from g2o_frontend_b200 import capi
    names, H, T = cases()
    om, ra = capi.statistics_tail_host(H, T)
    blocks = om.reshape(-1, 6, 6)  # [i, col, row]
    tnan = np.isnan(blocks[:, :3, :3]).any(axis=(1, 2))
    rnan = np.isnan(blocks[:, 3:, 3:]).any(axis=(1, 2))
    assert tnan.sum() > 100 and rnan.sum() > 100
    assert (ra[tnan, 0] == 0).all() and (ra[rnan, 1] == 0).all()
    i = names.index("zero @ identity")
    o_om, o_ra = oracle_tail(H[i], T[i])
    assert np.isnan(o_om).all() and (o_ra == 0).all() and (ra[i] == 0).all()


def test_tail_against_float64():
    from g2o_frontend_b200 import capi
    names, H, T = cases()
    om, ra = capi.statistics_tail_host(H, T)
    worst_om = worst_ra = 0.0
    compared = compared_random = 0
    for i, name in enumerate(names):
        ref = tail_f64(unc(H[i], 6), unc(T[i], 4))
        if ref is None:
            continue
        Om64, tr64, rr64 = ref
        assert np.isfinite(om[i]).all(), name
        ce = np.linalg.cond(unc(H[i], 6).astype(np.float64) + np.eye(6)) * EPS
        e = frob_rel(unc(om[i], 6), Om64)
        r = max(abs(ra[i, 0] - tr64) / tr64, abs(ra[i, 1] - rr64) / rr64)
        assert e <= OMEGA_RTOL + OMEGA_COND * ce, (name, e, ce)
        assert r <= RATIO_RTOL + RATIO_COND * ce, (name, r, ce, ra[i], tr64, rr64)
        compared += 1
        if name.startswith("random"):
            compared_random += 1
            worst_om, worst_ra = max(worst_om, e / (OMEGA_RTOL + OMEGA_COND * ce)), max(worst_ra, r / (RATIO_RTOL + RATIO_COND * ce))
    print("float32 tail vs float64: %d cases (%d random), worst Omega error / bar %.2f, worst ratio error / bar %.2f" %
          (compared, compared_random, worst_om, worst_ra))
    assert compared_random >= 500, compared_random


def test_gn_step_oracle_matches_align():
    """orc_gn_step is orc_align's step: chaining it over orc_align's own trace gives orc_align's poses bit for bit"""
    from conftest import get_scene
    from oracle import pwn_oracle as O
    s = get_scene(4)
    out = O.align(s.cloudA, s.cloudB, s.oracle_align_params(outer=4, num_threads=1))
    for i in range(4):
        Tn = O.gn_step(out.trace_H[i], out.trace_b[i], out.trace_T[i])
        want = out.trace_T[i + 1] if i < 3 else out.T
        assert np.array_equal(Tn.view(np.uint32), want.view(np.uint32)), i


# ---- GPU: the device tail ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", params=["verify", "default"])
def verify(request):
    return request.param == "verify"


@pytest.fixture(scope="module")
def ctx(verify):
    from g2o_frontend_b200 import capi
    c = capi.Context(0, verify=verify)
    yield c
    c.close()


@pytest.mark.gpu
def test_device_tail_equals_host_tail_bytes(ctx, verify):
    """k_statistics (a batch's records) and the host function (a single alignment's record) write the same bytes, NaNs
    included"""
    from g2o_frontend_b200 import capi
    names, H, T = cases()
    om_h, ra_h = capi.statistics_tail_host(H, T, verify)
    om_d, ra_d = ctx.statistics_tail(H, T)
    bad = [names[i] for i in range(len(names))
           if om_d[i].tobytes() != om_h[i].tobytes() or ra_d[i].tobytes() != ra_h[i].tobytes()]
    assert not bad, (len(bad), bad[:10])
    # a second, smaller call reuses the slots
    om2, ra2 = ctx.statistics_tail(H[:7], T[:7])
    assert om2.tobytes() == om_h[:7].tobytes() and ra2.tobytes() == ra_h[:7].tobytes()


# ---- GPU: hand-built pairs -------------------------------------------------------------------------------------------------
ROWS, COLS = 48, 64
KMAT = np.array([[50.0, 0, 32.0], [0, 50.0, 24.0], [0, 0, 1]], F)
MIN_D, MAX_D = 0.1, 10.0
PLANES = {  # (unit normal facing the camera, d) with n . p = d
    "back": (np.array([0.05, -0.1, -1.0]), -3.0),
    "floor": (np.array([0.0, -1.0, 0.0]), -1.0),
    "left": (np.array([1.0, 0.0, 0.0]), -1.2),
}
GEOMETRIES = ("none", "point", "plane", "two_planes", "three_planes", "sphere")
SCALES = (1e-3, 1.0, 1e3, 1e6)


def render(geometry):
    """points (n, 4) and normals (n, 4) of the current frame: one point per pixel, off the pixel boundaries"""
    v, u = np.mgrid[0:ROWS, 0:COLS]
    rays = np.stack([(u + 0.3 - KMAT[0, 2]) / KMAT[0, 0], (v + 0.3 - KMAT[1, 2]) / KMAT[1, 1], np.ones_like(u, float)], -1)
    rays = rays.reshape(-1, 3)
    best_t = np.full(len(rays), np.inf)
    best_n = np.zeros((len(rays), 3))
    planes = {"none": ["back"], "point": ["back"], "plane": ["back"], "two_planes": ["back", "floor"],
              "three_planes": ["back", "floor", "left"], "sphere": []}[geometry]
    for p in planes:
        n, d = PLANES[p]
        n = n / np.linalg.norm(n)
        den = rays @ n
        t = np.where(den < -1e-6, (d / np.linalg.norm(PLANES[p][0])) / np.where(den == 0, 1, den), np.inf)
        t = np.where(t > 0, t, np.inf)
        m = t < best_t
        best_t[m], best_n[m] = t[m], n
    if geometry == "sphere":
        c, r = np.array([0.1, 0.0, 2.5]), 0.9
        b = rays @ c
        a = (rays * rays).sum(1)
        disc = b * b - a * (c @ c - r * r)
        t = np.where(disc > 0, (b - np.sqrt(np.maximum(disc, 0))) / a, np.inf)
        best_t = t
        p = rays * t[:, None]
        best_n = np.where(np.isfinite(t)[:, None], (p - c) / r, 0)
    ok = np.isfinite(best_t)
    P = rays[ok] * best_t[ok, None]
    N = best_n[ok]
    if geometry == "point":
        k = len(P) // 2 + COLS // 2
        P, N = P[k:k + 1], N[k:k + 1]
    pts = np.concatenate([P, np.ones((len(P), 1))], 1).astype(F)
    nrm = np.concatenate([N, np.zeros((len(N), 1))], 1).astype(F)
    return pts, nrm


MOTIONS = {
    "small": (pose(axis_rot((0.3, 1.0, 0.2), 0.03), (0.03, -0.02, 0.04)), None),  # (T_true, guess = T_true * this)
    # near and exactly at pi: the alignment starts next to the truth, so t2v of every step takes its else branch
    "near_pi": (pose(axis_rot((0.2, 1.0, 0.1), np.pi - 1e-3), (0.05, 0.0, 0.1)),
                pose(axis_rot((0.0, 1.0, 0.0), 0.01), (0.01, 0.0, 0.0))),
    "pi": (pose(np.diag([-1.0, 1.0, -1.0]), (0.05, 0.0, 0.1)), pose(axis_rot((1.0, 0.0, 0.0), 0.01), (0.0, 0.01, 0.0))),
}


class Pair:
    def __init__(self, geometry, scale, motion):
        self.name = "%s s=%g %s" % (geometry, scale, motion)
        self.geometry, self.scale = geometry, scale
        Ttrue, pert = MOTIONS[motion]
        cur_p, cur_n = render(geometry)
        M = Ttrue.astype(np.float64)  # the reference seen from the current frame's camera at T_true
        if geometry == "none":
            M[:3, 3] += (100.0, 0.0, 0.0)  # the reference never projects into the image
        ref_p = (cur_p.astype(np.float64) @ M.T).astype(F)
        ref_n = (cur_n.astype(np.float64) @ M.T).astype(F)
        if geometry == "point":  # one point: its correspondence exists only at the true pose
            self.guess = Ttrue.copy()
        else:
            self.guess = np.eye(4, dtype=F) if pert is None else (Ttrue.astype(np.float64) @ pert).astype(F)
        self.ref = (ref_p, ref_n)
        self.cur = (cur_p, cur_n)

    def om6(self, n):
        o = np.zeros((n, 6), F)
        o[:, [0, 3, 5]] = self.scale
        return o

    def upload(self, ctx, which):
        p, n = getattr(self, which)
        cl = ctx.new_cloud(max(len(p), 1))
        cl.upload(p, n, np.zeros(len(p), F), self.om6(len(p)), self.om6(len(p)))
        return cl

    def oracle_cloud(self, which):
        from oracle import pwn_oracle as O
        p, n = getattr(self, which)
        c = O.Cloud(len(p))
        c.points[:], c.normals[:] = p, n
        om = np.zeros((len(p), 16), F)
        om[:, [0, 5, 10]] = self.scale
        c.omegaP[:], c.omegaN[:] = om, om
        return c


def pair_list():
    out = []
    for g in GEOMETRIES:
        for s in SCALES:
            out.append(Pair(g, s, "small"))
    for g in ("plane", "three_planes", "sphere"):
        for s in (1.0, 1e6):
            for m in ("near_pi", "pi"):
                out.append(Pair(g, s, m))
    return out


PRIOR_INFOS = (1e-6, 1.0, 1e8)


def priors_for(pair, kind, info):
    """(device priors, oracle priors): a prior towards the guess perturbed by a small motion"""
    from g2o_frontend_b200 import capi
    from oracle import pwn_oracle as O
    mean = (pair.guess.astype(np.float64) @ pose(axis_rot((1, 0, 0), 0.02), (0.01, 0.0, 0.0))).astype(F)
    ref = pose(axis_rot((0, 0, 1), 0.3), (0.2, -0.1, 0.0))
    I6 = (np.eye(6) * info).astype(F)
    dp = capi.make_prior(kind, mean, I6, ref if kind == 1 else None)
    op = O.make_prior(kind, mean, I6)
    op.refInv[:] = cm(iso_inverse(ref) if kind == 1 else np.eye(4)).tolist()
    return [dp], [op]


def prior_cases(pairs):
    out = []
    for p in pairs:
        if p.name in ("none s=1 small", "plane s=1 small", "three_planes s=1000 small", "plane s=1e+06 pi"):
            for kind in (0, 1):
                for info in PRIOR_INFOS:
                    out.append((p, kind, info))
    return out


_PAIRS = {}


def pairs():
    if not _PAIRS:
        _PAIRS["p"] = pair_list()
    return _PAIRS["p"]


def projector():
    from g2o_frontend_b200 import capi
    return capi.make_projector(KMAT, ROWS, COLS, MIN_D, MAX_D)


def align_params(outer, inner):
    from g2o_frontend_b200 import capi
    return capi.make_align_params(0.5, 0.95, 0.02, 1.3, 9e3, True, outer, inner)


def record_bytes(res):
    import ctypes as C
    return C.string_at(C.addressof(res), C.sizeof(res))


def f64_step(H, b, T):
    """(H + 1001 I) dx = -b in float64, composed as the aligner composes it: T' = (v2t(dx) T^-1)^-1.  -> (T', the bar)
    The bar: the solve's cond(H + 1001 I) eps |dx|, a few eps of the pose, and what the aligner's float32 t2v / v2t round
    trip of T' loses when q_w is small (a rotation near pi): v2t recomputes q_w from 1 - |q|^2."""
    Hd = H.astype(np.float64) + 1001.0 * np.eye(6)
    dx = np.linalg.solve(Hd, -b.astype(np.float64))
    Tn = np.linalg.inv(v2t64(dx) @ np.linalg.inv(T.astype(np.float64)))
    qw = t2v64(Tn)[1]
    bar = 1e-5 + 16 * EPS * np.linalg.cond(Hd) * max(float(np.abs(dx).max()), 1e-3) + 4 * (np.sqrt(qw * qw + 4 * EPS) - qw)
    return Tn, bar


def check_single(ctx, verify, pair, outer, prior=None):
    """one nicp_align of the pair: the step, the pose, the record and the state; returns the record's bytes"""
    from g2o_frontend_b200 import capi
    from oracle import pwn_oracle as O
    ref, cur = pair.upload(ctx, "ref"), pair.upload(ctx, "cur")
    dpri, opri = priors_for(pair, *prior) if prior else ((), ())
    res = ctx.align(ref, cur, projector(), align_params(outer, 1), guess=pair.guess, priors=list(dpri))
    tr = ctx.align_trace(outer)
    Ts = [unc(tr[i, :16], 4) for i in range(outer)] + [capi.result_T(res)]
    assert np.array_equal(Ts[0].view(np.uint32), pair.guess.view(np.uint32)), pair.name
    for i in range(outer):
        Hi, bi = unc(tr[i, 16:52], 6), tr[i, 52:58].copy()
        Tn = O.gn_step(Hi, bi, Ts[i], list(opri))
        # (a lost pose is NaN with the device's bits on one side and x86's on the other)
        assert same_or_both_nan(Tn, Ts[i + 1]), (pair.name, prior, outer, i, Tn, Ts[i + 1])
        if np.isnan(Ts[i + 1]).any():
            # exactly at pi the float32 t2v / v2t round trip of the step can take sqrt of a negative 1 - |q|^2 (the
            # reference's own arithmetic, the oracle's too): the pose is lost, only next to q_w = 0
            assert t2v64(f64_step(Hi, bi, Ts[i])[0])[1] < 1e-3, (pair.name, i)
            break
        if not prior:
            T64, bar = f64_step(Hi, bi, Ts[i])
            assert np.abs(Ts[i + 1] - T64).max() <= bar, (pair.name, i, np.abs(Ts[i + 1] - T64).max(), bar)
    st = ctx.align_state(ROWS, COLS)
    T = capi.result_T(res)
    # the record's tail: the oracle's at the state's H and the record's T, and the host hook's bytes
    o_om, o_ra = oracle_tail(cm(st["H"]), cm(T))
    assert same_or_both_nan(np.array(res.omega[:], F), o_om), pair.name
    assert same_or_both_nan(np.array([res.translational_eigen_ratio, res.rotational_eigen_ratio], F), o_ra), pair.name
    h_om, h_ra = capi.statistics_tail_host(cm(st["H"]), cm(T), verify)
    assert np.array(res.omega[:], F).tobytes() == h_om[0].tobytes(), pair.name
    assert np.array([res.translational_eigen_ratio, res.rotational_eigen_ratio], F).tobytes() == h_ra[0].tobytes()
    # the state's H: the linearisation at the final T over the state's correspondences
    if res.num_correspondences > 0:
        invT = iso_inverse(T)
        H64, b64, _, inl64 = O.linearize_f64(st["corr"], pair.oracle_cloud("ref"), pair.oracle_cloud("cur"), invT, 9e3, True)
        assert frob_rel(st["H"], H64) <= H_RTOL, (pair.name, frob_rel(st["H"], H64))
    else:
        assert not st["H"].any() and res.inliers == 0 and np.isnan(res.omega[:]).all()
    ref.close()
    cur.close()
    return record_bytes(res)


@pytest.mark.gpu
@pytest.mark.parametrize("outer", [1, 10])
def test_single_alignment_step_pose_and_record(ctx, verify, outer):
    weak = 0
    for p in pairs():
        check_single(ctx, verify, p, outer)
    for p, kind, info in prior_cases(pairs()):
        check_single(ctx, verify, p, outer, (kind, info))
    # the set reaches the NaN tail and the finite one
    from g2o_frontend_b200 import capi
    for p in pairs():
        ref, cur = p.upload(ctx, "ref"), p.upload(ctx, "cur")
        res = ctx.align(ref, cur, projector(), align_params(outer, 1), guess=p.guess)
        weak += bool(np.isnan(res.omega[:]).any())
    assert 3 <= weak <= len(pairs()) - 3, weak


@pytest.mark.gpu
def test_inner_iterations_follow_oracle_align(ctx):
    from g2o_frontend_b200 import capi
    from oracle import pwn_oracle as O
    cp = O.default_corr_params(inlierDistanceThreshold=0.5, inlierNormalAngularThreshold=0.95)
    checked = 0
    for p in pairs():
        if p.geometry in ("none", "point"):
            continue
        ref, cur = p.upload(ctx, "ref"), p.upload(ctx, "cur")
        res = ctx.align(ref, cur, projector(), align_params(4, 3), guess=p.guess)
        out = O.align(p.oracle_cloud("ref"), p.oracle_cloud("cur"),
                      O.make_align_params(KMAT, ROWS, COLS, MIN_D, MAX_D, cp, outer=4, inner=3, guess=p.guess, num_threads=1))
        T = capi.result_T(res)
        if np.isnan(out.T).any():  # a pose lost exactly at pi (test_single_alignment_step_pose_and_record) is lost on both
            assert np.array_equal(np.isnan(T), np.isnan(out.T)), p.name
            continue
        R = T[:3, :3].astype(np.float64).T @ out.T[:3, :3].astype(np.float64)
        ang = np.linalg.norm([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]]) / 2
        assert ang <= T_ROT_TOL and np.abs(T[:3, 3] - out.T[:3, 3]).max() <= T_TRA_TOL, (p.name, ang)
        checked += 1
    assert checked >= 20


@pytest.mark.gpu
def test_batches_equal_single_calls(ctx, verify):
    """every record of nicp_align_batch / _batch_priors equals its single call byte for byte: lone pairs (tiled kernel),
    pairs sharing a current cloud in groups of 3 and 4 (grouped kernel), weak and strong pairs mixed in one chunk; twice"""
    from g2o_frontend_b200 import capi
    ps = pairs()
    ap = align_params(10, 1)
    refs = [p.upload(ctx, "ref") for p in ps]
    curs = [p.upload(ctx, "cur") for p in ps]
    singles = [record_bytes(ctx.align(refs[i], curs[i], projector(), ap, guess=p.guess)) for i, p in enumerate(ps)]
    guesses = np.array([p.guess for p in ps])
    # lone pairs: every pair has its own current cloud
    for _ in range(2):
        recs = ctx.align_batch(refs, curs, projector(), ap, guesses=guesses)
        for i, p in enumerate(ps):
            assert recs[i].tobytes() == singles[i], (p.name, recs[i], np.frombuffer(singles[i], capi.RESULT_DTYPE))
    # with priors (some pairs without any)
    pc = prior_cases(ps)
    idx = [ps.index(p) for p, _, _ in pc]
    pri = [priors_for(p, k, info)[0] for p, k, info in pc]
    want = []
    for j, (p, k, info) in enumerate(pc):
        want.append(record_bytes(ctx.align(refs[idx[j]], curs[idx[j]], projector(), ap, guess=p.guess, priors=pri[j])))
    sel_r, sel_c = [refs[i] for i in idx] + refs[:3], [curs[i] for i in idx] + curs[:3]
    g = np.concatenate([guesses[idx], guesses[:3]])
    for _ in range(2):
        recs = ctx.align_batch(sel_r, sel_c, projector(), ap, guesses=g, priors=pri + [[], [], []])
        for j in range(len(pc)):
            assert recs[j].tobytes() == want[j], pc[j][0].name
        for j in range(3):
            assert recs[len(pc) + j].tobytes() == singles[j]
    # groups sharing a current cloud: the pairs of one geometry / motion over all scales share the cloud of the first
    # (same points and normals; the current cloud's Omega is the first pair's)
    groups = {}
    for i, p in enumerate(ps):
        groups.setdefault((p.geometry, p.name.split()[-1]), []).append(i)
    order, shared = [], []
    for key, members in groups.items():
        if len(members) >= 3:
            for i in members:
                order.append(i)
                shared.append(curs[members[0]])
    assert len(order) >= 20
    want = [record_bytes(ctx.align(refs[i], shared[k], projector(), ap, guess=ps[i].guess)) for k, i in enumerate(order)]
    for _ in range(2):
        recs = ctx.align_batch([refs[i] for i in order], shared, projector(), ap, guesses=guesses[order])
        for k, i in enumerate(order):
            assert recs[k].tobytes() == want[k], ps[i].name
    for c in refs + curs:
        c.close()

"""Sensor-model gaussians and local maps for MultiPointProjector rigs (nicp_multi_cloud_compute_gaussians,
nicp_multi_raw_depth_to_local_map).

The definition of a rig point's gaussian (DESIGN.md, known deviations) is restated here by oracle_rig_gaussians from the
oracle's own pieces: orc_multi_unproject for the points and their order, orc_unproject_gaussians on each camera's own image
for the sensor model, a float32 rotation in the rounding order of orc_gaussians_transform, then orc_gaussians_transform for
the rig's sensor offset.  CPU part: that restatement against the pinhole oracle and a float64 restatement, and the entries'
answers to null handles.  GPU part (-m gpu, both library builds): the single-frame
gaussians bit for bit against the oracle, the local-map entry against the chain of single calls it replaces byte for byte,
end to end against the oracle, and through the pwn:: C++ layer.
"""
import ctypes as C
import os
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest

from conftest import ROOT
from g2o_frontend_b200 import capi, synth
from test_rig_batch import composite, make_cams, render_raw_frame, rig_poses

DEPTH_SCALE, MAX_DEPTH_COV = 0.001, 0.01
# per-camera sensor models that differ between cameras (PinholePointProjector defaults: 0.075, 0.1)
BASELINES = [0.075, 0.05, 0.12, 0.09]
ALPHAS = [0.1, 0.2, 0.05, 0.15]


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _models(cams):
    n = len(cams)
    return np.array(BASELINES[:n], np.float32), np.array(ALPHAS[:n], np.float32)


def _offset():
    return synth.make_pose((0.05, 0.0, 0.1), (1.0, 0.2, 0.0), 3.0).astype(np.float32)


def _sp():
    return capi.make_stats_params(0.1, 3, 6, 10, 0.2, 0.02)


def _oracle_composite(frame, cams, step):
    """the composite depth image of one raw rig frame, converted and scaled by the oracle"""
    from oracle import pwn_oracle as O
    rows, cols = max(c["width"] for c in cams), sum(c["height"] for c in cams)
    out = np.zeros((rows, cols), np.float32)
    off = 0
    for r, c in zip(frame, cams):
        d = O.depth_u16_to_f32(r, DEPTH_SCALE)
        if step > 1:
            d = O.depth_scale(d, step, MAX_DEPTH_COV)
        out[:c["width"], off:off + c["height"]] = d.T
        off += c["height"]
    return out


def _dot3(a0, a1, a2, b0, b1, b2):
    """float32 (a0 b0 + a1 b1) + a2 b2, every operation rounded (dot3 of the oracle and of the device)"""
    return (a0 * b0 + a1 * b1) + a2 * b2


def _rotate_cov(R, cov):
    """(R cov) R^T of n column-major 3x3 float32 covariances in the order of orc_gaussians_transform (mat3_mulf, then
    mat3_mul_bt)"""
    C3 = cov.reshape(-1, 3, 3).transpose(0, 2, 1)  # C3[:, r, c]
    RC = np.empty_like(C3)
    for r in range(3):
        for c in range(3):
            RC[:, r, c] = _dot3(R[r, 0], R[r, 1], R[r, 2], C3[:, 0, c], C3[:, 1, c], C3[:, 2, c])
    out = np.empty_like(C3)
    for r in range(3):
        for c in range(3):
            out[:, r, c] = _dot3(RC[:, r, 0], RC[:, r, 1], RC[:, r, 2], R[c, 0], R[c, 1], R[c, 2])
    return np.ascontiguousarray(out.transpose(0, 2, 1)).reshape(-1, 9)


def oracle_rig_gaussians(cams, depth, baseline, alpha, sensor_offset=None):
    """the gaussians of a rig cloud by their definition: for a point of camera i at composite pixel (r, c), depth z,
      1. child i's sensor model (pinholepointprojector.cpp:93-133, orc_unproject_gaussians) at x = r, y = v = c - colOff_i:
         orc_unproject_gaussians on the camera's own image (its column block transposed), baseline[i], alpha[i];
      2. mean = the rig point of orc_multi_unproject; covariance R_i cov R_i^T with R_i the rotation of offset_i, skipped
         when offset_i is exactly the identity (as orc_gaussians_transform skips one);
      3. the rig's sensor offset by orc_gaussians_transform.
    Points in the order of orc_multi_unproject (camera by camera, raster order inside the camera's block).  Returns
    (gauss (n,24), flags (n,), points (n,4) before the sensor offset, index image)."""
    from oracle import pwn_oracle as O
    depth = np.ascontiguousarray(depth, np.float32)
    rows, cols = depth.shape
    m = O.make_multi(cams)
    pts = np.zeros((rows * cols, 4), np.float32)
    idx = np.zeros((rows, cols), np.int32)
    eye = capi.colmajor(np.eye(4))
    fp = lambda x: x.ctypes.data_as(C.POINTER(C.c_float))
    n = O.lib().orc_multi_unproject(C.byref(m), fp(eye), fp(depth), rows, cols, fp(pts), idx.ctypes.data_as(C.POINTER(C.c_int)))
    g = np.zeros((n, O.GAUSS_FLOATS), np.float32)
    f = np.full(n, O.GAUSS_MOMENTS, np.int32)
    g[:, :3] = pts[:n, :3]
    off = 0
    for i, c in enumerate(cams):
        w, h = c["width"], c["height"]
        own = np.ascontiguousarray(depth[:w, off:off + h].T)  # camera i's image: row = pixel v, column = pixel u
        gp, _, _, idxp = O.unproject_gaussians(own, c["K"], c["minD"], c["maxD"], float(np.float32(baseline[i])),
                                               float(np.float32(alpha[i])))
        block = idx[:w, off:off + h]
        valid = block >= 0
        assert np.array_equal(valid, idxp.T >= 0)
        cov = gp[idxp.T[valid], 3:12]
        M = np.asarray(c["offset"], np.float32).copy()
        M[3] = (0, 0, 0, 1)
        if not np.array_equal(M, np.eye(4, dtype=np.float32)):
            cov = _rotate_cov(M[:3, :3], cov)
        g[block[valid], 3:12] = cov
        off += h
    if sensor_offset is not None:
        g, f = O.gaussians_transform(sensor_offset, g, f)
    return g, f, pts[:n], idx


def _merge_view(cams):
    """the pinhole view rig maps are merged through: camera 0's intrinsics and image"""
    c = cams[0]
    return capi.make_projector(c["K"], c["height"], c["width"], c["minD"], c["maxD"])


# ================================================================================================
# CPU: the oracle's definition
# ================================================================================================
def test_one_camera_rig_equals_pinhole_oracle():
    """a one-camera rig at an identity offset: the gaussians of orc_unproject_gaussians on the transposed composite (the
    camera's own image), as a permutation of the points"""
    from oracle import pwn_oracle as O
    cams = make_cams("4cam")[:1]
    cams[0]["offset"] = np.eye(4, dtype=np.float32)
    frame = render_raw_frame(rig_poses(1, 5)[0], cams, 1, 40)
    d = _oracle_composite(frame, cams, 1)
    g, f, p, idx = oracle_rig_gaussians(cams, d, [0.09], [0.15])
    gp, fp_, pp, idxp = O.unproject_gaussians(np.ascontiguousarray(d.T), cams[0]["K"], cams[0]["minD"], cams[0]["maxD"], 0.09,
                                              0.15)
    assert g.shape[0] == gp.shape[0] > 0.3 * d.size
    valid = idx >= 0
    assert np.array_equal(valid, idxp.T >= 0)
    perm = idxp.T[valid]          # pinhole index of the rig's point idx[valid]
    order = idx[valid]
    assert np.array_equal(_bits(g[order]), _bits(gp[perm]))
    assert np.array_equal(f[order], fp_[perm])


@pytest.mark.parametrize("kind", ["4cam", "ragged"])
def test_rig_gaussian_definition(kind):
    """on both test rigs: means bit-identical to the rig points of orc_multi_unproject, covariances R_i Sigma_cam R_i^T of
    a float64 restatement to 1e-6 relative, with per-camera baseline / alpha"""
    from oracle import pwn_oracle as O
    cams = make_cams(kind)
    b, a = _models(cams)
    d = _oracle_composite(render_raw_frame(rig_poses(1, 7)[0], cams, 1, 60), cams, 1)
    m = O.make_multi(cams)
    g, f, p, idx = oracle_rig_gaussians(cams, d, b, a)
    cl, idx2 = O.multi_depth_to_cloud(m, d, O.default_stats_params(minImageRadius=3, maxImageRadius=6, minPoints=10))
    assert np.array_equal(idx, idx2) and g.shape[0] == cl.n > 0.3 * d.size
    assert np.array_equal(_bits(g[:, :3]), _bits(cl.points[:, :3])) and np.all(f == O.GAUSS_MOMENTS)
    assert not g[:, 12:].any()
    # the float32 rotation of the restatement is bit for bit the covariance part of orc_gaussians_transform
    R = np.asarray(cams[1]["offset"], np.float32)[:3, :3]
    Tr = np.eye(4, dtype=np.float32)
    Tr[:3, :3] = R
    gt, _ = O.gaussians_transform(Tr, g, f)
    assert np.array_equal(_bits(gt[:, 3:12]), _bits(_rotate_cov(R, g[:, 3:12])))
    off = 0
    rng = np.random.default_rng(1)
    for i, c in enumerate(cams):
        iK = np.linalg.inv(np.asarray(c["K"], np.float64))
        R = np.asarray(c["offset"], np.float64)[:3, :3]
        fB, ai = float(np.float32(b[i]) * np.float32(c["K"][0][0])), float(a[i])
        block = idx[:c["width"], off:off + c["height"]]
        pix = np.argwhere(block >= 0)
        for r, v in pix[rng.integers(0, len(pix), 40)]:
            z = float(d[r, off + v])
            J = iK @ np.array([[z, 0, r], [0, z, v], [0, 0, 1.0]])
            S = J @ np.diag([3.0, 3.0, ai * z * z / (fB + ai * z)]) @ J.T
            want = R @ S @ R.T
            got = g[block[r, v], 3:12].reshape(3, 3).T.astype(np.float64)
            assert np.abs(got - want).max() <= 1e-6 * np.abs(want).max()
        off += c["height"]


@pytest.mark.parametrize("verify", [False, True])
def test_null_handles_without_device(verify):
    """both entries answer null handles with NICP_ERR_INVALID before touching a device (no GPU needed)"""
    L = capi.load(verify)
    N, f0 = None, C.c_float(0)
    assert L.nicp_multi_cloud_compute_gaussians(N, N, N, N, N, N, N) == 1
    assert L.nicp_multi_raw_depth_to_local_map(N, 2, N, N, N, C.c_float(0.001), 1, C.c_float(0.01), N, N, N, N, N, N, N, N,
                                               N, f0, N, N, N, N, N) == 1


# ================================================================================================
# GPU
# ================================================================================================
@pytest.fixture(scope="module", params=["verify", "default"])
def ctx(request):
    c = capi.Context(0, verify=(request.param == "verify"))
    yield c
    c.close()


_FRAMES = {}


def _frames(kind, n, step):
    """the first n of up to 17 raw frames of a test rig (or "config5": synth.make_rig(4, 1280, 960) as the sensor
    delivers it), the rig after scaling and the frames' poses"""
    key = (kind, step)
    if kind == "config5":
        cams = synth.make_rig(4, 1280 // step, 960 // step, K=synth.scaled_K(synth.K_KINECT, 2.0 / step))
        count = 3
    else:
        cams = make_cams(kind)
        count = 17
    if key not in _FRAMES:
        poses = [p.astype(np.float32) for p in rig_poses(count, 11)]
        _FRAMES[key] = ([render_raw_frame(p, cams, step, 70 + 5 * f) for f, p in enumerate(poses)], poses)
    frames, poses = _FRAMES[key]
    assert n <= len(frames)
    return cams, frames[:n], poses[:n]


def _chain(ctx, cams, frames, poses, step, so, map_cloud, merge=None, mT=None, vres=0.0):
    """the calls the entry replaces, one frame at a time -> (collapsed or None, representatives or None)"""
    mp = capi.make_multi_projector(cams)
    b, a = _models(cams)
    for fr, T in zip(frames, poses):
        fc = ctx.multi_raw_depth_to_cloud_batch([fr], mp, _sp(), step=step, sensor_offset=so)[0]
        fc.multi_compute_gaussians(composite(ctx, fr, cams, step), mp, b, a, so)
        map_cloud.append(fc, T)
        fc.close()
    col = rep = None
    if merge is not None:
        _, col = map_cloud.merge(_merge_view(cams), mT, merge)
    if vres > 0:
        _, rep = map_cloud.voxelize(vres)
    return col, rep


def _entry(ctx, cams, frames, poses, step, so, map_cloud, merge=None, mT=None, vres=0.0):
    b, a = _models(cams)
    return ctx.multi_raw_depth_to_local_map(frames, capi.make_multi_projector(cams), _sp(), poses, map_cloud, step=step,
                                            sensor_offset=so, baseline=b, alpha=a,
                                            merge_proj=_merge_view(cams) if merge is not None else None,
                                            merge_params=merge, merge_transform=mT, voxel_resolution=vres)


def _snapshot(cl):
    d = cl.download()
    out = {"size": cl.size(), "points": _bits(d["points"]), "normals": _bits(d["normals"]), "curvature": _bits(d["curvature"]),
           "omega_p": _bits(d["omega_p"]), "omega_n": _bits(d["omega_n"]), "has_gauss": cl.has_gaussians()}
    if cl.has_gaussians():
        g, f = cl.download_gaussians()
        out["gauss"], out["gflags"] = _bits(g), f
    return out


def _assert_same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def _merge_args(merge, poses):
    if merge is None:
        return None, None
    if merge == "identity":
        return capi.make_merge_params(), np.eye(4, dtype=np.float32)
    return capi.make_merge_params(0.05, 0.99, 3.0), poses[len(poses) // 2]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,step,offset", [("4cam", 1, False), ("4cam", 2, True), ("ragged", 1, True),
                                              ("ragged", 2, False)])
def test_rig_gaussians_match_oracle(ctx, kind, step, offset):
    """nicp_multi_cloud_compute_gaussians on a rig cloud: every float and flag bit-exact against
    oracle_rig_gaussians with the sensor offset; a depth image of another frame is rejected"""
    from oracle import pwn_oracle as O
    cams, frames, _ = _frames(kind, 2, step)
    mp = capi.make_multi_projector(cams)
    b, a = _models(cams)
    so = _offset() if offset else np.eye(4, dtype=np.float32)
    d = composite(ctx, frames[0], cams, step)
    assert np.array_equal(_bits(d), _bits(_oracle_composite(frames[0], cams, step)))
    cl, _ = ctx.multi_depth_to_cloud(d, mp, _sp(), so)
    cl.multi_compute_gaussians(d, mp, b, a, so)
    g, f = cl.download_gaussians()
    og, of, _, _ = oracle_rig_gaussians(cams, d, b, a, so)
    assert g.shape == og.shape and g.shape[0] > 0.3 * d.size
    assert np.array_equal(_bits(g), _bits(og)) and np.array_equal(f, of)
    # the rig points before the offset are the means: with an identity offset they are the cloud's points
    if not offset:
        assert np.array_equal(_bits(cl.download()["points"][:, :3]), _bits(g[:, :3]))
    other = d.copy()
    other[:, :cams[0]["height"] // 2] = 0.0
    with pytest.raises(capi.NicpError, match="valid pixels"):
        cl.multi_compute_gaussians(other, mp, b, a, so)
    with pytest.raises(capi.NicpError):
        cl.multi_compute_gaussians(d, mp, np.zeros(len(cams), np.float32), a, so)
    cl.close()


# kind, n, step, sensor offset, merge (None / "identity" / "pose"), voxel resolution: a launch set of the test rigs holds 8
# frames, so 9 and 17 cross its boundary
CASES = [
    ("4cam", 1, 1, False, None, 0.0),
    ("4cam", 9, 2, True, "identity", 0.05),
    ("4cam", 17, 2, False, "pose", 0.0),
    ("ragged", 17, 1, True, "pose", 0.05),
    ("ragged", 9, 2, False, None, 0.0),
    ("ragged", 2, 1, False, "identity", 0.0),
    # config-5 rig: one frame per launch set at step 1, two at step 2
    ("config5", 3, 2, True, "pose", 0.05),
    ("config5", 2, 1, False, None, 0.0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n,step,offset,merge,vres", CASES)
def test_rig_local_map_equals_chain(ctx, kind, n, step, offset, merge, vres):
    cams, frames, poses = _frames(kind, n, step)
    so = _offset() if offset else None
    mp, mT = _merge_args(merge, poses)
    P = max(c["width"] for c in cams) * sum(c["height"] for c in cams)
    a, b = ctx.new_cloud(n * P), ctx.new_cloud(n * P)
    col_c, rep_c = _chain(ctx, cams, frames, poses, step, so, a, mp, mT, vres)
    appended, size, col_e, rep_e = _entry(ctx, cams, frames, poses, step, so, b, mp, mT, vres)
    sa, sb = _snapshot(a), _snapshot(b)
    _assert_same(sa, sb)
    assert size == sa["size"] and appended > 0.3 * n * P
    if mp is None:
        assert col_e is None and size == appended
    else:
        assert np.array_equal(col_e, col_c) and len(col_e) == appended
    if vres > 0:
        assert np.array_equal(rep_e, rep_c) and len(rep_e) == size
    else:
        assert rep_e is None
    a.close()
    b.close()


def _prefill(ctx, cl, with_gauss):
    """a map that already holds one rig frame's points (frame 16 of the 4-camera rig at step 2), with or without gaussians"""
    cams, frames, poses = _frames("4cam", 17, 2)
    mp = capi.make_multi_projector(cams)
    fc = ctx.multi_raw_depth_to_cloud_batch([frames[16]], mp, _sp(), step=2)[0]
    if with_gauss:
        fc.multi_compute_gaussians(composite(ctx, frames[16], cams, 2), mp, *_models(cams))
        cl.append(fc, poses[16])
    else:
        d = fc.download()
        cl.upload(d["points"], d["normals"], d["curvature"], d["omega_p"], d["omega_n"])
    fc.close()


RIG_PX = 160 * 480  # composite pixels of the 4-camera test rig


@pytest.mark.gpu
@pytest.mark.parametrize("with_gauss", [True, False])
def test_rig_local_map_behind_existing_points(ctx, with_gauss):
    cams, frames, poses = _frames("4cam", 9, 2)
    so = _offset()
    mp, mT = _merge_args("identity", poses)
    a, b = ctx.new_cloud(10 * RIG_PX), ctx.new_cloud(10 * RIG_PX)
    _prefill(ctx, a, with_gauss)
    _prefill(ctx, b, with_gauss)
    before = a.size()
    assert before > 0 and a.has_gaussians() == with_gauss
    col_c, _ = _chain(ctx, cams, frames, poses, 2, so, a, mp, mT)
    appended, size, col_e, _ = _entry(ctx, cams, frames, poses, 2, so, b, mp, mT)
    _assert_same(_snapshot(a), _snapshot(b))
    assert np.array_equal(col_e, col_c) and len(col_e) == before + appended
    if not with_gauss:
        # the points that were there get all-zero gaussians, as Cloud::add leaves them
        a2 = ctx.new_cloud(10 * RIG_PX)
        _prefill(ctx, a2, False)
        _entry(ctx, cams, frames, poses, 2, so, a2)
        g, f = a2.download_gaussians()
        assert not g[:before].any() and not f[:before].any()


@pytest.mark.gpu
def test_rig_local_map_too_small_leaves_the_map(ctx):
    cams, frames, poses = _frames("4cam", 9, 2)
    big = ctx.new_cloud(9 * RIG_PX)
    appended, _, _, _ = _entry(ctx, cams, frames, poses, 2, None, big)
    for with_gauss in (False, True):
        before = ctx.new_cloud(10 * RIG_PX)
        _prefill(ctx, before, with_gauss)
        n0 = before.size()
        # the first launch set of 8 frames fits, the ninth frame does not
        small = ctx.new_cloud(n0 + appended - 1)
        _prefill(ctx, small, with_gauss)
        snap = _snapshot(small)
        with pytest.raises(capi.NicpError) as e:
            _entry(ctx, cams, frames, poses, 2, None, small, *_merge_args("identity", poses), vres=0.05)
        assert e.value.needed_size == n0 + appended
        _assert_same(_snapshot(small), snap)
        fits = ctx.new_cloud(n0 + appended)
        _prefill(ctx, fits, with_gauss)
        assert _entry(ctx, cams, frames, poses, 2, None, fits)[1] == n0 + appended


def _good_args(ctx, cams, frames, poses, map_cloud, step=2):
    mp = capi.make_multi_projector(cams)
    imgs, rr, rc = capi._rig_frames(frames, len(cams))
    b, a = _models(cams)
    keep = SimpleNamespace(mp=mp, sp=_sp(), view=_merge_view(cams), merge=capi.make_merge_params(), so=capi.colmajor(np.eye(4)),
                           mt=capi.colmajor(np.eye(4)), b=b, a=a, rr=rr, rc=rc, imgs=imgs,
                           poses=np.ascontiguousarray(np.asarray(poses, np.float32).transpose(0, 2, 1)).reshape(-1),
                           RA=(C.c_void_p * len(imgs))(*[im.ctypes.data for im in imgs]))
    fp = lambda x: x.ctypes.data_as(C.POINTER(C.c_float))
    ip = lambda x: x.ctypes.data_as(C.POINTER(C.c_int))
    args = [ctx.handle, len(frames), keep.RA, ip(rr), ip(rc), C.c_float(DEPTH_SCALE), step, C.c_float(MAX_DEPTH_COV),
            C.byref(keep.mp), C.byref(keep.sp), fp(keep.so), fp(b), fp(a), fp(keep.poses), C.byref(keep.view),
            C.byref(keep.merge), fp(keep.mt), C.c_float(0.0), map_cloud.handle, None, None, None, None]
    return args, keep


@pytest.mark.gpu
def test_rig_local_map_rejects_bad_arguments(ctx):
    """every bad argument is refused before anything is queued: the launch count and the map stay, the context stays usable"""
    cams, frames, poses = _frames("4cam", 3, 2)
    m = ctx.new_cloud(3 * RIG_PX)
    L = ctx.L
    good, keep = _good_args(ctx, cams, frames, poses, m)
    fp = lambda x: x.ctypes.data_as(C.POINTER(C.c_float))
    ip = lambda x: x.ctypes.data_as(C.POINTER(C.c_int))
    null_raw = (C.c_void_p * len(keep.imgs))(*[None if k == 5 else im.ctypes.data for k, im in enumerate(keep.imgs)])
    wrong_rows = keep.rr.copy()
    wrong_rows[2] += 2
    b0, a_neg = keep.b.copy(), keep.a.copy()
    b0[1] = 0.0
    a_neg[3] = -0.1
    bad = {"ctx": (0, None), "n=0": (1, 0), "n<0": (1, -2), "raws": (2, None), "raw image": (2, null_raw),
           "raw_rows": (3, None), "raw size vs rig": (3, ip(wrong_rows)), "mp": (8, None), "sp": (9, None),
           "sensor_offset": (10, None), "baseline": (11, None), "baseline 0": (11, fp(b0)), "alpha": (12, None),
           "alpha < 0": (12, fp(a_neg)), "poses": (13, None), "merge_proj": (14, None), "merge_transform": (16, None),
           "map": (18, None)}
    launches = ctx.launch_count()
    for name, (i, v) in bad.items():
        args = list(good)
        args[i] = v
        assert L.nicp_multi_raw_depth_to_local_map(*args) == 1, name
        assert ctx.launch_count() == launches, name
    assert m.size() == 0 and not m.has_gaussians()
    # merge_proj and merge_transform may be NULL when no merge is asked for; the good call goes through
    args = list(good)
    args[14], args[15], args[16] = None, None, None
    assert L.nicp_multi_raw_depth_to_local_map(*args) == 0 and m.size() > 0
    m.upload(np.zeros((0, 4), np.float32))
    assert L.nicp_multi_raw_depth_to_local_map(*good) == 0 and m.size() > 0


@pytest.mark.gpu
def test_rig_local_map_deterministic_after_alignment_batches(ctx):
    """the same call gives the same bytes on fresh maps, also after rig alignment batches reused the context's scratch"""
    cams, frames, poses = _frames("ragged", 11, 1)
    so = _offset()
    mp, mT = _merge_args("pose", poses)
    snaps = []
    for rnd in range(3):
        cl = ctx.new_cloud(11 * 64 * 136)
        res = _entry(ctx, cams, frames, poses, 1, so, cl, mp, mT, 0.05)
        snaps.append((_snapshot(cl), res[0], res[1], res[2], res[3]))
        cl.close()
        if rnd == 1:
            c4, f4, _ = _frames("4cam", 9, 2)
            m4 = capi.make_multi_projector(c4)
            clouds = ctx.multi_raw_depth_to_cloud_batch(f4, m4, _sp(), step=2)
            ap = capi.make_align_params(1.0, 0.95, 0.02, 1.3, 9e3, True, 5, 1)
            assert len(ctx.multi_align_batch(clouds[:8], clouds[1:9], m4, ap)) == 8
    for s in snaps[1:]:
        _assert_same(s[0], snaps[0][0])
        assert s[1:3] == snaps[0][1:3]
        assert np.array_equal(s[3], snaps[0][3]) and np.array_equal(s[4], snaps[0][4])


@pytest.mark.gpu
def test_rig_local_map_matches_oracle():
    """two rig frames through the entry against the oracle: orc_multi_depth_to_cloud with eigen variant 2 (the
    trigonometry evaluated like the CUDA path), oracle_rig_gaussians with the sensor offset, Cloud::add and
    Merger::merge with the pinhole merge view; the bars of test_local_map.test_local_map_matches_oracle"""
    from oracle import pwn_oracle as O
    cams, frames, poses = _frames("4cam", 2, 2)
    b, a = _models(cams)
    so = _offset()
    om = O.make_multi(cams)
    osp = O.default_stats_params(minImageRadius=3, maxImageRadius=6, minPoints=10, curvatureThreshold=0.2)
    view = _merge_view(cams)
    O.set_eigen_variant(2)
    try:
        parts = []
        for fr, T in zip(frames, poses):
            d = _oracle_composite(fr, cams, 2)
            cl, _ = O.multi_depth_to_cloud(om, d, osp, so)
            g, f, _, _ = oracle_rig_gaussians(cams, d, b, a, so)
            assert g.shape[0] == cl.n
            pts, nrm, st, op, on = (cl.points.copy(), cl.normals.copy(), cl.statsM.copy(), cl.omegaP.copy(), cl.omegaN.copy())
            fp = lambda x: x.ctypes.data_as(C.POINTER(C.c_float))
            Tc = O.colmajor(T)
            O.lib().orc_cloud_transform(fp(Tc), cl.n, fp(pts), fp(nrm), fp(st), fp(op), fp(on))
            g, f = O.gaussians_transform(T, g, f)
            parts.append((cl, pts, nrm, st, op, on, g, f))
        n = sum(p[0].n for p in parts)
        m = O.Cloud(n)
        m.points = np.ascontiguousarray(np.concatenate([p[1] for p in parts]))
        m.normals = np.ascontiguousarray(np.concatenate([p[2] for p in parts]))
        m.statsM = np.ascontiguousarray(np.concatenate([p[3] for p in parts]))
        m.omegaP = np.ascontiguousarray(np.concatenate([p[4] for p in parts]))
        m.omegaN = np.ascontiguousarray(np.concatenate([p[5] for p in parts]))
        m.eigvals = np.ascontiguousarray(np.concatenate([p[0].eigvals for p in parts]))
        m.statsN = np.ascontiguousarray(np.concatenate([p[0].statsN for p in parts]))
        m.curvature = np.ascontiguousarray(np.concatenate([p[0].curvature for p in parts]))
        g = np.ascontiguousarray(np.concatenate([p[6] for p in parts]))
        f = np.ascontiguousarray(np.concatenate([p[7] for p in parts]))
        for verify in (True, False):
            ctx = capi.Context(0, verify=verify)
            for T, mp in ((np.eye(4, dtype=np.float32), capi.make_merge_params()), (poses[1], capi.make_merge_params(0.05, 0.99, 3.0))):
                res, go, fo, col = O.merge(m, g, f, view.rows, view.cols, cams[0]["K"], T, cams[0]["minD"], cams[0]["maxD"],
                                           mp.distance_threshold, mp.normal_threshold, mp.max_point_depth)
                cl = ctx.new_cloud(n)
                appended, k, col_d, _ = _entry(ctx, cams, frames, poses, 2, so, cl, mp, T)
                assert appended == n
                assert np.array_equal(col_d, col) and (col >= 0).sum() > 0
                assert k == res.n == cl.size()
                d = cl.download()
                assert np.array_equal(_bits(d["points"]), _bits(res.points))
                assert np.array_equal(_bits(d["normals"][:, :3]), _bits(res.normals[:, :3]))
                assert np.array_equal(_bits(d["curvature"]), _bits(res.curvature))
                # information matrices (both frames are moved by Cloud::add): the device rotates the symmetric completion of the stored upper
                # triangle and the oracle the full matrix, the bar of test_gpu_parity.test_cloud_append
                for got, ref in ((d["omega_p"], res.omegaP6()), (d["omega_n"], res.omegaN6())):
                    err = np.abs(got - ref).max(1) / np.maximum(np.abs(ref).max(1), 1e-9)
                    assert np.nanquantile(err, 0.999) < 1e-5
                gd, fd = cl.download_gaussians()
                assert np.array_equal(fd, fo)
                mom = (fo & O.GAUSS_MOMENTS) != 0
                inf = (fo & O.GAUSS_INFO) != 0
                assert np.array_equal(_bits(gd[mom, :12]), _bits(go[mom, :12]))
                assert np.array_equal(_bits(gd[inf, 12:]), _bits(go[inf, 12:]))
                cl.close()
            ctx.close()
    finally:
        O.set_eigen_variant(0)


# ---- the pwn:: layer -----------------------------------------------------------------------------------------------------
PWN_DRIVER = r"""
// a rig converter with setKeepGaussians(true), then Merger::merge through a pinhole view (tests/test_rig_local_map.py)
#include <cstdio>
#include <vector>
#include "pwn/pwn.h"
using namespace pwn;

static void readf(FILE *f, float *p, size_t n) { if (fread(p, sizeof(float), n, f) != n) throw std::runtime_error("short input"); }

int main(int argc, char **argv) {
  FILE *in = fopen(argv[1], "rb");
  float hdr[3];
  readf(in, hdr, 3);
  const int nc = (int)hdr[0], rows = (int)hdr[1], cols = (int)hdr[2];
  MultiPointProjector mp;
  std::vector<PinholePointProjector> cams(nc);
  for (int i = 0; i < nc; i++) {
    float v[9 + 16 + 6];
    readf(in, v, 31);
    Matrix3f K;
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) K(r, c) = v[c * 3 + r];
    cams[i].setCameraMatrix(K);
    cams[i].setMinDistance(v[27]);
    cams[i].setMaxDistance(v[28]);
    cams[i].setBaseline(v[29]);
    cams[i].setAlpha(v[30]);
    Isometry3f off;
    for (int k = 0; k < 16; k++) off.data()[k] = v[9 + k];
    mp.addPointProjector(&cams[i], off, (int)v[25], (int)v[26]);
  }
  DepthImage depth(rows, cols);
  readf(in, depth.data(), (size_t)rows * cols);
  float view[13];
  readf(in, view, 13);
  fclose(in);
  StatsCalculatorIntegralImage sc;
  sc.setMinImageRadius(3);
  sc.setMaxImageRadius(6);
  sc.setMinPoints(10);
  PointInformationMatrixCalculator pic;
  NormalInformationMatrixCalculator nic;
  DepthImageConverterIntegralImage conv(&mp, &sc, &pic, &nic);
  conv.setKeepGaussians(true);
  Cloud cloud;
  conv.compute(cloud, depth);
  if (!cloud.hasGaussians()) throw std::runtime_error("no gaussians");
  Gaussian3fVector g = cloud.gaussians();
  FILE *out = fopen(argv[2], "wb");
  for (size_t i = 0; i < g.size(); i++) {
    float rec[13];
    for (int k = 0; k < 3; k++) rec[k] = g[i].mean()(k);
    for (int c = 0; c < 3; c++)
      for (int r = 0; r < 3; r++) rec[3 + c * 3 + r] = g[i].covarianceMatrix()(r, c);
    rec[12] = g[i]._momentsUpdated ? 1.0f : 0.0f;
    fwrite(rec, sizeof(float), 13, out);
  }
  fclose(out);
  // the merge view: a PinholePointProjector of the Merger's image size
  PinholePointProjector pinhole;
  Matrix3f K;
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) K(r, c) = view[c * 3 + r];
  pinhole.setCameraMatrix(K);
  pinhole.setMinDistance(view[11]);
  pinhole.setMaxDistance(view[12]);
  DepthImageConverterIntegralImage viewConv(&pinhole, &sc, &pic, &nic);
  Merger merger;
  merger.setDepthImageConverter(&viewConv);
  merger.setImageSize((int)view[9], (int)view[10]);
  const size_t before = cloud.size();
  merger.merge(&cloud);
  printf("merged %zu %zu\n", before, cloud.size());
  return 0;
}
"""


@pytest.mark.gpu
def test_pwn_rig_converter_keeps_gaussians(tmp_path):
    """pwn::DepthImageConverterIntegralImage with a MultiPointProjector and setKeepGaussians(true): the cloud's gaussians
    equal nicp_multi_cloud_compute_gaussians (the children's baseline() / alpha()), and Merger::merge with a pinhole view
    fuses the rig cloud"""
    cams, frames, _ = _frames("ragged", 1, 1)
    b, a = _models(cams)
    lib = os.path.join(ROOT, "g2o_frontend_b200", "lib")
    src, exe = tmp_path / "rig_gaussians.cpp", str(tmp_path / "rig_gaussians")
    src.write_text(PWN_DRIVER)
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([cxx, "-std=c++17", "-O1", "-ffp-contract=off", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           "-o", exe, str(src), "-L", lib, "-lnicp_b200", "-Wl,-rpath," + lib])
    ctx = capi.Context(0)
    d = composite(ctx, frames[0], cams, 1)
    view = _merge_view(cams)
    rows, cols = d.shape
    blob = [np.array([len(cams), rows, cols], np.float32)]
    for i, c in enumerate(cams):
        blob.append(np.concatenate([capi.colmajor(c["K"]), capi.colmajor(c["offset"]),
                                    np.array([c["width"], c["height"], c["minD"], c["maxD"], b[i], a[i]], np.float32)]))
    blob += [d.reshape(-1), np.concatenate([np.asarray(view.K[:], np.float32),
                                            np.array([view.rows, view.cols, view.min_distance, view.max_distance], np.float32)])]
    (tmp_path / "in.bin").write_bytes(np.concatenate(blob).astype(np.float32).tobytes())
    out = subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    _, before, after = out.stdout.split()
    got = np.fromfile(tmp_path / "out.bin", np.float32).reshape(-1, 13)
    mp = capi.make_multi_projector(cams)
    cl, _ = ctx.multi_depth_to_cloud(d, mp, _sp())
    cl.multi_compute_gaussians(d, mp, b, a)
    g, f = cl.download_gaussians()
    assert got.shape[0] == g.shape[0] == int(before) > 0.3 * d.size
    assert np.array_equal(_bits(got[:, :12]), _bits(g[:, :12])) and np.all(got[:, 12] == 1.0)
    assert 0 < int(after) < int(before)
    ctx.close()

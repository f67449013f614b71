"""Local maps from raw frames in one call (nicp_raw_depth_to_local_map).

GPU part (-m gpu, both library builds): the entry against the chain of single calls it replaces -- per frame
nicp_raw_depth_to_cloud, nicp_depth_prepare, nicp_cloud_compute_gaussians, nicp_cloud_append, then nicp_merge and
nicp_voxelize -- byte for byte, and end to end against the oracle.  CPU part: argument checks that need no device.
"""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest

from conftest import get_scene

BASELINE, ALPHA = 0.075, 0.1  # PinholePointProjector defaults (pinholepointprojector.cpp:5-13)
MIN_D, MAX_D = 0.5, 4.5


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _offset():
    from g2o_frontend_b200 import synth
    return synth.make_pose((0.1, -0.05, 0.3), (0.3, 1.0, 0.2), 7.0).astype(np.float32)


_FRAMES = {}


def _frames(n, noisy):
    """the first n of 17 raw 640x480 frames along synth.trajectory, with their poses"""
    from g2o_frontend_b200 import synth
    if noisy not in _FRAMES:
        poses = [p.astype(np.float32) for p in synth.trajectory(17, seed=3)]
        raws = [synth.render_depth_u16(p, seed=100 + i if noisy else None, dropout=0.05 if noisy else 0.0)
                for i, p in enumerate(poses)]
        _FRAMES[noisy] = (raws, poses)
    raws, poses = _FRAMES[noisy]
    return raws[:n], poses[:n]


def _camera(step):
    from g2o_frontend_b200 import capi, synth
    K = synth.scaled_K(synth.K_KINECT, 1.0 / step)
    proj = capi.make_projector(K, 480 // step, 640 // step, MIN_D, MAX_D)
    sp = capi.make_stats_params(0.1, 10, 30, 50, 0.2, 0.02) if step == 1 else capi.make_stats_params(0.1, 3, 6, 10, 0.2, 0.02)
    return proj, sp


@pytest.fixture(scope="module", params=["verify", "default"])
def ctx(request):
    from g2o_frontend_b200 import capi
    c = capi.Context(0, verify=(request.param == "verify"))
    yield c
    c.close()


def _chain(ctx, raws, poses, step, so, map_cloud, mp=None, mT=None, vres=0.0):
    """the calls the entry replaces, one frame at a time -> (collapsed or None, representatives or None)"""
    proj, sp = _camera(step)
    for raw, T in zip(raws, poses):
        fc, _ = ctx.raw_depth_to_cloud(raw, proj, sp, step=step, sensor_offset=so)
        fc.compute_gaussians(ctx.depth_prepare(raw, step=step), proj, BASELINE, ALPHA, so)
        map_cloud.append(fc, T)
        fc.close()
    col = rep = None
    if mp is not None:
        _, col = map_cloud.merge(proj, np.eye(4, dtype=np.float32) if mT is None else mT, mp)
    if vres > 0:
        _, rep = map_cloud.voxelize(vres)
    return col, rep


def _entry(ctx, raws, poses, step, so, map_cloud, mp=None, mT=None, vres=0.0):
    proj, sp = _camera(step)
    return ctx.raw_depth_to_local_map(raws, proj, sp, poses, map_cloud, step=step, sensor_offset=so, baseline=BASELINE,
                                      alpha=ALPHA, merge_params=mp, merge_transform=mT, voxel_resolution=vres)


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


def _prefill(ctx, cl, with_gauss):
    """a map that already holds one frame's points (frame 16 at step 4), with or without gaussians"""
    raws, poses = _frames(17, True)
    proj, sp = _camera(4)
    fc, _ = ctx.raw_depth_to_cloud(raws[16], proj, sp, step=4)
    if with_gauss:
        fc.compute_gaussians(ctx.depth_prepare(raws[16], step=4), proj, BASELINE, ALPHA)
        cl.append(fc, poses[16])
    else:
        d = fc.download()
        cl.upload(d["points"], d["normals"], d["curvature"], d["omega_p"], d["omega_n"])
    fc.close()


# n, step, sensor offset, noise + 5 % dropout, merge (None / "identity" / "pose"), voxel resolution: every value of each
# axis appears, the sub-batch boundary (8) is crossed at 9 and 17 frames
CASES = [
    (1, 4, False, False, None, 0.0),
    (2, 2, True, True, "identity", 0.05),
    (8, 4, True, True, "pose", 0.0),
    (9, 4, False, True, "identity", 0.05),
    (17, 4, True, True, "pose", 0.05),
    (17, 2, False, False, None, 0.0),
    (9, 1, True, True, "identity", 0.05),
    (2, 1, False, False, "pose", 0.0),
]


def _merge_args(merge, poses):
    from g2o_frontend_b200 import capi
    if merge is None:
        return None, None
    if merge == "identity":
        return capi.make_merge_params(), np.eye(4, dtype=np.float32)
    return capi.make_merge_params(0.05, 0.99, 3.0), poses[len(poses) // 2]


@pytest.mark.gpu
@pytest.mark.parametrize("n,step,offset,noisy,merge,vres", CASES)
def test_local_map_equals_chain(ctx, n, step, offset, noisy, merge, vres):
    raws, poses = _frames(n, noisy)
    so = _offset() if offset else None
    mp, mT = _merge_args(merge, poses)
    P = (480 // step) * (640 // step)
    a, b = ctx.new_cloud(n * P), ctx.new_cloud(n * P)
    col_c, rep_c = _chain(ctx, raws, poses, step, so, a, mp, mT, vres)
    appended, size, col_e, rep_e = _entry(ctx, raws, poses, step, so, b, mp, mT, vres)
    sa, sb = _snapshot(a), _snapshot(b)
    _assert_same(sa, sb)
    assert size == sa["size"] and appended > 0.3 * n * P
    if mp is None:
        assert col_e is None and size == appended
    else:
        assert np.array_equal(col_e, col_c) and len(col_e) == appended
        assert (col_e >= 0).sum() > 0
    if vres > 0:
        assert np.array_equal(rep_e, rep_c) and len(rep_e) == size
    else:
        assert rep_e is None
    a.close()
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("with_gauss", [True, False])
def test_local_map_behind_existing_points(ctx, with_gauss):
    raws, poses = _frames(9, True)
    so = _offset()
    mp, mT = _merge_args("identity", poses)
    a, b = ctx.new_cloud(10 * 19200), ctx.new_cloud(10 * 19200)
    _prefill(ctx, a, with_gauss)
    _prefill(ctx, b, with_gauss)
    before = a.size()
    assert before > 0 and a.has_gaussians() == with_gauss
    col_c, _ = _chain(ctx, raws, poses, 4, so, a, mp, mT)
    appended, size, col_e, _ = _entry(ctx, raws, poses, 4, so, b, mp, mT)
    _assert_same(_snapshot(a), _snapshot(b))
    assert np.array_equal(col_e, col_c) and len(col_e) == before + appended
    if not with_gauss:
        # the points that were there get all-zero gaussians, as Cloud::add leaves them
        a2 = ctx.new_cloud(10 * 19200)
        _prefill(ctx, a2, False)
        _entry(ctx, raws, poses, 4, so, a2)
        g, f = a2.download_gaussians()
        assert not g[:before].any() and not f[:before].any()


@pytest.mark.gpu
def test_local_map_matches_oracle():
    """two frames at 160x120 through the entry against the oracle's two_frame_map + Merger::merge, with the oracle's
    eigen variant that evaluates the trigonometry like the CUDA path (variant 2): bit-exact arrays, gaussians where
    their flags say they are valid (the bars of test_map_ops.test_gpu_merge_bit_exact), and the information matrices of
    the transformed frame within the bar of the device's Cloud::add against the oracle"""
    from oracle import pwn_oracle as O
    from g2o_frontend_b200 import capi
    from test_map_ops import two_frame_map
    s = get_scene(4, 0, 0.05, True)
    c = s.conf
    O.set_eigen_variant(2)
    try:
        oA, _ = O.depth_to_cloud(s.depthA, s.K, c["minD"], c["maxD"], s.sp, s.sensor_offset)
        oB, _ = O.depth_to_cloud(s.depthB, s.K, c["minD"], c["maxD"], s.sp, s.sensor_offset)
        m, g, f = two_frame_map(SimpleNamespace(conf=c, depthA=s.depthA, depthB=s.depthB, K=s.K, sensor_offset=s.sensor_offset,
                                                gt=s.gt, cloudA=oA, cloudB=oB))
        for verify in (True, False):
            ctx = capi.Context(0, verify=verify)
            for T, mp in ((np.eye(4, dtype=np.float32), capi.make_merge_params()), (s.gt, capi.make_merge_params(0.05, 0.99, 3.0))):
                res, go, fo, col = O.merge(m, g, f, s.rows, s.cols, s.K, T, c["minD"], c["maxD"], mp.distance_threshold,
                                           mp.normal_threshold, mp.max_point_depth)
                cl = ctx.new_cloud(2 * s.rows * s.cols)
                appended, k, col_d, _ = ctx.raw_depth_to_local_map([s.rawA, s.rawB], s.projector(), s.stats_params(),
                                                                    [np.eye(4, dtype=np.float32), s.gt], cl, step=4,
                                                                    sensor_offset=s.sensor_offset, baseline=BASELINE,
                                                                    alpha=ALPHA, merge_params=mp, merge_transform=T)
                assert appended == m.n
                assert np.array_equal(col_d, col)
                assert k == res.n == cl.size()
                d = cl.download()
                assert np.array_equal(_bits(d["points"]), _bits(res.points))
                assert np.array_equal(_bits(d["normals"][:, :3]), _bits(res.normals[:, :3]))
                assert np.array_equal(_bits(d["curvature"]), _bits(res.curvature))
                # information matrices: bit-exact for frame A (appended at identity); frame B's were moved by Cloud::add, where
                # the device rotates the symmetric completion of the stored upper triangle and the oracle the full matrix, the
                # bar of test_gpu_parity.test_cloud_append
                src = np.nonzero((col < 0) | (col == np.arange(m.n)))[0]
                fromA = src < oA.n
                for got, ref in ((d["omega_p"], res.omegaP6()), (d["omega_n"], res.omegaN6())):
                    assert np.array_equal(_bits(got[fromA]), _bits(ref[fromA]))
                    err = np.abs(got[~fromA] - ref[~fromA]).max(1) / np.maximum(np.abs(ref[~fromA]).max(1), 1e-9)
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


@pytest.mark.gpu
def test_local_map_too_small_leaves_the_map(ctx):
    from g2o_frontend_b200 import capi
    raws, poses = _frames(9, True)
    big = ctx.new_cloud(9 * 19200)
    appended, _, _, _ = _entry(ctx, raws, poses, 4, None, big)
    for with_gauss in (False, True):
        before = ctx.new_cloud(10 * 19200)
        _prefill(ctx, before, with_gauss)
        n0 = before.size()
        # the first launch set of 8 frames fits, the ninth frame does not
        small = ctx.new_cloud(n0 + appended - 1)
        _prefill(ctx, small, with_gauss)
        snap = _snapshot(small)
        with pytest.raises(capi.NicpError) as e:
            _entry(ctx, raws, poses, 4, None, small, *_merge_args("identity", poses), vres=0.05)
        assert e.value.needed_size == n0 + appended
        _assert_same(_snapshot(small), snap)
        # and exactly the needed capacity is enough
        fits = ctx.new_cloud(n0 + appended)
        _prefill(ctx, fits, with_gauss)
        assert _entry(ctx, raws, poses, 4, None, fits)[1] == n0 + appended


def _good_args(ctx, raws, poses, map_cloud, step=4, merge=True):
    from g2o_frontend_b200 import capi
    proj, sp = _camera(step)
    keep = SimpleNamespace(proj=proj, sp=sp, mp=capi.make_merge_params(), so=capi.colmajor(np.eye(4)),
                           mt=capi.colmajor(np.eye(4)),
                           poses=np.ascontiguousarray(np.asarray(poses, np.float32).transpose(0, 2, 1)).reshape(-1),
                           RA=(C.c_void_p * len(raws))(*[r.ctypes.data for r in raws]))
    rows, cols = raws[0].shape
    fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
    args = [ctx.handle, len(raws), keep.RA, rows, cols, C.c_float(0.001), step, C.c_float(0.01), C.byref(keep.proj),
            C.byref(keep.sp), fp(keep.so), C.c_float(BASELINE), C.c_float(ALPHA), fp(keep.poses),
            C.byref(keep.mp) if merge else None, fp(keep.mt), C.c_float(0.0), map_cloud.handle, None, None, None, None]
    return args, keep


@pytest.mark.gpu
def test_local_map_rejects_bad_arguments(ctx):
    """every bad argument is refused in the calling thread before anything is queued: the launch count and the map stay"""
    raws, poses = _frames(3, False)
    m = ctx.new_cloud(3 * 19200)
    L = ctx.L
    good, keep = _good_args(ctx, raws, poses, m)
    null_raw = (C.c_void_p * 3)(raws[0].ctypes.data, None, raws[2].ctypes.data)
    bad_proj = _camera(2)[0]
    bad = {"ctx": (0, None), "n=0": (1, 0), "n<0": (1, -2), "raws": (2, None), "raw image": (2, null_raw),
           "raw_rows": (3, 0), "size vs projector": (8, C.byref(bad_proj)), "proj": (8, None), "sp": (9, None),
           "sensor_offset": (10, None), "poses": (13, None), "merge_transform": (15, None), "map": (17, None)}
    launches = ctx.launch_count()
    for name, (i, v) in bad.items():
        args = list(good)
        args[i] = v
        assert L.nicp_raw_depth_to_local_map(*args) == 1, name
        assert ctx.launch_count() == launches, name
    assert m.size() == 0 and not m.has_gaussians()
    # merge_transform may be NULL when no merge is asked for; the good call itself goes through
    args, keep2 = _good_args(ctx, raws, poses, m, merge=False)
    args[15] = None
    assert L.nicp_raw_depth_to_local_map(*args) == 0 and m.size() > 0


@pytest.mark.gpu
def test_local_map_deterministic_after_alignment_batches(ctx):
    """the same call twice on fresh maps gives the same bytes, also after pinhole alignment batches (at another image size)
    have reused and regrown the context's scratch"""
    from g2o_frontend_b200 import capi
    raws, poses = _frames(11, True)
    so = _offset()
    mp, mT = _merge_args("pose", poses)
    snaps = []
    for rnd in range(3):
        cl = ctx.new_cloud(11 * 19200)
        res = _entry(ctx, raws, poses, 4, so, cl, mp, mT, 0.05)
        snaps.append((_snapshot(cl), res[0], res[1], res[2], res[3]))
        cl.close()
        if rnd == 1:
            proj, sp = _camera(1)
            clouds = ctx.raw_depth_to_cloud_batch(raws[:9], proj, sp, step=1)
            ap = capi.make_align_params(1.0, 0.95, 0.02, 1.3, 9e3, True, 5, 1)
            assert len(ctx.align_batch(clouds[:8], clouds[1:9], proj, ap)) == 8
    for s in snaps[1:]:
        _assert_same(s[0], snaps[0][0])
        assert s[1:3] == snaps[0][1:3]
        assert np.array_equal(s[3], snaps[0][3]) and np.array_equal(s[4], snaps[0][4])


@pytest.mark.parametrize("verify", [False, True])
def test_local_map_null_handles_without_device(verify):
    """the entry answers a null context or map with NICP_ERR_INVALID before touching a device (no GPU needed)"""
    from g2o_frontend_b200 import capi
    L = capi.load(verify)
    N = None
    f0 = C.c_float(0)
    assert L.nicp_raw_depth_to_local_map(N, 2, N, 4, 4, C.c_float(0.001), 1, C.c_float(0.01), N, N, N, f0, f0, N, N, N, f0,
                                         N, N, N, N, N) == 1

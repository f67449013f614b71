"""Batched frame preparation from raw rig frames and batched rig alignment (MultiPointProjector, BASELINE config 5):
nicp_multi_raw_depth_to_cloud_batch must equal the composition of the single-frame entries bit for bit, and every record of
nicp_multi_align_batch must equal nicp_multi_align on that pair byte for byte."""
import ctypes as C

import numpy as np
import pytest

from g2o_frontend_b200 import capi, synth

DEPTH_SCALE, MAX_DEPTH_COV = 0.001, 0.01  # the defaults of the raw entry points


@pytest.fixture(scope="module", params=["verify", "default"])
def ctx(request):
    c = capi.Context(0, verify=(request.param == "verify"))
    assert bool(c.L.nicp_is_verification_build()) == (request.param == "verify")
    yield c
    c.close()


def make_cams(kind):
    """the two rigs of test_multi_point_projector: 4 x 160x120, and a ragged 3-camera rig (sizes and ranges differ)"""
    if kind == "4cam":
        return synth.make_rig(4, 160, 120, K=synth.scaled_K(synth.K_KINECT, 160 / 640.0))
    cams = synth.make_rig(3, 64, 48, K=synth.scaled_K(synth.K_KINECT, 64 / 640.0))
    cams[1]["width"], cams[1]["height"] = 48, 40
    cams[2]["maxD"] = 3.0
    return cams


def render_raw_frame(rig_pose, cams, step, seed):
    """one raw image per camera in sensor orientation ((height * step) x (width * step), row = v), noisy with holes"""
    out = []
    for i, c in enumerate(cams):
        out.append(synth.render_depth_u16(rig_pose @ c["offset"].astype(np.float64), c["height"] * step, c["width"] * step,
                                          synth.scaled_K(c["K"], step), seed=seed + 17 * i, dropout=0.02,
                                          zmin=c["minD"], zmax=c["maxD"]))
    return out


def composite(ctx, raws, cams, step):
    """per camera depth_prepare(raw_i, step), transposed into the composite image on the host"""
    rows = max(c["width"] for c in cams)
    cols = sum(c["height"] for c in cams)
    out = np.zeros((rows, cols), np.float32)
    off = 0
    for r, c in zip(raws, cams):
        d = ctx.depth_prepare(r, DEPTH_SCALE, step, MAX_DEPTH_COV)
        assert d.shape == (c["height"], c["width"])
        out[:c["width"], off:off + c["height"]] = d.T
        off += c["height"]
    return out


def rig_poses(n, seed):
    rng = np.random.default_rng(seed)
    base = synth.make_pose((0.1, -0.05, 0.2), (0, 1, 0), 10.0)
    return [synth.perturbed_pose(rng, base, 0.04, 3.0) for _ in range(n)]


def pinned_copy(a):
    import torch
    t = torch.empty(a.shape, dtype=torch.int16).pin_memory()
    v = t.numpy().view(np.uint16)
    v[...] = a
    return v, t


def assert_clouds_equal(a, b, keep_stats, what):
    assert a.size() == b.size(), what
    da, db = a.download(), b.download()
    for k in da:
        assert np.array_equal(da[k].view(np.uint32), db[k].view(np.uint32)), (what, k)
    if keep_stats and a.size():
        for x, y in zip(a.download_stats(), b.download_stats()):
            assert np.array_equal(np.asarray(x).view(np.uint32), np.asarray(y).view(np.uint32)), what


@pytest.mark.parametrize("verify", [False, True])
def test_null_handles_are_rejected(verify):
    L = capi.load(verify)
    N, f0 = None, C.c_float(0)
    assert L.nicp_multi_raw_depth_to_cloud_batch(N, 2, N, N, N, C.c_float(0.001), 1, C.c_float(0.01), N, N, N, 0, N) == 1
    assert L.nicp_multi_align_batch(N, 2, N, N, N, N, N, N, N, N, N, f0, N) == 1


@pytest.mark.gpu
@pytest.mark.parametrize("kind,step,offset,pinned", [("4cam", 1, False, False), ("4cam", 2, True, True),
                                                     ("ragged", 1, True, True), ("ragged", 2, False, False)])
def test_raw_rig_prep_equals_single_frame_composition(ctx, kind, step, offset, pinned):
    """11 frames (one all-zero; a sub-batch boundary inside) through one batch call against, per frame, depth_prepare of
    each camera + a host transpose + multi_depth_to_cloud: every cloud array bit for bit; frame 0 also against the oracle"""
    from oracle import pwn_oracle as O
    cams = make_cams(kind)
    mp = capi.make_multi_projector(cams)
    rows, cols = capi.multi_image_size(mp, ctx.verify)
    so = (synth.make_pose((0.05, 0.0, 0.1), (1.0, 0.2, 0.0), 3.0).astype(np.float32) if offset
          else np.eye(4, dtype=np.float32))
    sp = capi.make_stats_params(0.1, 3, 6, 10, 0.2, 0.02)
    keep_stats = step == 1
    n = 11
    frames = [render_raw_frame(p, cams, step, 40 + 3 * f) for f, p in enumerate(rig_poses(n, 5))]
    frames[7] = [np.zeros_like(r) for r in frames[7]]
    pins = []
    if pinned:
        pinned_frames = []
        for fr in frames:
            views = [pinned_copy(r) for r in fr]
            pins += [t for _, t in views]
            pinned_frames.append([v for v, _ in views])
        src = pinned_frames
    else:
        src = frames
    batch = ctx.multi_raw_depth_to_cloud_batch(src, mp, sp, step=step, sensor_offset=so, keep_stats=keep_stats)
    ctx.synchronize()
    comps = [composite(ctx, fr, cams, step) for fr in frames]
    for f in range(n):
        ref, _ = ctx.multi_depth_to_cloud(comps[f], mp, sp, so, keep_stats=keep_stats)
        assert_clouds_equal(ref, batch[f], keep_stats, f)
    assert batch[7].size() == 0 and batch[0].size() > 0.3 * rows * cols
    # frame 0 against the oracle: index image (of the single-frame entry) and points bit-exact
    om = O.make_multi(cams)
    osp = O.default_stats_params(minImageRadius=3, maxImageRadius=6, minPoints=10, curvatureThreshold=0.2)
    d0 = np.zeros((rows, cols), np.float32)
    off = 0
    for r, c in zip(frames[0], cams):
        d = O.depth_u16_to_f32(r)
        if step > 1:
            d = O.depth_scale(d, step)
        d0[:c["width"], off:off + c["height"]] = d.T
        off += c["height"]
    assert np.array_equal(d0.view(np.uint32), comps[0].view(np.uint32))
    oc, oidx = O.multi_depth_to_cloud(om, d0, osp, so)
    _, gidx = ctx.multi_depth_to_cloud(d0, mp, sp, so)
    assert np.array_equal(gidx, oidx)
    assert oc.n == batch[0].size()
    assert np.array_equal(batch[0].download()["points"].view(np.uint32), oc.points.view(np.uint32))
    del pins


@pytest.mark.gpu
def test_raw_rig_prep_rejects_bad_input(ctx):
    cams = make_cams("ragged")
    mp = capi.make_multi_projector(cams)
    rows, cols = capi.multi_image_size(mp, ctx.verify)
    sp = capi.make_stats_params(0.1, 3, 6, 10, 0.2, 0.02)
    frame = render_raw_frame(rig_poses(1, 1)[0], cams, 1, 3)

    def expect(msg, frames, clouds=None, step=1):
        with pytest.raises(capi.NicpError, match=msg):
            ctx.multi_raw_depth_to_cloud_batch(frames, mp, sp, step=step, clouds=clouds)

    wrong = list(frame)
    wrong[1] = np.zeros((frame[1].shape[0] + 1, frame[1].shape[1]), np.uint16)
    expect("camera 1: raw image", [wrong])
    expect("camera 0: raw image", [frame], step=2)
    expect("capacity", [frame], clouds=[ctx.new_cloud(rows * cols - 1)])
    c = ctx.new_cloud(rows * cols)
    expect("same object", [frame, frame], clouds=[c, c])
    # a null camera image, through the C-ABI directly
    L = ctx.L
    imgs = frame + frame
    RA = (C.c_void_p * 6)(*[im.ctypes.data for im in imgs])
    RA[4] = None
    rr = np.array([im.shape[0] for im in frame], np.int32)
    rc = np.array([im.shape[1] for im in frame], np.int32)
    c2 = ctx.new_cloud(rows * cols)
    CA = (C.c_void_p * 2)(c.handle, c2.handle)
    so = capi.colmajor(np.eye(4))
    rc_ = L.nicp_multi_raw_depth_to_cloud_batch(ctx.handle, 2, RA, capi._iptr(rr), capi._iptr(rc), C.c_float(0.001), 1,
                                                C.c_float(0.01), C.byref(mp), C.byref(sp), capi._fptr(so), 0, CA)
    assert rc_ == 1
    assert b"null raw image of camera 1 in frame 1" in L.nicp_last_error()


def _align_case(c, kind):
    """7 rig pairs over 3 frames built from raw (shared and distinct current clouds), guesses, sensor offsets, priors"""
    cams = make_cams(kind)
    mp = capi.make_multi_projector(cams)
    sp = capi.make_stats_params(0.1, 3, 6, 10, 0.2, 0.02)
    so = synth.make_pose((0.05, 0.0, 0.1), (1.0, 0.2, 0.0), 3.0).astype(np.float32)
    poses = rig_poses(3, 11)
    frames = [render_raw_frame(p, cams, 1, 60 + f) for f, p in enumerate(poses)]
    clouds = c.multi_raw_depth_to_cloud_batch(frames, mp, sp, sensor_offset=so)
    A, B, D = clouds
    refs = [A, A, B, A, D, B, A]
    curs = [B, B, A, D, B, D, B]
    rng = np.random.default_rng(2)
    guesses = np.stack([synth.perturbed_pose(rng, np.eye(4), 0.02, 1.0) for _ in refs]).astype(np.float32)
    mean = synth.make_pose((0.05, -0.03, 0.08), (0.1, 1.0, 0.3), 3.0).astype(np.float32)
    refT = synth.make_pose((0.2, 0.1, -0.1), (1.0, 0.2, 0.1), 5.0).astype(np.float32)
    info = (np.diag([2e5, 1e5, 3e5, 5e6, 4e6, 6e6]) + 1e3).astype(np.float32)
    priors = [[], [capi.make_prior(0, mean, info, None)], [], [capi.make_prior(1, mean, info, refT)],
              [capi.make_prior(0, mean, info, None), capi.make_prior(1, mean, info * 0.5, refT)], [], []]
    ap = capi.make_align_params(0.5, 0.95, 0.02, 1.3, 9e3, True, 10, 1)
    singles = [bytes(c.multi_align(r, q, mp, ap, so, so, g, priors=pl)) for r, q, g, pl in zip(refs, curs, guesses, priors)]
    batch = c.multi_align_batch(refs, curs, mp, ap, guesses, so, so, priors=priors)
    again = c.multi_align_batch(refs, curs, mp, ap, guesses, so, so, priors=priors)
    return singles, batch, again


@pytest.mark.gpu
@pytest.mark.parametrize("setup", ["grouped", "per_pair", "slots3"])
@pytest.mark.parametrize("kind", ["4cam", "ragged"])
def test_rig_align_batch_equals_single(ctx, monkeypatch, setup, kind):
    """every record of the batch equals nicp_multi_align on that pair, byte for byte, through the grouped kernel, the
    per-pair kernel and with chunk boundaries inside the batch; a second batch run is byte-identical"""
    if setup == "grouped":
        monkeypatch.setenv("NICP_GROUP_MIN_AVG", "0")
    elif setup == "per_pair":
        monkeypatch.setenv("NICP_GROUP_MIN_AVG", "1000")
    else:
        monkeypatch.setenv("NICP_BATCH_SLOTS", "3")
    c = capi.Context(0, verify=ctx.verify)
    singles, batch, again = _align_case(c, kind)
    for i, s in enumerate(singles):
        assert batch[i].tobytes() == s, i
    assert batch.tobytes() == again.tobytes()
    assert (batch["status"] == 0).all() and (batch["inliers"] > 0).all()
    assert singles[0] != singles[1]  # the prior of pair 1 changed its result
    c.close()


@pytest.mark.gpu
def test_rig_batches_at_config5_full_size():
    """BASELINE config 5 at full size (4 x 1280x960, composite 1280 x 3840), default build: 3 rig frames prepared from raw
    in one call, 4 pairs aligned in one batch; records equal the single calls, poses recovered"""
    c = capi.Context(0)
    cams = synth.make_rig(4, 1280, 960)
    mp = capi.make_multi_projector(cams)
    assert capi.multi_image_size(mp) == (1280, 3840)
    sp = capi.make_stats_params(0.1, 10, 30, 50, 0.2, 0.02)
    poseA = synth.make_pose((0.1, -0.05, 0.2), (0, 1, 0), 10.0)
    poses = [poseA, poseA @ synth.make_pose((0.03, -0.01, 0.04), (0.2, 1.0, 0.1), 2.0),
             poseA @ synth.make_pose((-0.02, 0.01, 0.03), (0.1, 1.0, -0.2), -1.5)]
    frames = [render_raw_frame(p, cams, 1, 90 + f) for f, p in enumerate(poses)]
    clouds = c.multi_raw_depth_to_cloud_batch(frames, mp, sp)
    assert min(cl.size() for cl in clouds) > 4_000_000
    pairs = [(0, 1), (1, 0), (0, 2), (2, 1)]
    refs = [clouds[r] for r, _ in pairs]
    curs = [clouds[q] for _, q in pairs]
    gts = [np.linalg.inv(poses[r]) @ poses[q] for r, q in pairs]
    rng = np.random.default_rng(4)
    guesses = np.stack([gt @ synth.perturbed_pose(rng, np.eye(4), 0.01, 1.0) for gt in gts]).astype(np.float32)
    ap = capi.make_align_params(1.0, 0.95, 0.02, 1.3, 9e3, True, 10, 1)
    batch = c.multi_align_batch(refs, curs, mp, ap, guesses)
    for i, (r, q) in enumerate(zip(refs, curs)):
        assert batch[i].tobytes() == bytes(c.multi_align(r, q, mp, ap, guess=guesses[i])), i
        T = batch["T"][i].reshape(4, 4).T.astype(np.float64)
        dR = T[:3, :3].T @ gts[i][:3, :3]
        ang = np.arccos(np.clip((np.trace(dR) - 1) / 2, -1, 1))
        assert ang < 5e-3 and np.abs(T[:3, 3] - gts[i][:3, 3]).max() < 1e-2, (i, ang)
    c.close()

"""Rig loop closure over the workers of a shard pool (nicp_multi_align_frames_sharded): raw rig frames in, records out.
Every record must equal nicp_multi_align on the clouds nicp_multi_raw_depth_to_cloud_batch builds from its two frames,
byte for byte, whatever the device list, the workers per device and the per-worker frame cap (NICP_SHARD_FRAMES)."""
import ctypes as C

import numpy as np
import pytest

from conftest import CONF_1_4
from g2o_frontend_b200 import capi, synth
from test_rig_batch import make_cams, render_raw_frame, rig_poses

SP = (0.1, 3, 6, 10, 0.2, 0.02)  # stats parameters of the small test rigs (test_rig_batch)


@pytest.fixture(scope="module", params=["verify", "default"])
def verify(request):
    return request.param == "verify"


def _rig_case(kind, step, pairs=None):
    """2 current rig frames (0, 1) x 4 candidates (2..5), current-major unless pairs are given, with a sensor offset,
    guesses near the truth and priors on some pairs"""
    cams = make_cams(kind)
    mp = capi.make_multi_projector(cams)
    sp = capi.make_stats_params(*SP)
    so = synth.make_pose((0.05, 0.0, 0.1), (1.0, 0.2, 0.0), 3.0).astype(np.float32)
    poses = rig_poses(6, 23)
    frames = [render_raw_frame(p, cams, step, 70 + 5 * f) for f, p in enumerate(poses)]
    if pairs is None:
        pairs = [(r, c) for c in (0, 1) for r in (2, 3, 4, 5)]
    rng = np.random.default_rng(7)
    guesses = np.stack([synth.perturbed_pose(rng, np.linalg.inv(poses[r]) @ poses[c], 0.01, 0.5)
                        for r, c in pairs]).astype(np.float32)
    mean = synth.make_pose((0.05, -0.03, 0.08), (0.1, 1.0, 0.3), 3.0).astype(np.float32)
    refT = synth.make_pose((0.2, 0.1, -0.1), (1.0, 0.2, 0.1), 5.0).astype(np.float32)
    info = (np.diag([2e5, 1e5, 3e5, 5e6, 4e6, 6e6]) + 1e3).astype(np.float32)
    priors = [[] for _ in pairs]
    priors[1] = [capi.make_prior(0, mean, info, None)]
    priors[len(pairs) // 2] = [capi.make_prior(1, mean, info, refT)]
    priors[-1] = [capi.make_prior(0, mean, info, None), capi.make_prior(1, mean, info * 0.5, refT)]
    ap = capi.make_align_params(0.5, 0.95, 0.02, 1.3, 9e3, True, 10, 1)
    return dict(frames=frames, mp=mp, sp=sp, so=so, ref=[r for r, _ in pairs], cur=[c for _, c in pairs],
                guesses=guesses, priors=priors, ap=ap, step=step)


def _singles(case, verify):
    """the records of nicp_multi_align on clouds from one nicp_multi_raw_depth_to_cloud_batch call on a plain context"""
    c = capi.Context(0, verify=verify)
    clouds = c.multi_raw_depth_to_cloud_batch(case["frames"], case["mp"], case["sp"], step=case["step"],
                                              sensor_offset=case["so"])
    out = [bytes(c.multi_align(clouds[r], clouds[q], case["mp"], case["ap"], case["so"], case["so"], g, priors=pl))
           for r, q, g, pl in zip(case["ref"], case["cur"], case["guesses"], case["priors"])]
    c.close()
    return out


def _run(pool, case):
    return pool.multi_align_frames(case["frames"], case["mp"], case["sp"], case["ref"], case["cur"], case["guesses"],
                                   case["ap"], priors=case["priors"], step=case["step"], sensor_offset=case["so"])


def _check_pools(case, singles, device_lists, verify=False):
    for devs in device_lists:
        pool = capi.ShardPool(devs, verify=verify)
        recs = _run(pool, case)
        again = _run(pool, case)  # the rig cloud cache is reused
        pool.close()
        for i, s in enumerate(singles):
            assert recs[i].tobytes() == s, (devs, i)
        assert again.tobytes() == recs.tobytes(), devs
        assert (recs["status"] == 0).all() and (recs["inliers"] > 0).all(), devs


@pytest.mark.parametrize("v", [False, True])
def test_null_arguments_are_rejected(v):
    """no pool, projector or parameters: status 1 before any device is touched"""
    L = capi.load(v)
    N, f0 = None, C.c_float(0)
    assert L.nicp_multi_align_frames_sharded(N, 2, N, N, N, C.c_float(0.001), 1, C.c_float(0.01), N, N, N, 1, N, N, N, N, N,
                                             N, f0, N) == 1
    assert L.nicp_multi_align_frames_sharded(N, 0, N, N, N, C.c_float(0.001), 1, C.c_float(0.01), N, N, N, 0, N, N, N, N, N,
                                             N, f0, N) == 1


@pytest.mark.gpu
@pytest.mark.parametrize("kind,step", [("4cam", 1), ("4cam", 2), ("ragged", 1), ("ragged", 2)])
def test_rig_sharded_equals_single_calls(verify, kind, step):
    """one, two and three workers on GPU 0: every record equals nicp_multi_align on that pair, byte for byte; a second
    call on the same pool gives the same bytes"""
    case = _rig_case(kind, step)
    singles = _singles(case, verify)
    assert singles[0] != singles[1]  # the prior of pair 1 changed its result
    _check_pools(case, singles, [[0], [0, 0], [0, 0, 0]], verify)


@pytest.mark.gpu
@pytest.mark.parametrize("cap", ["2", "3"])
def test_frame_cap_windows_change_no_record(verify, monkeypatch, cap):
    """NICP_SHARD_FRAMES = 2 and 3 cut the blocks into windows of a few frames: a self-pair, a window boundary inside the
    pairs of one current frame, frames evicted and built again; the records are those of the default cap"""
    pairs = [(2, 0), (3, 0), (0, 0), (4, 0), (5, 0), (2, 1), (3, 1), (1, 1), (4, 1), (5, 1), (2, 0)]
    case = _rig_case("4cam", 1, pairs)
    singles = _singles(case, verify)
    default = []
    for devs in ([0], [0, 0]):
        pool = capi.ShardPool(devs, verify=verify)
        default.append(_run(pool, case).tobytes())
        pool.close()
    monkeypatch.setenv("NICP_SHARD_FRAMES", cap)  # read when a pool is created
    for devs, d in zip(([0], [0, 0]), default):
        pool = capi.ShardPool(devs, verify=verify)
        recs = _run(pool, case)
        assert recs.tobytes() == d, devs
        assert _run(pool, case).tobytes() == d, devs
        pool.close()
        for i, s in enumerate(singles):
            assert recs[i].tobytes() == s, (devs, i)


def _pinhole_case():
    """3 currents x 4 candidates at 160x120 for nicp_align_frames_sharded"""
    step = 4
    rows, cols = 480 // step, 640 // step
    K = synth.scaled_K(synth.K_KINECT, 1.0 / step)
    rng = np.random.default_rng(13)
    poses = [synth.perturbed_pose(rng, np.eye(4), 0.15, 4.0) for _ in range(7)]
    raws = [synth.render_depth_u16(p, seed=50 + i) for i, p in enumerate(poses)]
    ref_frame, cur_frame, guesses = [], [], []
    for c in (0, 1, 2):
        for r in (3, 4, 5, 6):
            ref_frame.append(r)
            cur_frame.append(c)
            guesses.append(synth.perturbed_pose(rng, np.linalg.inv(poses[r]) @ poses[c], 0.02, 1.0))
    conf = CONF_1_4
    proj = capi.make_projector(K, rows, cols, conf["minD"], conf["maxD"])
    sp = capi.make_stats_params(conf["worldRadius"], conf["minImageRadius"], conf["maxImageRadius"], conf["minPoints"],
                                conf["curvatureThreshold"], conf["omegaCurvatureThreshold"])
    ap = capi.make_align_params(conf["inlierDistanceThreshold"], conf["inlierNormalAngularThreshold"],
                                conf["flatCurvatureThreshold"], conf["inlierCurvatureRatioThreshold"], conf["inlierMaxChi2"],
                                True, 10, 1)
    return lambda pool: pool.align_frames(raws, proj, sp, ref_frame, cur_frame, np.stack(guesses).astype(np.float32), ap,
                                          step=step)


@pytest.mark.gpu
def test_rig_calls_leave_the_pinhole_entry_unchanged():
    """pinhole, rig, pinhole on one pool: both pinhole calls give the records of a fresh pool"""
    pinhole = _pinhole_case()
    fresh = capi.ShardPool([0, 0])
    expect = pinhole(fresh).tobytes()
    fresh.close()
    pool = capi.ShardPool([0, 0])
    assert pinhole(pool).tobytes() == expect
    case = _rig_case("4cam", 1)
    _run(pool, case)
    assert pinhole(pool).tobytes() == expect
    pool.close()


@pytest.mark.gpu
def test_bad_input_is_rejected_before_any_worker(verify):
    case = _rig_case("ragged", 1)
    pool = capi.ShardPool([0, 0], verify=verify)
    L = pool.L
    nc = case["mp"].num_cameras
    frames = case["frames"]
    n = len(case["ref"])

    def call(frames=frames, ref=case["ref"], offs=None, null_image=None):
        imgs = [np.ascontiguousarray(im) for fr in frames for im in fr]
        RA = (C.c_void_p * len(imgs))(*[im.ctypes.data for im in imgs])
        if null_image is not None:
            RA[null_image] = None
        rr = np.array([im.shape[0] for im in frames[0]], np.int32)
        rc = np.array([im.shape[1] for im in frames[0]], np.int32)
        rf = np.ascontiguousarray(ref, np.int32)
        cf = np.ascontiguousarray(case["cur"], np.int32)
        so = capi.colmajor(case["so"])
        parr = (capi.Prior * 2)(*case["priors"][-1])
        res = np.zeros(n, capi.RESULT_DTYPE)
        status = L.nicp_multi_align_frames_sharded(
            pool.handle, len(frames), RA, capi._iptr(rr), capi._iptr(rc), C.c_float(0.001), 1, C.c_float(0.01),
            C.byref(case["mp"]), C.byref(case["sp"]), capi._fptr(so), n, capi._iptr(rf), capi._iptr(cf), None, parr,
            None if offs is None else capi._iptr(offs), C.byref(case["ap"]), C.c_float(50.0),
            res.ctypes.data_as(C.POINTER(capi.AlignResult)))
        return status, L.nicp_last_error().decode()

    assert call()[0] == 0
    ref = list(case["ref"])
    ref[5] = len(frames)
    assert call(ref=ref) == (1, "pair 5 references frame 6 / 1 outside [0, 6)")
    assert call(null_image=3 * nc + 1) == (1, "null raw image of camera 1 in frame 3")
    wrong = [list(fr) for fr in frames]
    for fr in wrong:
        fr[2] = np.zeros((fr[2].shape[0], fr[2].shape[1] + 1), np.uint16)
    status, msg = call(frames=wrong)
    assert status == 1 and msg.startswith("camera 2: raw image"), msg
    offs = np.array([0, 0, 1, 2, 2, 1, 1, 2, 2], np.int32)[:n + 1]
    assert call(offs=offs) == (1, "prior_offsets decrease at pair 4 (2 -> 1)")
    pool.close()


@pytest.mark.gpu
def test_rig_sharded_over_the_visible_gpus():
    """the case of the equality test over every GPU the box has (two workers on GPU 0 when it has one)"""
    import torch
    n = torch.cuda.device_count()
    lists = [list(range(n)), list(range(n))[::-1] + [0]] if n >= 2 else [[0, 0]]
    case = _rig_case("4cam", 1)
    _check_pools(case, _singles(case, False), lists)


@pytest.mark.gpu
def test_rig_sharded_at_config5_full_size():
    """BASELINE config 5 at full size (4 x 1280x960, composite 1280 x 3840), default build: 3 rig frames, 4 pairs over two
    workers; records equal the single calls, poses recovered"""
    import torch
    cams = synth.make_rig(4, 1280, 960)
    mp = capi.make_multi_projector(cams)
    assert capi.multi_image_size(mp) == (1280, 3840)
    sp = capi.make_stats_params(0.1, 10, 30, 50, 0.2, 0.02)
    poseA = synth.make_pose((0.1, -0.05, 0.2), (0, 1, 0), 10.0)
    poses = [poseA, poseA @ synth.make_pose((0.03, -0.01, 0.04), (0.2, 1.0, 0.1), 2.0),
             poseA @ synth.make_pose((-0.02, 0.01, 0.03), (0.1, 1.0, -0.2), -1.5)]
    frames = [render_raw_frame(p, cams, 1, 90 + f) for f, p in enumerate(poses)]
    pairs = [(0, 1), (1, 0), (0, 2), (2, 1)]
    gts = [np.linalg.inv(poses[r]) @ poses[q] for r, q in pairs]
    rng = np.random.default_rng(4)
    guesses = np.stack([gt @ synth.perturbed_pose(rng, np.eye(4), 0.01, 1.0) for gt in gts]).astype(np.float32)
    ap = capi.make_align_params(1.0, 0.95, 0.02, 1.3, 9e3, True, 10, 1)
    pool = capi.ShardPool([0, 1] if torch.cuda.device_count() >= 2 else [0, 0])
    recs = pool.multi_align_frames(frames, mp, sp, [r for r, _ in pairs], [q for _, q in pairs], guesses, ap)
    pool.close()
    c = capi.Context(0)
    clouds = c.multi_raw_depth_to_cloud_batch(frames, mp, sp)
    for i, (r, q) in enumerate(pairs):
        assert recs[i].tobytes() == bytes(c.multi_align(clouds[r], clouds[q], mp, ap, guess=guesses[i])), i
        T = recs["T"][i].reshape(4, 4).T.astype(np.float64)
        dR = T[:3, :3].T @ gts[i][:3, :3]
        ang = np.arccos(np.clip((np.trace(dR) - 1) / 2, -1, 1))
        assert ang < 5e-3 and np.abs(T[:3, 3] - gts[i][:3, 3]).max() < 1e-2, (i, ang)
    c.close()

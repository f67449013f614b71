"""Loop-closure frames resident on a shard pool across calls (nicp_frame_store_*): raw frames added once under 64-bit ids,
pairs aligned by id.  Every record must equal nicp_align / nicp_multi_align on the clouds the batched prep builds from its
two frames, byte for byte, whatever the device list, the frame cap, the store's history or what is resident; the counters
show which clouds were prepared and which were found resident."""
import ctypes as C

import numpy as np
import pytest

from conftest import CONF_1_1
from g2o_frontend_b200 import capi, synth
from test_rig_sharded import _pinhole_case as _sharded_pinhole_case, _pinhole_run, _rig_case, _run

POOLS = ([0], [0, 0], [0, 0, 0])
BASE_ID = 1 << 40  # ids are 64-bit: frame f of a case is stored as BASE_ID + 7 f


@pytest.fixture(scope="module", params=["verify", "default"])
def verify(request):
    return request.param == "verify"


def _pinhole_case(step):
    """7 pinhole frames at 640x480 / step with a sensor offset: currents 0, 1, 2 x candidates 3..6, current-major, guesses
    near the truth and priors on some pairs"""
    rows, cols = 480 // step, 640 // step
    K = synth.scaled_K(synth.K_KINECT, 1.0 / step)
    rng = np.random.default_rng(29 + step)
    poses = [synth.perturbed_pose(rng, np.eye(4), 0.15, 4.0) for _ in range(7)]
    frames = [synth.render_depth_u16(p, seed=60 + i) for i, p in enumerate(poses)]
    pairs = [(r, c) for c in (0, 1, 2) for r in (3, 4, 5, 6)]
    guesses = np.stack([synth.perturbed_pose(rng, np.linalg.inv(poses[r]) @ poses[c], 0.02, 1.0)
                        for r, c in pairs]).astype(np.float32)
    mean = synth.make_pose((0.04, -0.02, 0.05), (0.1, 1.0, 0.3), 2.0).astype(np.float32)
    refT = synth.make_pose((0.2, 0.1, -0.1), (1.0, 0.2, 0.1), 5.0).astype(np.float32)
    info = (np.diag([2e5, 1e5, 3e5, 5e6, 4e6, 6e6]) + 1e3).astype(np.float32)
    priors = [[] for _ in pairs]
    priors[1] = [capi.make_prior(0, mean, info, None)]
    priors[6] = [capi.make_prior(1, mean, info, refT)]
    priors[-1] = [capi.make_prior(0, mean, info, None), capi.make_prior(1, mean, info * 0.5, refT)]
    c = CONF_1_1
    proj = capi.make_projector(K, rows, cols, c["minD"], c["maxD"])
    sp = capi.make_stats_params(c["worldRadius"], c["minImageRadius"], c["maxImageRadius"], c["minPoints"],
                                c["curvatureThreshold"], c["omegaCurvatureThreshold"])
    ap = capi.make_align_params(c["inlierDistanceThreshold"], c["inlierNormalAngularThreshold"], c["flatCurvatureThreshold"],
                                c["inlierCurvatureRatioThreshold"], c["inlierMaxChi2"], True, 10, 1)
    so = synth.make_pose((0.05, 0.0, 0.1), (1.0, 0.2, 0.0), 3.0).astype(np.float32)
    return dict(rig=False, camera=proj, raw_shape=frames[0].shape, frames=frames, sp=sp, so=so, step=step,
                ref=[r for r, _ in pairs], cur=[q for _, q in pairs], guesses=guesses, priors=priors, ap=ap)


def _rig(kind, pairs=None):
    case = _rig_case(kind, 1, pairs)
    return dict(case, rig=True, camera=case["mp"], raw_shape=[im.shape for im in case["frames"][0]])


def _case(kind):
    return _pinhole_case(int(kind[-1])) if kind.startswith("pinhole") else _rig(kind)


def ids_of(frames):
    return [BASE_ID + 7 * f for f in frames]


def _clouds(c, case, frames=None):
    frames = case["frames"] if frames is None else frames
    if case["rig"]:
        return c.multi_raw_depth_to_cloud_batch(frames, case["camera"], case["sp"], step=case["step"], sensor_offset=case["so"])
    return c.raw_depth_to_cloud_batch(frames, case["camera"], case["sp"], step=case["step"], sensor_offset=case["so"])


def _single(c, case, ref_cloud, cur_cloud, i):
    align = c.multi_align if case["rig"] else c.align
    return bytes(align(ref_cloud, cur_cloud, case["camera"], case["ap"], case["so"], case["so"], case["guesses"][i],
                       priors=case["priors"][i]))


def _singles(case, verify):
    """the records of nicp_align / nicp_multi_align on clouds from one batched prep call on a plain context"""
    c = capi.Context(0, verify=verify)
    clouds = _clouds(c, case)
    out = [_single(c, case, clouds[r], clouds[q], i) for i, (r, q) in enumerate(zip(case["ref"], case["cur"]))]
    c.close()
    return out


def _store(pool, case, frames=None):
    st = capi.FrameStore(pool, case["camera"], case["sp"], case["raw_shape"], step=case["step"], sensor_offset=case["so"])
    frames = range(len(case["frames"])) if frames is None else frames
    st.add(ids_of(frames), [case["frames"][f] for f in frames])
    return st


def _align(st, case, sel=None):
    sel = range(len(case["ref"])) if sel is None else list(sel)
    return st.align(ids_of([case["ref"][i] for i in sel]), ids_of([case["cur"][i] for i in sel]),
                    case["guesses"][list(sel)], case["ap"], priors=[case["priors"][i] for i in sel])


def _blocks(n, G):
    return [range(g * n // G, (g + 1) * n // G) for g in range(G)]


@pytest.mark.parametrize("v", [False, True])
def test_null_handles_and_arguments_are_rejected(v):
    """no store, pool, projector or parameters: status 1 (size -1) before any device is touched"""
    L = capi.load(v)
    L.nicp_frame_store_destroy.restype = None
    N, f0 = None, C.c_float(0)
    h = C.c_void_p(1)
    assert L.nicp_frame_store_create(N, 480, 640, C.c_float(0.001), 1, C.c_float(0.01), N, N, N, C.byref(h)) == 1
    assert not h
    assert L.nicp_frame_store_create(N, 480, 640, C.c_float(0.001), 1, C.c_float(0.01), N, N, N, N) == 1
    h = C.c_void_p(1)
    assert L.nicp_multi_frame_store_create(N, N, N, C.c_float(0.001), 1, C.c_float(0.01), N, N, N, C.byref(h)) == 1
    assert not h
    assert L.nicp_multi_frame_store_create(N, N, N, C.c_float(0.001), 1, C.c_float(0.01), N, N, N, N) == 1
    assert L.nicp_frame_store_add(N, 1, N, N) == 1
    assert L.nicp_frame_store_add(N, 0, N, N) == 1
    assert L.nicp_frame_store_remove(N, 1, N) == 1
    assert L.nicp_frame_store_size(N) == -1
    assert L.nicp_frame_store_align(N, 1, N, N, N, N, N, N, f0, N) == 1
    assert L.nicp_frame_store_align(N, 0, N, N, N, N, N, N, f0, N) == 1
    assert L.nicp_frame_store_counters(N, N, N) == 1
    L.nicp_frame_store_destroy(N)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["pinhole1", "pinhole2", "4cam", "ragged"])
def test_store_records_equal_single_calls(verify, kind):
    """one, two and three workers on GPU 0: every record equals the single call on that pair, priors included, byte for
    byte; a second call gives the same bytes and prepares nothing"""
    case = _case(kind)
    singles = _singles(case, verify)
    for devs in POOLS:
        pool = capi.ShardPool(devs, verify=verify)
        st = _store(pool, case)
        recs = _align(st, case)
        built, reused = st.counters()
        again = _align(st, case)
        assert st.counters() == (built, reused + built), devs  # every frame of every block was resident
        st.close()
        pool.close()
        for i, s in enumerate(singles):
            assert recs[i].tobytes() == s, (devs, i)
        assert again.tobytes() == recs.tobytes(), devs
        assert (recs["status"] == 0).all() and (recs["inliers"] > 0).all(), devs


@pytest.mark.gpu
def test_resident_clouds_are_reused(verify):
    """one worker: the same pairs again build nothing; two new frames aligned against resident candidates build exactly
    two.  Several workers build at most the distinct frames of each block."""
    case = _pinhole_case(2)
    singles = _singles(case, verify)
    first = [i for i, q in enumerate(case["cur"]) if q == 2]   # current 2 x candidates 3..6
    later = [i for i, q in enumerate(case["cur"]) if q != 2]   # currents 0, 1 x the same candidates
    pool = capi.ShardPool([0], verify=verify)
    st = _store(pool, case, [2, 3, 4, 5, 6])
    recs = _align(st, case, first)
    assert st.counters() == (5, 0)
    again = _align(st, case, first)
    assert st.counters() == (5, 5)
    assert again.tobytes() == recs.tobytes()
    st.add(ids_of([0, 1]), [case["frames"][0], case["frames"][1]])
    assert st.size() == 7
    new = _align(st, case, later)
    assert st.counters() == (7, 9)  # 2 built, the 4 candidates found
    st.close()
    pool.close()
    for k, i in enumerate(first):
        assert recs[k].tobytes() == singles[i], i
    for k, i in enumerate(later):
        assert new[k].tobytes() == singles[i], i

    n = len(case["ref"])
    for devs in POOLS[1:]:
        pool = capi.ShardPool(devs, verify=verify)
        st = _store(pool, case)
        recs = _align(st, case)
        bound = sum(len({case["ref"][i] for i in b} | {case["cur"][i] for i in b}) for b in _blocks(n, len(devs)))
        built, reused = st.counters()
        assert built <= bound and built + reused == bound, (devs, built, reused, bound)
        st.close()
        pool.close()
        for i, s in enumerate(singles):
            assert recs[i].tobytes() == s, (devs, i)


@pytest.mark.gpu
@pytest.mark.parametrize("cap", ["2", "3"])
def test_frame_cap_evicts_without_changing_a_record(verify, monkeypatch, cap):
    """NICP_SHARD_FRAMES = 2 and 3 (read when the pool is created): a self-pair, a window boundary inside the pairs of one
    current frame, frames evicted and built again within a call and across calls; the records are those of the default cap
    and of the single calls"""
    pairs = [(2, 0), (3, 0), (0, 0), (4, 0), (5, 0), (2, 1), (3, 1), (1, 1), (4, 1), (5, 1), (2, 0)]
    case = _rig("4cam", pairs)
    singles = _singles(case, verify)
    default = {}
    for devs in POOLS:
        pool = capi.ShardPool(devs, verify=verify)
        st = _store(pool, case)
        default[len(devs)] = _align(st, case).tobytes()
        st.close()
        pool.close()
    monkeypatch.setenv("NICP_SHARD_FRAMES", cap)
    n = len(pairs)
    for devs in POOLS:
        pool = capi.ShardPool(devs, verify=verify)
        st = _store(pool, case)
        recs = _align(st, case)
        assert recs.tobytes() == default[len(devs)], devs
        built, _ = st.counters()
        distinct = sum(len({pairs[i][0] for i in b} | {pairs[i][1] for i in b}) for b in _blocks(n, len(devs)))
        assert built >= distinct, (devs, built, distinct)
        if len(devs) < 3:  # frame 2 opens and closes a block: evicted and built again within the call
            assert built > distinct, (devs, built, distinct)
        assert _align(st, case).tobytes() == recs.tobytes(), devs
        assert st.counters()[0] > built, devs  # the cap is too small for the second call to find everything
        st.close()
        pool.close()
        for i, s in enumerate(singles):
            assert recs[i].tobytes() == s, (devs, i)


@pytest.mark.gpu
def test_least_recently_used_slot_is_evicted(verify, monkeypatch):
    """NICP_SHARD_FRAMES = 3, one worker, frames A B C D: (A, B), then (A, A), then (C, D), then (A, C).  C takes the third
    slot; D must evict B, which was last used before A, so (A, C) finds both frames resident.  Evicting any other slot
    would rebuild A in the last call."""
    case = _pinhole_case(2)
    A, B, Cf, D = 3, 4, 5, 6
    ctx = capi.Context(0, verify=verify)
    clouds = _clouds(ctx, case)
    expect = bytes(ctx.align(clouds[A], clouds[Cf], case["camera"], case["ap"], case["so"], case["so"]))
    ctx.close()
    monkeypatch.setenv("NICP_SHARD_FRAMES", "3")
    pool = capi.ShardPool([0], verify=verify)
    st = _store(pool, case, [A, B, Cf, D])
    counters = []
    for r, q in ((A, B), (A, A), (Cf, D), (A, Cf)):
        recs = st.align(ids_of([r]), ids_of([q]), None, case["ap"])
        counters.append(st.counters())
    st.close()
    pool.close()
    assert counters == [(2, 0), (2, 1), (4, 1), (4, 3)]
    assert recs[0].tobytes() == expect


@pytest.mark.gpu
def test_removed_and_re_added_id_is_built_from_its_new_frame(verify):
    """remove a candidate's id, add it again with another image: every worker that held its cloud prepares it again, and the
    records are those of the new image, not of the old one"""
    case = _pinhole_case(2)
    singles = _singles(case, verify)
    c = capi.Context(0, verify=verify)
    clouds = _clouds(c, case)
    sel = [i for i, r in enumerate(case["ref"]) if r == 3]  # (3, 0), (3, 1), (3, 2): in the blocks of several workers
    expect = [_single(c, case, clouds[6], clouds[case["cur"][i]], i) for i in sel]
    c.close()
    for devs in POOLS:
        pool = capi.ShardPool(devs, verify=verify)
        st = _store(pool, case, [0, 1, 2, 3])
        old = _align(st, case, sel)
        st.remove(ids_of([3]))
        assert st.size() == 3
        with pytest.raises(capi.NicpError, match="not in the store"):
            _align(st, case, sel)
        st.add(ids_of([3]), [case["frames"][6]])
        new = _align(st, case, sel)
        st.close()
        pool.close()
        for k, i in enumerate(sel):
            assert old[k].tobytes() == singles[i], (devs, i)
            assert new[k].tobytes() == expect[k], (devs, i)
            assert new[k].tobytes() != old[k].tobytes(), (devs, i)


@pytest.mark.gpu
def test_store_calls_and_sharded_entries_share_a_pool(verify):
    """store, pinhole sharded, rig sharded, store calls interleaved on one pool: each gets the records it gets alone"""
    case = _pinhole_case(2)
    pinhole = _sharded_pinhole_case()
    rig = _rig_case("4cam", 1)
    alone = capi.ShardPool([0, 0], verify=verify)
    st = _store(alone, case)
    expect_store = _align(st, case).tobytes()
    st.close()
    expect_pinhole = _pinhole_run(alone, pinhole).tobytes()
    expect_rig = _run(alone, rig).tobytes()
    alone.close()
    pool = capi.ShardPool([0, 0], verify=verify)
    st = _store(pool, case)
    assert _pinhole_run(pool, pinhole).tobytes() == expect_pinhole
    assert _align(st, case).tobytes() == expect_store
    assert _run(pool, rig).tobytes() == expect_rig
    built = st.counters()[0]
    assert _align(st, case).tobytes() == expect_store
    assert st.counters()[0] == built  # the sharded calls left the store's clouds alone
    assert _pinhole_run(pool, pinhole).tobytes() == expect_pinhole
    assert _run(pool, rig).tobytes() == expect_rig
    st.close()
    pool.close()


@pytest.mark.gpu
def test_raw_images_of_another_shape_are_refused(verify):
    """add copies the store's raw size from every pointer: an image of another shape (an already-stepped pinhole frame, a
    rig frame with two cameras swapped or one missing) raises before the library is called and adds nothing"""
    pool = capi.ShardPool([0], verify=verify)
    case = _pinhole_case(2)
    st = _store(pool, case, [0])
    stepped = np.ascontiguousarray(case["frames"][1][::2, ::2])
    with pytest.raises(ValueError, match=r"frame 1, camera 0: raw image of shape \(240, 320\)"):
        st.add(ids_of([1, 2]), [case["frames"][2], stepped])
    assert st.size() == 1 and st.counters() == (0, 0)
    st.close()
    rig = _rig("ragged")
    st = _store(pool, rig, [0])
    swapped = list(rig["frames"][1])
    swapped[0], swapped[1] = swapped[1], swapped[0]  # 40x48 and 48x64
    assert swapped[0].shape != rig["frames"][1][0].shape
    with pytest.raises(ValueError, match="frame 0, camera 0: raw image of shape"):
        st.add(ids_of([1]), [swapped])
    with pytest.raises(ValueError, match="frame 0 has 2 images for 3 cameras"):
        st.add(ids_of([1]), [rig["frames"][1][:2]])
    assert st.size() == 1
    st.add(ids_of([1]), [rig["frames"][1]])
    assert st.size() == 2
    st.close()
    pool.close()


@pytest.mark.gpu
def test_bad_input_is_rejected_and_changes_nothing(verify):
    case = _pinhole_case(2)
    pool = capi.ShardPool([0, 0], verify=verify)
    L = pool.L
    msg = lambda: L.nicp_last_error().decode()  # noqa: E731
    # frame descriptions that do not scale to the projector
    proj, sp = case["camera"], case["sp"]
    with pytest.raises(capi.NicpError, match="does not match the scaled raw image"):
        capi.FrameStore(pool, proj, sp, (480, 644), step=2)
    rig = _rig("ragged")
    shapes = [(r, c + 1) if k == 2 else (r, c) for k, (r, c) in enumerate(rig["raw_shape"])]
    with pytest.raises(capi.NicpError, match="camera 2: raw image"):
        capi.FrameStore(pool, rig["camera"], rig["sp"], shapes)

    st = _store(pool, case, [0, 1, 3, 4])
    recs = _align(st, case, [0, 1, 4, 5])
    state = (st.size(), st.counters())
    assert state[0] == 4

    def unchanged():
        assert (st.size(), st.counters()) == state

    frame = case["frames"][5]
    with pytest.raises(capi.NicpError, match="frame id %d is added twice" % ids_of([5])[0]):
        st.add(ids_of([5, 5]), [frame, frame])
    unchanged()
    with pytest.raises(capi.NicpError, match="frame id %d is already in the store" % ids_of([3])[0]):
        st.add(ids_of([5, 3]), [frame, frame])
    unchanged()
    RA = (C.c_void_p * 2)(frame.ctypes.data, None)
    ids = np.array(ids_of([5, 6]), np.int64)
    assert L.nicp_frame_store_add(st.handle, 2, capi._llptr(ids), RA) == 1
    assert msg() == "null raw image of camera 0 in frame 1"
    unchanged()
    with pytest.raises(capi.NicpError, match="frame id %d is not in the store" % ids_of([6])[0]):
        st.remove(ids_of([0, 6]))
    unchanged()
    with pytest.raises(capi.NicpError, match="frame id %d is removed twice" % ids_of([0])[0]):
        st.remove(ids_of([0, 0]))
    unchanged()
    with pytest.raises(capi.NicpError, match="pair 1 references frame id %d, which is not in the store" % ids_of([6])[0]):
        st.align(ids_of([3, 6]), ids_of([0, 0]), None, case["ap"])
    unchanged()
    # prior_offsets that decrease
    n = 4
    rf, cf = np.array(ids_of([3, 4, 3, 4]), np.int64), np.array(ids_of([0, 0, 1, 1]), np.int64)
    offs = np.array([0, 1, 0, 1, 1], np.int32)
    parr = (capi.Prior * 1)(case["priors"][1][0])
    res = np.zeros(n, capi.RESULT_DTYPE)
    status = L.nicp_frame_store_align(st.handle, n, capi._llptr(rf), capi._llptr(cf), None, parr, capi._iptr(offs),
                                      C.byref(case["ap"]), C.c_float(50.0), res.ctypes.data_as(C.POINTER(capi.AlignResult)))
    assert (status, msg()) == (1, "prior_offsets decrease at pair 1 (1 -> 0)")
    unchanged()
    # n = 0 is a valid empty call
    st.add([], [])
    st.remove([])
    assert len(st.align([], [], None, case["ap"])) == 0
    unchanged()
    assert _align(st, case, [0, 1, 4, 5]).tobytes() == recs.tobytes()
    st.close()
    pool.close()


@pytest.mark.gpu
def test_store_outlived_by_nothing_after_its_pool_is_destroyed(verify):
    """destroying the pool releases the store's clouds; every later store call but destroy returns NICP_ERR_INVALID"""
    case = _pinhole_case(2)
    gone = "the frame store's shard pool has been destroyed"
    for devs in POOLS:
        pool = capi.ShardPool(devs, verify=verify)
        st = _store(pool, case, [0, 1, 3, 4])
        _align(st, case, [0, 1, 4, 5])
        pool.close()
        L = st.L
        with pytest.raises(capi.NicpError, match=gone):
            st.add(ids_of([5]), [case["frames"][5]])
        with pytest.raises(capi.NicpError, match=gone):
            st.remove(ids_of([0]))
        with pytest.raises(capi.NicpError, match=gone):
            _align(st, case, [0])
        with pytest.raises(capi.NicpError, match=gone):
            st.counters()
        assert st.size() == -1
        assert L.nicp_frame_store_add(st.handle, 0, None, None) == 1
        st.close()
        assert not st.handle

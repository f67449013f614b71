"""Batched keyframe tracking of independent depth sequences on a shard pool (nicp_tracker_*, capi.Tracker,
pwn::BatchTracker).  Every sequence must do exactly what pwn::SequentialTracker::processFrame does on its frames:
  - each record is byte-identical to nicp_raw_depth_to_cloud + nicp_align (nicp_multi_raw_depth_to_cloud_batch +
    nicp_multi_align for a rig) on the sequence's keyframe and frame, with the result's guess;
  - guess, global pose, keyframe flag and keyframe count equal a float32 restatement of processFrame's bookkeeping in the
    operation order of include/pwn/compat.h, bit for bit;
  - results do not depend on the worker count, on which other sequences a step lists or in which order, or on rejected
    calls made before it."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import CONF_1_1, CONF_1_4, ROOT
from g2o_frontend_b200 import capi, synth
from test_rig_batch import make_cams, render_raw_frame
from test_rig_sharded import SP as RIG_SP

POOLS = ([0], [0, 0], [0, 0, 0])
FRACTION = 0.6  # keyframe threshold that makes the synthetic sweeps switch keyframes (test_sequential_tracker_*)
# a pair without a single inlier: the batched alignment every tracker step runs (as nicp_align_batch and the sharded
# entries do) reports another Omega than nicp_align; every other field, and so the tracker's bookkeeping, is identical
ZERO_INLIER_FIELDS = ("omega",)
f32 = np.float32


@pytest.fixture(scope="module", params=["verify", "default"])
def verify(request):
    return request.param == "verify"


# ---- float32 restatement of SequentialTracker::processFrame's bookkeeping (include/pwn/tracker.h:54-99) ----------------
def iso_mul(A, B):
    """Isometry3f::operator* (compat.h): rows 0-2 of both operands, last row (0, 0, 0, 1)"""
    o = np.eye(4, dtype=f32)
    for r in range(3):
        for c in range(3):
            o[r, c] = (A[r, 0] * B[0, c] + A[r, 1] * B[1, c]) + A[r, 2] * B[2, c]
        o[r, 3] = ((A[r, 0] * B[0, 3] + A[r, 1] * B[1, 3]) + A[r, 2] * B[2, 3]) + A[r, 3]
    return o


def iso_inverse(A):
    """Isometry3f::inverse (compat.h): R^T, -(R^T t)"""
    o = np.eye(4, dtype=f32)
    o[:3, :3] = A[:3, :3].T
    for r in range(3):
        o[r, 3] = -((o[r, 0] * A[0, 3] + o[r, 1] * A[1, 3]) + o[r, 2] * A[2, 3])
    return o


def mat3_mul(A, B):
    """Matrix<3, 3>::operator* (compat.h): a sum from 0.0f over the inner index, ascending"""
    o = np.zeros((3, 3), f32)
    for r in range(3):
        for k in range(3):
            s = f32(0.0)
            for c in range(3):
                s = s + A[r, c] * B[c, k]
            o[r, k] = s
    return o


class SeqModel:
    """one sequence's SequentialTracker state"""

    def __init__(self):
        self.reset()

    def reset(self):
        self.has_key = False
        self.G = np.eye(4, dtype=f32)
        self.keyT = np.eye(4, dtype=f32)
        self.counter = 0
        self.nkey = 0

    def guess(self, odometry):
        g = iso_mul(iso_mul(iso_inverse(self.keyT), self.G), np.eye(4, dtype=f32) if odometry is None else odometry)
        g[3] = (0, 0, 0, 1)  # Aligner::setInitialGuess -> fixLastRow
        return g

    def frame(self, odometry, T, inliers, pixels, fraction):
        """-> (aligned, guess, keyframe); T / inliers are the alignment's, ignored for a first frame"""
        if not self.has_key:
            self.has_key, self.keyT = True, self.G.copy()
            self.nkey += 1
            self.counter += 1
            return False, np.eye(4, dtype=f32), True
        g = self.guess(odometry)
        self.G = iso_mul(self.keyT, T) if inliers > 0 else iso_mul(self.G, g)
        if self.counter % 50 == 0:
            R = self.G[:3, :3].copy()
            E = mat3_mul(R.T.copy(), R)
            for i in range(3):
                E[i, i] = E[i, i] - f32(1.0)
            self.G[:3, :3] = R - mat3_mul(R, E) * f32(0.5)
        self.G[3] = (0, 0, 0, 1)
        key = bool(f32(inliers) / f32(pixels) < f32(fraction))
        if key:
            self.keyT = self.G.copy()
            self.nkey += 1
        self.counter += 1
        return True, g, key


def cm(M):
    return capi.colmajor(M).view(np.uint32)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


# ---- synthetic sequences ---------------------------------------------------------------------------------------------
_FRAMES = {}


def sequence(i, n):
    """sequence i: n 640x480 frames of a camera sweeping far enough to switch keyframes (seed and sweep differ per i), and
    its true poses"""
    key = (i, n)
    if key not in _FRAMES:
        poses = synth.trajectory(n, seed=10 + i, step_t=0.02, step_deg=1.0)
        sweep = 0.8 + 0.2 * i
        poses = [p @ synth.make_pose((0.015 * sweep * k, 0, 0), (0, 1, 0), 1.2 * sweep * k) for k, p in enumerate(poses)]
        _FRAMES[key] = ([synth.render_depth_u16(p, seed=300 + 41 * i + k) for k, p in enumerate(poses)], poses)
    return _FRAMES[key]


def odometry_of(poses, seed):
    """frame k's initialGuess: the true motion from frame k - 1, perturbed"""
    rng = np.random.default_rng(seed)
    out = [np.eye(4, dtype=f32)]
    for k in range(1, len(poses)):
        out.append(synth.perturbed_pose(rng, np.linalg.inv(poses[k - 1]) @ poses[k], 0.005, 0.3).astype(f32))
    return out


def pinhole_params(step, distance=None):
    c = CONF_1_1 if step == 1 else CONF_1_4
    K = synth.scaled_K(synth.K_KINECT, f32(1.0) / f32(step))
    proj = capi.make_projector(K, 480 // step, 640 // step, c["minD"], c["maxD"])
    sp = capi.make_stats_params(c["worldRadius"], c["minImageRadius"], c["maxImageRadius"], c["minPoints"],
                                c["curvatureThreshold"], c["omegaCurvatureThreshold"])
    ap = capi.make_align_params(c["inlierDistanceThreshold"] if distance is None else distance,
                                c["inlierNormalAngularThreshold"], c["flatCurvatureThreshold"],
                                c["inlierCurvatureRatioThreshold"], c["inlierMaxChi2"], True, 10, 1)
    return proj, sp, ap


SENSOR_OFFSET = synth.make_pose((0.05, -0.02, 0.1), (0.3, 1.0, 0.2), 4.0).astype(f32)


def pinhole_case(step, lengths=(14, 18, 22, 26, 30), odometry_seq=3, distance=None):
    proj, sp, ap = pinhole_params(step, distance)
    seqs = [sequence(i, n) for i, n in enumerate(lengths)]
    frames = [s[0] for s in seqs]
    odo = [odometry_of(s[1], 7 + i) if i == odometry_seq else None for i, s in enumerate(seqs)]
    return dict(rig=False, camera=proj, sp=sp, ap=ap, step=step, raw_shape=(480, 640), frames=frames, odometry=odo,
                pixels=proj.rows * proj.cols)


def schedule(case, order=None):
    """the default schedule: step t lists every sequence that still has a frame t (reversed on odd t)"""
    n = max(len(f) for f in case["frames"])
    out = []
    for t in range(n):
        seqs = [s for s in range(len(case["frames"])) if t < len(case["frames"][s])]
        out.append([(s, t) for s in (seqs[::-1] if t % 2 else seqs)])
    return out


def make_tracker(pool, case, n_sequences, offset=None):
    return capi.Tracker(pool, case["camera"], case["sp"], case["ap"], case["raw_shape"], n_sequences, step=case["step"],
                        sensor_offset=offset, new_frame_inliers_fraction=FRACTION)


def run_steps(tr, case, steps, seq_map=None):
    """steps: lists of (tracker sequence, frame index); seq_map maps a tracker sequence to the case's sequence.  Returns
    {tracker sequence: [result, ...]} in frame order"""
    seq_map = seq_map or {}
    out = {}
    for st in steps:
        seqs = [s for s, _ in st]
        src = [seq_map.get(s, s) for s in seqs]
        frames = [case["frames"][q][t] for q, (_, t) in zip(src, st)]
        odo = [case["odometry"][q][t] if case["odometry"][q] is not None else np.eye(4, dtype=f32)
               for q, (_, t) in zip(src, st)]
        res = tr.step(seqs, frames, odo if any(case["odometry"][q] is not None for q in src) else None)
        for s, r in zip(seqs, res):
            out.setdefault(s, []).append(r.copy())
    return out


class Chain:
    """the single-call chain on a plain context: clouds from nicp_raw_depth_to_cloud (nicp_multi_raw_depth_to_cloud_batch
    for a rig), records from nicp_align (nicp_multi_align), cached per frame"""

    def __init__(self, case, verify, offset=None):
        self.case, self.offset = case, offset
        self.ctx = capi.Context(0, verify=verify)
        self.clouds = {}

    def cloud(self, q, t):
        if (q, t) not in self.clouds:
            c = self.case
            if c["rig"]:
                self.clouds[(q, t)] = self.ctx.multi_raw_depth_to_cloud_batch([c["frames"][q][t]], c["camera"], c["sp"],
                                                                              step=c["step"], sensor_offset=self.offset)[0]
            else:
                self.clouds[(q, t)] = self.ctx.raw_depth_to_cloud(c["frames"][q][t], c["camera"], c["sp"], step=c["step"],
                                                                  sensor_offset=self.offset)[0]
        return self.clouds[(q, t)]

    def align(self, q, key, t, guess):
        c = self.case
        fn = self.ctx.multi_align if c["rig"] else self.ctx.align
        return bytes(fn(self.cloud(q, key), self.cloud(q, t), c["camera"], c["ap"], self.offset, self.offset, guess))

    def close(self):
        for cl in self.clouds.values():
            cl.close()
        self.ctx.close()


def check_sequence(results, q, case, chain):
    """results of one sequence (case sequence q, frames 0, 1, ... in order, no reset) against the chain and the model"""
    model = SeqModel()
    key = None
    for t, r in enumerate(results):
        odo = case["odometry"][q][t] if case["odometry"][q] is not None else None
        T = capi.from_colmajor(r["record"]["T"], 4)
        aligned, g, kf = model.frame(odo, T, int(r["record"]["inliers"]), case["pixels"], FRACTION)
        assert (r["aligned"], r["keyframe"], r["num_keyframes"], r["frame"]) == (aligned, kf, model.nkey, t), (q, t)
        assert np.array_equal(r["guess"].view(np.uint32), cm(g)), (q, t)
        assert np.array_equal(r["global_T"].view(np.uint32), cm(model.G)), (q, t)
        if aligned:
            want = np.frombuffer(chain.align(q, key, t, capi.from_colmajor(r["guess"], 4)), capi.RESULT_DTYPE)[0]
            got = r["record"]
            differ = [f for f in capi.RESULT_DTYPE.names if got[f].tobytes() != want[f].tobytes()]
            allowed = ZERO_INLIER_FIELDS if int(got["inliers"]) == 0 else ()
            assert set(differ) <= set(allowed), (q, t, {f: (got[f], want[f]) for f in differ})
            assert np.array_equal(r["relative_T"].view(np.uint32), r["record"]["T"].view(np.uint32)), (q, t)
            assert r["record"]["status"] == 0
        else:
            assert not r["record"].tobytes().strip(b"\0") and np.array_equal(r["relative_T"], capi.colmajor(np.eye(4)))
        if kf:
            key = t
    return model.nkey


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_track_result_layout():
    """nicp_track_result: 464 bytes, the record at byte 208"""
    T = capi.TrackResult
    assert C.sizeof(T) == 464
    offsets = dict(global_T=0, relative_T=64, guess=128, frame=192, aligned=196, keyframe=200, num_keyframes=204, record=208)
    for name, off in offsets.items():
        assert getattr(T, name).offset == off, name
        assert capi.TRACK_DTYPE.fields[name][1] == off, name
    assert C.sizeof(capi.AlignResult) == 256


@pytest.mark.parametrize("v", [False, True])
def test_null_handles_are_rejected(v):
    """no pool, tracker, projector or parameters: status 1 (size -1, destroy a no-op) before any device is touched"""
    L = capi.load(v)
    L.nicp_tracker_destroy.restype = None
    N, f = None, C.c_float
    h = C.c_void_p(1)
    assert L.nicp_tracker_create(N, 2, 480, 640, f(0.001), 1, f(0.01), N, N, N, N, f(50), f(0.4), C.byref(h)) == 1
    assert not h
    assert L.nicp_tracker_create(N, 2, 480, 640, f(0.001), 1, f(0.01), N, N, N, N, f(50), f(0.4), N) == 1
    h = C.c_void_p(1)
    assert L.nicp_multi_tracker_create(N, 2, N, N, f(0.001), 1, f(0.01), N, N, N, N, f(50), f(0.4), C.byref(h)) == 1
    assert not h
    assert L.nicp_multi_tracker_create(N, 2, N, N, f(0.001), 1, f(0.01), N, N, N, N, f(50), f(0.4), N) == 1
    assert L.nicp_tracker_size(N) == -1
    assert L.nicp_tracker_step(N, 1, N, N, N, N) == 1
    assert L.nicp_tracker_step(N, 0, N, N, N, N) == 1
    assert L.nicp_tracker_reset(N, 1, N) == 1
    assert L.nicp_tracker_reset(N, 0, N) == 1
    L.nicp_tracker_destroy(N)


def test_model_reorthogonalises_like_the_class():
    """the restatement's re-orthogonalisation R - 0.5 R (R^T R - I) pulls a drifted rotation back towards SO(3)"""
    R = synth.make_pose((0, 0, 0), (0.3, 1.0, 0.2), 20.0)[:3, :3].astype(f32) * f32(1.001)
    E = mat3_mul(R.T.copy(), R) - np.eye(3, dtype=f32)
    R2 = R - mat3_mul(R, E) * f32(0.5)
    assert np.abs(R2.T @ R2 - np.eye(3)).max() < 0.1 * np.abs(R.T @ R - np.eye(3)).max()


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("step", [4, 1])
def test_tracker_matches_single_calls_and_the_model(verify, step):
    """five sequences (one with odometry) on one tracker and two of them again on a tracker with a sensor offset, sharing
    pools of one, two and three workers: records equal the single-call chain, poses the float32 restatement, and nothing
    depends on the worker count; a second identical run gives identical bytes"""
    case = pinhole_case(step)
    steps = schedule(case)
    off_map = {0: 1, 1: 4}
    off_steps = [[(s, t) for s, q in off_map.items() if t < len(case["frames"][q])] for t in range(len(steps))]
    runs = []
    for devs in POOLS + ([0],):
        pool = capi.ShardPool(devs, verify=verify)
        tr = make_tracker(pool, case, 5)
        tro = make_tracker(pool, case, 2, SENSOR_OFFSET)
        assert (tr.size(), tro.size()) == (5, 2)
        res, reso = {}, {}
        for st, sto in zip(steps, off_steps):  # the two trackers interleaved on one pool
            for s, r in run_steps(tr, case, [st]).items():
                res.setdefault(s, []).extend(r)
            for s, r in run_steps(tro, case, [sto], off_map).items():
                reso.setdefault(s, []).extend(r)
        tr.close()
        tro.close()
        pool.close()
        runs.append((b"".join(np.array(res[s]).tobytes() for s in range(5)),
                     b"".join(np.array(reso[s]).tobytes() for s in range(2))))
    assert all(r == runs[0] for r in runs[1:])  # workers 1, 2, 3 and a repeated run: the same bytes

    chain = Chain(case, verify)
    keyframes = [check_sequence(res[q], q, case, chain) for q in range(5)]
    chain.close()
    chain = Chain(case, verify, SENSOR_OFFSET)
    for s, q in off_map.items():
        check_sequence(reso[s], q, case, chain)
    chain.close()
    assert sum(keyframes) > 5, keyframes  # keyframe switches happened


@pytest.mark.gpu
def test_rejecting_every_correspondence_takes_the_guess(verify):
    """inlier_distance_threshold 0 rejects every correspondence: globalT = globalT * guess and a keyframe on every frame, as
    SequentialTracker does (the C++ comparison is in test_batch_tracker_class_matches_sequential_trackers)"""
    case = pinhole_case(4, lengths=(6, 8), odometry_seq=1, distance=0.0)
    pool = capi.ShardPool([0, 0], verify=verify)
    tr = make_tracker(pool, case, 2)
    res = run_steps(tr, case, schedule(case))
    tr.close()
    pool.close()
    chain = Chain(case, verify)
    for q in range(2):
        assert (np.array([r["record"]["inliers"] for r in res[q]]) == 0).all()
        assert check_sequence(res[q], q, case, chain) == len(case["frames"][q])
        assert all(r["keyframe"] for r in res[q])
    chain.close()


@pytest.mark.gpu
def test_subsets_orders_and_resets(verify):
    """steps list different subsets in different orders and sequence 2 is reset mid-run: every sequence's results equal those
    of a tracker that only ever saw that sequence (reset at the same point)"""
    case = pinhole_case(4, lengths=(9, 9, 9, 9), odometry_seq=0)
    rng = np.random.default_rng(3)
    nxt = [0, 0, 0, 0]
    steps, reset_at = [], None
    while any(n < 9 for n in nxt):
        pick = [s for s in rng.permutation(4) if nxt[s] < 9 and rng.random() < 0.7]
        if not pick:
            continue
        steps.append([(int(s), nxt[s]) for s in pick])
        for s in pick:
            nxt[s] += 1
        if reset_at is None and nxt[2] >= 4:
            reset_at = len(steps)
    alone = {}
    pool = capi.ShardPool([0, 0], verify=verify)
    for s in range(4):
        tr = make_tracker(pool, case, 1)
        mine = [[(0, t) for q, t in st if q == s] for st in steps]
        out = []
        for k, st in enumerate(mine):
            if k == reset_at and s == 2:
                tr.reset([0])
            if st:
                out += run_steps(tr, case, [st], {0: s})[0]
        alone[s] = np.array(out).tobytes()
        tr.close()
    tr = make_tracker(pool, case, 4)
    got = {s: [] for s in range(4)}
    for k, st in enumerate(steps):
        if k == reset_at:
            tr.reset([2])
        for s, r in run_steps(tr, case, [st]).items():
            got[s] += r
    tr.close()
    pool.close()
    for s in range(4):
        assert np.array(got[s]).tobytes() == alone[s], s
    frames2 = [int(r["frame"]) for r in got[2]]
    assert frames2.count(0) == 2 and sum(int(r["aligned"]) == 0 for r in got[2]) == 2  # restarted once


def rig_case(kind, step, n_seq=3, n_frames=5):
    cams = make_cams(kind)
    mp = capi.make_multi_projector(cams)
    rows, cols = capi.multi_image_size(mp)
    frames = []
    for i in range(n_seq):
        base = synth.make_pose((0.1, -0.05, 0.2), (0, 1, 0), 10.0 + 3 * i)
        poses = [base @ synth.make_pose((0.01 * k, 0.005 * k, 0), (0.2, 1, 0), 1.0 * k) for k in range(n_frames)]
        frames.append([render_raw_frame(p, cams, step, 90 + 13 * i + k) for k, p in enumerate(poses)])
    ap = capi.make_align_params(0.5, 0.95, 0.02, 1.3, 9e3, True, 10, 1)
    return dict(rig=True, camera=mp, sp=capi.make_stats_params(*RIG_SP), ap=ap, step=step,
                raw_shape=[im.shape for im in frames[0][0]], frames=frames, odometry=[None] * n_seq, pixels=rows * cols)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["4cam", "ragged"])
@pytest.mark.parametrize("step", [1, 2])
def test_rig_tracker_matches_single_calls_and_the_model(verify, kind, step):
    """both test rigs: records equal nicp_multi_raw_depth_to_cloud_batch + nicp_multi_align, poses the restatement (the
    keyframe fraction over composite pixels), on pools of one and two workers"""
    case = rig_case(kind, step)
    runs = []
    for devs in POOLS[:2]:
        pool = capi.ShardPool(devs, verify=verify)
        tr = make_tracker(pool, case, 3)
        runs.append(run_steps(tr, case, schedule(case)))
        tr.close()
        pool.close()
    res = runs[0]
    assert all(np.array(runs[1][s]).tobytes() == np.array(res[s]).tobytes() for s in range(3))
    chain = Chain(case, verify)
    for q in range(3):
        check_sequence(res[q], q, case, chain)
        assert (np.array([r["record"]["inliers"] for r in res[q][1:]]) > 0).all()
    chain.close()


@pytest.mark.gpu
def test_bad_input_is_rejected_and_changes_nothing(verify, monkeypatch):
    case = pinhole_case(4, lengths=(6, 6, 6), odometry_seq=None)
    steps = schedule(case)
    pool = capi.ShardPool([0, 0], verify=verify)
    clean = make_tracker(pool, case, 3)
    expect = [run_steps(clean, case, [st]) for st in steps]
    clean.close()
    tr = make_tracker(pool, case, 3)
    L = tr.L
    frame = case["frames"][0][0]
    bad = [
        lambda: tr.step([0, 3], [frame, frame]),
        lambda: tr.step([1, 1], [frame, frame]),
        lambda: tr.step([-1], [frame]),
        lambda: tr.reset([0, 0]),
        lambda: tr.reset([3]),
    ]
    match = ["sequence 3 outside", "sequence 1 is listed twice", "sequence -1 outside", "sequence 0 is listed twice",
             "sequence 3 outside"]
    for k, st in enumerate(steps):
        if k < len(bad):
            with pytest.raises(capi.NicpError, match=match[k]):
                bad[k]()
        if k == 1:
            with pytest.raises(ValueError, match=r"frame 1, camera 0: raw image of shape \(240, 320\)"):
                tr.step([0, 1], [frame, np.ascontiguousarray(frame[::2, ::2])])
            seqs = np.array([0, 2], np.int32)
            RA = (C.c_void_p * 2)(frame.ctypes.data, None)
            res = np.zeros(2, capi.TRACK_DTYPE)
            assert L.nicp_tracker_step(tr.handle, 2, capi._iptr(seqs), RA, None,
                                       res.ctypes.data_as(C.POINTER(capi.TrackResult))) == 1
            assert L.nicp_last_error().decode() == "null raw image of camera 0 in entry 1 (sequence 2)"
            assert L.nicp_tracker_step(tr.handle, 2, None, RA, None, res.ctypes.data_as(C.POINTER(capi.TrackResult))) == 1
        got = run_steps(tr, case, [st])
        assert all(np.array(got[s]).tobytes() == np.array(expect[k][s]).tobytes() for s in got), k
    assert len(tr.step([], [])) == 0
    tr.reset([])
    # a destroyed pool: every call but destroy returns NICP_ERR_INVALID
    pool.close()
    gone = "the tracker's shard pool has been destroyed"
    with pytest.raises(capi.NicpError, match=gone):
        tr.step([0], [frame])
    with pytest.raises(capi.NicpError, match=gone):
        tr.reset([0])
    assert tr.size() == -1
    tr.close()
    assert not tr.handle

    # more sequences than a worker's frame cap holds at two clouds each
    monkeypatch.setenv("NICP_SHARD_FRAMES", "4")
    pool = capi.ShardPool([0], verify=verify)
    with pytest.raises(capi.NicpError, match="3 sequences at two clouds each, more than its frame cap of 4"):
        make_tracker(pool, case, 3)
    make_tracker(pool, case, 2).close()
    pool.close()
    pool = capi.ShardPool([0, 0], verify=verify)  # 1 + 2 sequences
    tr = make_tracker(pool, case, 3)
    assert tr.size() == 3
    with pytest.raises(capi.NicpError, match="does not match the scaled raw image"):
        capi.Tracker(pool, case["camera"], case["sp"], case["ap"], (480, 644), 2, step=2)
    tr.close()
    pool.close()


def _write_driver_input(path, case, n_seq, n_frames, step, distance):
    c = CONF_1_1 if step == 1 else CONF_1_4
    hdr = np.array([n_seq, n_frames, 480, 640, step, 1, c["minImageRadius"], c["maxImageRadius"], c["minPoints"]], np.int32)
    vals = np.concatenate([capi.colmajor(synth.K_KINECT), capi.colmajor(SENSOR_OFFSET),
                           np.array([FRACTION, distance, c["minD"], c["maxD"]], f32)]).astype(f32)
    raws = np.stack([np.stack([case["frames"][s][t] for s in range(n_seq)]) for t in range(n_frames)]).astype(np.uint16)
    odo = np.stack([np.stack([capi.colmajor(odometry_of(sequence(s, len(case["frames"][s]))[1], 50 + s)[t])
                              for s in range(n_seq)]) for t in range(n_frames)]).astype(f32)
    path.write_bytes(hdr.tobytes() + vals.tobytes() + raws.tobytes() + odo.tobytes())


@pytest.mark.gpu
@pytest.mark.parametrize("lib", ["nicp_b200", "nicp_b200_verify"])
@pytest.mark.parametrize("distance", [0.5, 0.0])
def test_batch_tracker_class_matches_sequential_trackers(tmp_path, lib, distance):
    """tests/cpp/batch_tracker.cpp: three sequences through pwn::BatchTracker on two workers and through three
    pwn::SequentialTrackers, with a sensor offset and odometry; globalT, lastRelative, lastInliers, numKeyframes and
    lastWasKeyframe bit-identical after every frame, also when every correspondence is rejected (distance 0)"""
    step, n_frames = 4, 14
    case = pinhole_case(step, lengths=(14, 18, 22))
    libdir = os.path.join(ROOT, "g2o_frontend_b200", "lib")
    exe = str(tmp_path / "batch_tracker")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([cxx, "-std=c++17", "-O1", "-ffp-contract=off", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           "-o", exe, os.path.join(ROOT, "tests", "cpp", "batch_tracker.cpp"), "-L", libdir, "-l" + lib,
                           "-Wl,-rpath," + libdir])
    _write_driver_input(tmp_path / "in.bin", case, 3, n_frames, step, distance)
    out = subprocess.run([exe, str(tmp_path / "in.bin"), "2"], capture_output=True, text=True)
    assert out.returncode == 0 and "batch_tracker ok" in out.stdout, out.stdout[-3000:] + out.stderr
    lines = [l.split() for l in out.stdout.splitlines() if l.startswith("frame ")]
    assert len(lines) == sum(1 for f in range(n_frames) for s in range(3) if (f + s) % 4 != 3)
    keyframes = {int(l[3]): int(l[7]) for l in lines}
    if distance > 0:
        assert sum(keyframes.values()) > 3, keyframes
        assert all(int(l[5]) > 0 for l in lines[3:])
    else:
        assert all(int(l[5]) == 0 for l in lines)

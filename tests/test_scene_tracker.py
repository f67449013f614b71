"""Batched scene-based odometry of independent depth sequences on a shard pool (nicp_scene_tracker_*, capi.SceneTracker).
Every sequence must do exactly what one iteration of the mapping loop of pwn_core/pwn_aligner.cpp does on its frame, as
the chain of single C-ABI calls below restates it:
  - the result (record bytes, both poses, added, map_points, new_map) and every downloaded map array equal the chain's
    after every step, byte for byte;
  - results do not depend on the worker count, on which other sequences a step lists or in which order, or on rejected
    calls made before it;
  - one sequence follows tests/test_reference_pwn_core.py::oracle_scene_odometry within the tolerances of
    tests/test_host_cpp.py::test_local_map_matches_oracle_loop."""
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import CONF_1_4, ROOT
from g2o_frontend_b200 import capi, synth
from test_tracker import iso_mul

f32 = np.float32
MAP_CAP = 1000000
BASELINE, ALPHA = 0.075, 0.1
SENSOR_OFFSET = synth.make_pose((0.05, -0.02, 0.1), (0.3, 1.0, 0.2), 4.0).astype(f32)
INITIAL_POSE = synth.make_pose((0.2, -0.1, 0.3), (0.1, 0.2, 1.0), 15.0).astype(f32)


@pytest.fixture(scope="module", params=["verify", "default"])
def verify(request):
    return request.param == "verify"


def params(step):
    c = CONF_1_4
    K = synth.scaled_K(synth.K_KINECT, f32(1.0) / f32(step))
    proj = capi.make_projector(K, 480 // step, 640 // step, c["minD"], c["maxD"])
    sp = capi.make_stats_params(c["worldRadius"], c["minImageRadius"], c["maxImageRadius"], c["minPoints"],
                                c["curvatureThreshold"], c["omegaCurvatureThreshold"])
    ap = capi.make_align_params(c["inlierDistanceThreshold"], c["inlierNormalAngularThreshold"],
                                c["flatCurvatureThreshold"], c["inlierCurvatureRatioThreshold"], c["inlierMaxChi2"], True,
                                10, 1)
    return K, proj, sp, ap, capi.make_merge_params()


_SEQS = {}


def sequences():
    """five synthetic 640x480 sequences: three trajectories, the map sequence of the reference driver test and one whose
    frames are all zero depth (empty map, empty render, no inliers)"""
    if not _SEQS:
        from test_reference_pwn_core import map_sequence
        for i, n in enumerate((7, 6, 5)):
            poses = synth.trajectory(n, seed=21 + i, step_t=0.02, step_deg=1.0)
            _SEQS[i] = [synth.render_depth_u16(p, seed=500 + 31 * i + k) for k, p in enumerate(poses)]
        _SEQS[3] = map_sequence(6)[1]
        _SEQS[4] = [np.zeros((480, 640), np.uint16) for _ in range(4)]
    return [_SEQS[i] for i in range(5)]


def initial_pose(s):
    """sequence 2 starts from a configured initial pose (the driver's initialT)"""
    return INITIAL_POSE if s == 2 else None


class Chain:
    """one sequence through the single C-ABI calls on a plain context (pwn_simple_aligner.cpp's localmap loop)"""

    def __init__(self, ctx, step, chunk_step, offset=None, initial=None):
        self.ctx, self.step, self.chunk = ctx, step, chunk_step
        self.K, self.proj, self.sp, self.ap, self.mp = params(step)
        self.so = np.eye(4, dtype=f32) if offset is None else offset
        self.G = np.eye(4, dtype=f32) if initial is None else initial.copy()
        self.S = self.G.copy()
        self.map = ctx.new_cloud(MAP_CAP)
        self.frames = self.counter = 0

    def frame(self, raw):
        ctx, proj = self.ctx, self.proj
        cloud = ctx.raw_depth_to_cloud(raw, proj, self.sp, step=self.step, sensor_offset=self.so)[0]
        cloud.compute_gaussians(ctx.depth_prepare(raw, step=self.step), proj, BASELINE, ALPHA, self.so)
        r = np.zeros(1, capi.SCENE_TRACK_DTYPE)[0]
        r["frame"] = self.frames
        if self.frames > 0:
            KRt = capi.update_matrices(self.K, iso_mul(self.S, self.so), ctx.verify)[0]
            depth = ctx.project(self.map, KRt, proj.rows, proj.cols, proj.min_distance, proj.max_distance)[1]
            sub = ctx.depth_to_cloud(depth, proj, self.sp, sensor_offset=self.so, want_index=False)[0]
            rec = ctx.align(sub, cloud, proj, self.ap, self.so, self.so)
            T = capi.result_T(rec)
            self.G, self.S = iso_mul(self.G, T), iso_mul(self.S, T)
            r["aligned"] = 1
            r["record"] = np.frombuffer(bytes(rec), capi.RESULT_DTYPE)[0]
            if self.chunk > 0:
                if self.counter % self.chunk == 0:
                    self.S = np.eye(4, dtype=f32)
                    self.map.upload(np.zeros((1, 4), f32)[:0])  # referenceScene.clear(): the map keeps its storage
                    r["new_map"] = 1
                self.counter += 1
        self.map.append(cloud, self.S)
        r["added"] = self.map.size()
        if r["added"]:
            self.map.merge(proj, iso_mul(self.S, self.so), self.mp)
        r["map_points"] = self.map.size()
        r["global_T"] = capi.colmajor(self.G)
        r["scene_T"] = capi.colmajor(self.S)
        self.frames += 1
        return r

    def map_arrays(self):
        if self.map.size() == 0:
            return None
        d = self.map.download()
        d["gauss"], d["gflags"] = self.map.download_gaussians()
        return d


def same_map(got, want):
    if want is None:
        assert len(got["points"]) == 0
        return
    for k in ("points", "normals", "curvature", "omega_p", "omega_n", "gauss", "gflags"):
        assert got[k].shape == want[k].shape, k
        assert got[k].tobytes() == want[k].tobytes(), k


def make_tracker(pool, step, chunk_step, n_sequences, offset=None, map_capacity=MAP_CAP):
    _, proj, sp, ap, mp = params(step)
    return capi.SceneTracker(pool, proj, sp, ap, (480, 640), n_sequences, map_capacity, mp=mp, step=step,
                             sensor_offset=offset, baseline=BASELINE, alpha=ALPHA, chunk_step=chunk_step)


def schedule(frames):
    """step t lists every sequence that still has a frame t (reversed on odd t)"""
    out = []
    for t in range(max(len(f) for f in frames)):
        seqs = [s for s in range(len(frames)) if t < len(frames[s])]
        out.append([(s, t) for s in (seqs[::-1] if t % 2 else seqs)])
    return out


_CHAINS = {}


def chain_results(verify, step, chunk_step, s, offset=None):
    """[(result, map arrays) after every frame] of the chain on sequence s, cached per configuration"""
    key = (verify, step, chunk_step, s, offset is not None)
    if key not in _CHAINS:
        ctx = capi.Context(0, verify=verify)
        ch = Chain(ctx, step, chunk_step, offset, initial_pose(s))
        _CHAINS[key] = [(ch.frame(raw), ch.map_arrays()) for raw in sequences()[s]]
        ctx.close()
    return _CHAINS[key]


def check_step(tr, results, want, seqs_frames):
    for (s, t), r in zip(seqs_frames, results):
        wr, wmap = want[s][t]
        assert r.tobytes() == wr.tobytes(), (s, t, r, wr)
        same_map(tr.download_map(s), wmap)


CASES = [(4, 0, [0]), (4, 2, [0, 0]), (4, 10, [0, 0, 0]), (2, 0, [0, 0, 0]), (2, 2, [0]), (2, 10, [0, 0])]


@pytest.mark.gpu
@pytest.mark.parametrize("step,chunk_step,devices", CASES)
def test_steps_equal_the_single_call_chain(verify, step, chunk_step, devices):
    """five sequences (one from a configured initial pose, one all zero depth) on pools of one to three workers: after
    every step each listed sequence's result and map equal the chain of single calls byte for byte"""
    frames = sequences()
    want = {s: chain_results(verify, step, chunk_step, s) for s in range(len(frames))}
    pool = capi.ShardPool(devices, verify=verify)
    tr = make_tracker(pool, step, chunk_step, len(frames))
    assert tr.size() == len(frames)
    tr.reset([2], [INITIAL_POSE])
    for st in schedule(frames):
        res = tr.step([s for s, _ in st], [frames[s][t] for s, t in st])
        check_step(tr, res, want, st)
    # the all-zero sequence: an empty map, aligned against an empty render with no inliers
    assert tr.download_map(4)["points"].shape == (0, 4)
    assert want[4][-1][0]["aligned"] == 1 and want[4][-1][0]["record"]["inliers"] == 0
    # the chunk decisions took place
    new_maps = sum(int(want[s][t][0]["new_map"]) for s in range(5) for t in range(len(frames[s])))
    assert (new_maps > 0) == (chunk_step > 0)
    tr.close()
    pool.close()


@pytest.mark.gpu
def test_sensor_offset_equals_the_chain(verify):
    """a tracker with a sensor offset: preparation, gaussians, render and merge views and both alignment sides use it"""
    frames = sequences()
    want = chain_results(verify, 4, 2, 0, SENSOR_OFFSET)
    pool = capi.ShardPool([0, 0], verify=verify)
    tr = make_tracker(pool, 4, 2, 2, offset=SENSOR_OFFSET)
    for t, raw in enumerate(frames[0]):
        res = tr.step([1], [raw])
        check_step(tr, res, {1: want}, [(1, t)])
    tr.close()
    pool.close()


@pytest.mark.gpu
def test_subsets_orders_and_resets(verify):
    """different subsets in different orders per step, a mid-run reset with and without an initial pose: each sequence
    gets exactly the results of a tracker that saw only it"""
    frames = sequences()
    step, chunk = 4, 2
    pool = capi.ShardPool([0, 0], verify=verify)
    tr = make_tracker(pool, step, chunk, 4)
    # tracker sequence -> case sequence; sequences 0 and 1 are reset after frame 2 (1 with the initial pose) and replay
    src = {0: 0, 1: 1, 2: 3, 3: 2}
    nxt = {s: 0 for s in src}
    plan = [[0, 1, 2, 3], [3, 0], [1, 2], [2, 0, 3, 1], "reset", [1, 0], [0, 3, 2, 1], [2, 1, 0], [0, 1], [1, 0], [0, 1]]
    got = {s: [] for s in src}
    for entry in plan:
        if entry == "reset":
            tr.reset([0])
            tr.reset([1], [INITIAL_POSE])
            for s in (0, 1):
                got[s].append("reset")
                nxt[s] = 0
            continue
        entry = [s for s in entry if nxt[s] < len(frames[src[s]])]
        res = tr.step(entry, [frames[src[s]][nxt[s]] for s in entry])
        for s, r in zip(entry, res):
            got[s].append((r.copy(), tr.download_map(s)))
            nxt[s] += 1
    ctx = capi.Context(0, verify=verify)
    for s, q in src.items():
        ch = Chain(ctx, step, chunk)
        for g in got[s]:
            if g == "reset":
                ch = Chain(ctx, step, chunk, None, INITIAL_POSE if s == 1 else None)
                continue
            want = ch.frame(frames[q][ch.frames])
            assert g[0].tobytes() == want.tobytes(), (s, g[0], want)
            same_map(g[1], ch.map_arrays())
    ctx.close()
    tr.close()
    pool.close()


def state_of(tr, n):
    return [tr.download_map(s) for s in range(n)]


@pytest.mark.gpu
def test_rejected_calls_change_nothing(verify):
    """null handles or arrays, a sequence out of range or listed twice, a map too small for the frame, create over the
    frame cap and a destroyed pool are rejected, and the poses, counters and maps stay as they were"""
    import ctypes as C
    frames = sequences()
    step = 4
    pool = capi.ShardPool([0], verify=verify)
    L = pool.L
    # a map that holds one frame but not two: the second step is rejected before any map is touched
    tr = make_tracker(pool, step, 0, 2)
    small = make_tracker(pool, step, 0, 1, map_capacity=(480 // step) * (640 // step))
    tr.step([0, 1], [frames[0][0], frames[1][0]])
    before = state_of(tr, 2)
    assert small.step([0], [frames[0][0]])["map_points"][0] > 0
    small_map = small.download_map(0)
    with pytest.raises(capi.NicpError, match="exceed the map capacity"):
        small.step([0], [frames[0][1]])
    same_map(small.download_map(0), small_map)
    raw = np.ascontiguousarray(frames[0][1])
    RA = (C.c_void_p * 1)(raw.ctypes.data)
    seq = np.array([0], np.int32)
    out = np.zeros(2, capi.SCENE_TRACK_DTYPE)
    optr = out.ctypes.data_as(C.POINTER(capi.SceneTrackResult))
    assert L.nicp_scene_tracker_step(None, 1, capi._iptr(seq), RA, optr) != 0
    assert L.nicp_scene_tracker_step(tr.handle, 1, None, RA, optr) != 0
    assert L.nicp_scene_tracker_step(tr.handle, 1, capi._iptr(seq), None, optr) != 0
    assert L.nicp_scene_tracker_step(tr.handle, 1, capi._iptr(seq), RA, None) != 0
    assert L.nicp_scene_tracker_step(tr.handle, 1, capi._iptr(seq), (C.c_void_p * 1)(None), optr) != 0
    assert L.nicp_scene_tracker_step(tr.handle, -1, capi._iptr(seq), RA, optr) != 0
    with pytest.raises(capi.NicpError, match="outside"):
        tr.step([2], [frames[0][1]])
    with pytest.raises(capi.NicpError, match="listed twice"):
        tr.step([1, 1], [frames[1][1], frames[1][1]])
    with pytest.raises(capi.NicpError, match="outside"):
        tr.reset([-1])
    with pytest.raises(ValueError, match="raw image of shape"):
        tr.step([0], [frames[0][1][:240]])
    assert L.nicp_scene_tracker_download_map(tr.handle, 5, MAP_CAP, None, None, None, None, None, None, None, None) != 0
    n = C.c_int(0)
    assert L.nicp_scene_tracker_download_map(tr.handle, 0, 1, None, None, None, None, None, None, None, C.byref(n)) != 0
    assert n.value == len(before[0]["points"])
    for a, b in zip(state_of(tr, 2), before):
        same_map(a, b)
    # the next step continues exactly where the chain is after one frame
    want = [chain_results(verify, step, 0, s) for s in (0, 1)]
    res = tr.step([1, 0], [frames[1][1], frames[0][1]])
    check_step(tr, res, {0: want[0], 1: want[1]}, [(1, 1), (0, 1)])
    # create over the frame cap (NICP_SHARD_FRAMES is read when a pool is created)
    with pytest.raises(capi.NicpError, match="more than its frame cap"):
        make_tracker(pool, step, 0, 100000, map_capacity=10 ** 7)
    h = C.c_void_p()
    _, proj, sp, ap, mp = params(step)
    assert L.nicp_scene_tracker_create(pool.handle, 1, 480, 640, C.c_float(0.001), step, C.c_float(0.01), C.byref(proj),
                                       C.byref(sp), None, C.c_float(BASELINE), C.c_float(ALPHA), C.byref(ap),
                                       C.c_float(50.0), None, 0, MAP_CAP, C.byref(h)) != 0
    assert L.nicp_scene_tracker_create(pool.handle, 1, 480, 640, C.c_float(0.001), step, C.c_float(0.01), C.byref(proj),
                                       C.byref(sp), None, C.c_float(BASELINE), C.c_float(ALPHA), C.byref(ap),
                                       C.c_float(50.0), C.byref(mp), -1, MAP_CAP, C.byref(h)) != 0
    assert not h
    # a destroyed pool: every call except destroy fails
    pool.close()
    gone = "shard pool has been destroyed"
    assert tr.size() == -1
    with pytest.raises(capi.NicpError, match=gone):
        tr.step([0], [frames[0][2]])
    with pytest.raises(capi.NicpError, match=gone):
        tr.reset([0])
    with pytest.raises(capi.NicpError, match=gone):
        tr.download_map(0)
    with pytest.raises(capi.NicpError, match=gone):
        tr.phase_ms()
    tr.close()
    small.close()


@pytest.mark.gpu
def test_two_runs_are_byte_identical(verify):
    frames = sequences()
    outs = []
    for _ in range(2):
        pool = capi.ShardPool([0, 0], verify=verify)
        tr = make_tracker(pool, 2, 2, 5)
        run = []
        for st in schedule(frames):
            run.append(tr.step([s for s, _ in st], [frames[s][t] for s, t in st]).tobytes())
        run += [b"".join(v.tobytes() for v in tr.download_map(s).values()) for s in range(5)]
        p1, p2 = tr.phase_ms()
        assert p1 > 0 and p2 > 0
        outs.append(run)
        tr.close()
        pool.close()
    assert outs[0] == outs[1]


@pytest.mark.gpu
def test_one_sequence_follows_the_oracle(verify):
    """the map sequence against oracle_scene_odometry (the restatement checked against the reference's own pwn_aligner),
    within the tolerances of test_local_map_matches_oracle_loop"""
    from test_reference_pwn_core import map_sequence, oracle_scene_odometry
    raws = map_sequence(6)[1]
    scale = 4
    conf = CONF_1_4
    pool = capi.ShardPool([0], verify=verify)
    tr = make_tracker(pool, scale, 2, 1)
    got = [tr.step([0], [r])[0] for r in raws]
    poses, sizes = oracle_scene_odometry(raws, conf, scale, chunk_step=2)
    for r, P, n in zip(got, poses, sizes):
        G = capi.from_colmajor(r["global_T"], 4)
        assert np.abs(G - P).max() < 1e-3, (G, P)
        assert abs(int(r["map_points"]) - n) <= 5e-3 * n + 8, (r["map_points"], n)
    tr.close()
    pool.close()


@pytest.mark.gpu
def test_many_launch_sets_and_append_launches(verify, monkeypatch):
    """70 sequences on one worker with NICP_PREP_BATCH = 3 (read on every call): a step walks 24 prep launch sets that
    reuse the same depth and integral scratch slots for frames, renders and subscenes, and two append launches (64 frames
    per launch); every sequence still equals the chain"""
    monkeypatch.setenv("NICP_PREP_BATCH", "3")
    frames = sequences()
    cases = (0, 1, 3, 4)  # no initial pose
    step, chunk, S, F = 4, 2, 70, 4
    want = {c: chain_results(verify, step, chunk, c) for c in cases}
    pool = capi.ShardPool([0], verify=verify)
    tr = make_tracker(pool, step, chunk, S, map_capacity=(F + 1) * (480 // step) * (640 // step))
    for t in range(F):
        seqs = list(range(S))[::-1] if t % 2 else list(range(S))
        res = tr.step(seqs, [frames[cases[s % 4]][t] for s in seqs])
        for s, r in zip(seqs, res):
            wr, wmap = want[cases[s % 4]][t]
            assert r.tobytes() == wr.tobytes(), (s, t)
            if s % 7 == 0 or t == F - 1:
                same_map(tr.download_map(s), wmap)
    tr.close()
    pool.close()


def _cxx():
    return "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"


@pytest.mark.gpu
@pytest.mark.parametrize("lib", ["nicp_b200", "nicp_b200_verify"])
@pytest.mark.parametrize("chunk_step", [0, 2])
def test_batch_scene_tracker_class_matches_the_cli_driver(tmp_path, lib, chunk_step):
    """tests/cpp/scene_tracker.cpp: three sequences through pwn::BatchSceneTracker on two workers, and each through
    host/pwn_simple_aligner.cpp in localmap mode built against the same library: globalT through %.9g, inliers, added,
    map_points and new_map equal after every frame, and the voxel count of each final map equal"""
    from test_host_cpp import write_conf, write_pgm16
    libdir = os.path.join(ROOT, "g2o_frontend_b200", "lib")
    link = ["-I", os.path.join(ROOT, "include"), "-L", libdir, "-l" + lib, "-Wl,-rpath," + libdir]
    exe, drv = str(tmp_path / "scene_tracker"), str(tmp_path / "pwn_simple_aligner")
    subprocess.check_call([_cxx(), "-std=c++17", "-O1", "-ffp-contract=off", "-Wall", "-Werror", "-o", exe,
                           os.path.join(ROOT, "tests", "cpp", "scene_tracker.cpp")] + link)
    subprocess.check_call([_cxx(), "-std=c++17", "-O2", "-ffp-contract=off", "-Wall", "-o", drv,
                           os.path.join(ROOT, "g2o_frontend_b200", "host", "pwn_simple_aligner.cpp")] + link +
                          ["-Wl,-z,lazy"])
    F = 5
    seqs = [sequences()[i][:F] for i in (0, 1, 3)]
    files = []
    for s, fr in enumerate(seqs):
        files.append([])
        for f, raw in enumerate(fr):
            files[s].append(str(tmp_path / ("s%d_f%02d.pgm" % (s, f))))
            write_pgm16(files[s][-1], raw)
    cfg = str(tmp_path / "map.conf")
    off_v = [0.05, -0.02, 0.1, 0.02, 0.05, -0.01]
    write_conf(cfg, CONF_1_4, 4, off_v, extra={"localmap": 1, "voxelResolution": 0.02, "chunkStep": chunk_step})
    out = str(tmp_path / "batch.jsonl")
    run = subprocess.run([exe, cfg, out, "2", str(len(seqs)), str(F)] + [p for fs in files for p in fs],
                         capture_output=True, text=True)
    assert run.returncode == 0, run.stdout[-2000:] + run.stderr
    got = [json.loads(l) for l in open(out)]
    new_maps = 0
    for s in range(len(seqs)):
        ref = str(tmp_path / ("driver%d.jsonl" % s))
        subprocess.check_call([drv, cfg, ref] + files[s])
        want = [json.loads(l) for l in open(ref)]
        mine = [g for g in got if g["seq"] == s]
        assert len(mine) == F + 1 and len(want) == F + 1
        for f in range(F):
            g, w = mine[f], want[f]
            assert g["frame"] == w["frame"] == f
            for k in ("inliers", "added", "map_points", "new_map", "globalT"):
                assert g[k] == w[k], (s, f, k, g[k], w[k])
            new_maps += g["new_map"]
        assert mine[F]["map_points"] == want[F]["map_points"] and mine[F]["voxel_points"] == want[F]["voxel_points"], \
            (s, mine[F], want[F])
        assert want[F]["voxel_points"] > 0
    assert (new_maps > 0) == (chunk_step > 0)

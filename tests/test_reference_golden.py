"""The comparisons of tests/test_reference_pwn_core.py without the reference's library: the oracle against the outputs
stored in tests/golden/reference_cases.npz (tests/reference_cases.py names the cases; make_reference_golden.py writes
the file). Every array is pinned bit for bit by its SHA-256 and shape. A fixed sample of its elements is stored too, so a
failure shows values. CPU only."""
import hashlib
import os

import numpy as np
import pytest

from conftest import ROOT
import reference_cases as RC

GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_cases.npz")
SAMPLE = 64


def digest(a):
    a = np.ascontiguousarray(a)
    return hashlib.sha256(a.dtype.str.encode() + str(a.shape).encode() + a.tobytes()).hexdigest()


def sample_index(a):
    n = np.asarray(a).size
    return np.arange(n) if n <= SAMPLE else np.sort(np.random.default_rng(0).choice(n, SAMPLE, replace=False))


def record(case, outputs):
    """the stored form of one case: digest, shape and element sample of every output (whole values where tolerant)"""
    rec = {}
    for name, a in outputs.items():
        a = np.asarray(a)
        key = case + "|" + name
        rec[key + "|sha256"] = np.array(digest(a))
        rec[key + "|shape"] = np.array(a.shape, np.int64)
        rec[key + "|sample"] = a.reshape(-1)[sample_index(a)]
    return rec


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


@pytest.mark.parametrize("case", sorted(RC.all_cases()))
def test_oracle_reproduces_the_reference_outputs(golden, case):
    outputs = RC.all_cases()[case]()
    stored = sorted(k.split("|")[1] for k in golden.files if k.startswith(case + "|") and k.endswith("|sha256"))
    assert stored == sorted(outputs), (stored, sorted(outputs))
    for name, a in outputs.items():
        a = np.asarray(a)
        key = case + "|" + name
        assert tuple(golden[key + "|shape"]) == a.shape, name
        want = golden[key + "|sample"]
        got = a.reshape(-1)[sample_index(a)]
        if name in RC.TOLERANT:
            assert np.abs(got - want).max() <= RC.TOLERANT[name] * np.abs(want).max(), name
            continue
        assert np.array_equal(got, want, equal_nan=True), (name, got[got != want][:8], want[got != want][:8])
        assert digest(a) == str(golden[key + "|sha256"]), name
    if case.startswith("align-") and case not in ("align-sensor_offset", "align-one_iteration", "align-inner_iterations"):
        from g2o_frontend_b200 import synth
        assert np.abs(outputs["T"] - synth.POSE_B).max() < 5e-3  # a real alignment: the ground-truth motion is recovered
    if case.startswith("depth_to_cloud-"):
        assert (np.abs(outputs["cloud_normals"][:, :3]).sum(1) > 0).mean() > 0.5  # not vacuous: most points have a normal
    if case.startswith("finder_linearizer-"):
        assert len(outputs["corr"]) > 5000


def golden_equal(golden, key, a):
    """a (cast to the stored outputs' layout) is bit-identical to the stored output `key`"""
    a = np.ascontiguousarray(a).reshape(tuple(golden[key + "|shape"]))
    return digest(a) == str(golden[key + "|sha256"])


@pytest.fixture(scope="module", params=["verify", "default"])
def ctx(request):
    from g2o_frontend_b200 import capi
    c = capi.Context(0, verify=(request.param == "verify"))
    yield c
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["clean", "noise_dropout", "sensor_offset", "full_resolution"])
def test_frame_prep_reproduces_the_reference_outputs(golden, ctx, case):
    """the GPU frame prep against the stored outputs: index, interval and integral images, points and Stats::n bit-exact
    (the bar of test_vs_reference_gpu.py::test_frame_prep_against_the_reference_sources)"""
    from conftest import get_scene
    s = {"clean": lambda: get_scene(4), "noise_dropout": lambda: get_scene(4, seed=1, dropout=0.05),
         "sensor_offset": lambda: get_scene(4, offset=True), "full_resolution": lambda: get_scene(1)}[case]()
    key = "depth_to_cloud-" + case + "|"
    cl, idx = ctx.depth_to_cloud(s.depthA, s.projector(), s.stats_params(), s.sensor_offset, keep_stats=True)
    assert golden_equal(golden, key + "index", np.asarray(idx, np.int32))
    assert golden_equal(golden, key + "interval", np.asarray(ctx.last_interval_image(s.rows, s.cols), np.int32))
    assert golden_equal(golden, key + "integral", np.asarray(ctx.last_integral_image(s.rows, s.cols), np.float32))
    assert golden_equal(golden, key + "cloud_points", np.asarray(cl.download()["points"], np.float32))
    assert golden_equal(golden, key + "cloud_statsN", np.asarray(cl.download_stats()[2], np.int32))


@pytest.mark.gpu
def test_projection_reproduces_the_reference_outputs(golden, ctx):
    """the GPU z-buffer projection against the stored index and depth images, bit-exact"""
    from conftest import get_scene
    from oracle import pwn_oracle as O
    from test_vs_reference_gpu import upload
    s = get_scene(4)
    c = s.conf
    cl = upload(ctx, s.cloudA)
    for j, v in enumerate(RC.PROJECTION_POSES[:3]):  # the poses test_vs_reference_gpu.py checks the GPU at
        KRt, _ = O.update_matrices(s.K, O.v2t(np.array(v, np.float32)))
        gi, gd = ctx.project(cl, KRt, s.rows, s.cols, c["minD"], c["maxD"])
        assert golden_equal(golden, "projection|index_%d" % j, np.asarray(gi, np.int32)), v
        assert golden_equal(golden, "projection|depth_%d" % j, np.asarray(gd, np.float32)), v

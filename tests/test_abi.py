"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol that
include/nicp_b200.h declares, struct layouts match, and -- with no GPU -- it fails loudly instead of
falling back to a CPU path.  No compute calls are made here."""
import ctypes as C
import os
import re

import pytest

from conftest import ROOT
from g2o_frontend_b200 import capi


def header_symbols():
    text = open(os.path.join(ROOT, "include", "nicp_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(nicp_[a-z0-9_]+)\s*\(", text)))


@pytest.mark.parametrize("verify", [False, True])
def test_library_exports_every_declared_symbol(verify):
    L = capi.load(verify)
    names = header_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(L, n), n
    assert sorted(capi.SYMBOLS) == names
    assert bool(L.nicp_is_verification_build()) == verify


def test_struct_layouts():
    assert C.sizeof(capi.AlignResult) == 256
    assert C.sizeof(capi.Projector) == 9 * 4 + 4 * 4
    assert C.sizeof(capi.StatsParams) == 6 * 4 + 9 * 4
    assert C.sizeof(capi.AlignParams) == 8 * 4
    assert C.sizeof(capi.Prior) == 4 + (16 + 16 + 36) * 4


def test_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    L = capi.load()
    h = C.c_void_p()
    rc = L.nicp_create(0, C.byref(h))
    assert rc != 0 and not h
    assert b"no CPU fallback" in L.nicp_last_error()
    with pytest.raises(capi.NicpError):
        capi.Context(0)


def test_missing_library_raises(monkeypatch, tmp_path):
    monkeypatch.setattr(capi, "LIB_DIR", str(tmp_path))
    monkeypatch.setattr(capi, "_LIBS", {})
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        capi.load()


def test_product_does_not_import_oracle():
    """only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline legs may touch oracle/"""
    pkg = os.path.join(ROOT, "g2o_frontend_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                text = open(os.path.join(dirpath, f)).read()
                assert "pwn_oracle" not in text and "liboracle" not in text, os.path.join(dirpath, f)
    for sub in ("include", "tools", "integration"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, sub)):
            for f in files:
                text = open(os.path.join(dirpath, f), errors="ignore").read()  # built tools (binaries) are scanned as bytes-ish text
                assert "pwn_oracle" not in text and "liboracle" not in text and "voxel_oracle" not in text, os.path.join(dirpath, f)


@pytest.mark.parametrize("verify", [False, True])
def test_null_handles_are_rejected_not_dereferenced(verify):
    """the reference only asserts on misuse (undefined behaviour in release builds); the C-ABI answers with a status code.
    Every entry point is called with null handles -- no GPU needed, nothing may crash."""
    import ctypes as C
    L = capi.load(verify)
    N = None
    f0 = C.c_float(0)
    L.nicp_cloud_size.restype = C.c_int
    L.nicp_launch_count.restype = C.c_longlong
    L.nicp_stream.restype = C.c_void_p
    assert L.nicp_synchronize(N) == 1                      # NICP_ERR_INVALID
    assert L.nicp_cloud_create(N, 10, N) == 1
    assert L.nicp_cloud_size(N) == -1
    assert L.nicp_launch_count(N) == 0
    assert L.nicp_stream(N) is None
    assert L.nicp_set_kernel_timing(N, 1) == 1
    assert L.nicp_get_kernel_timing(N, N, N, N, N) == 1
    assert L.nicp_cloud_upload(N, N, 0, N, N, N, N, N) == 1
    assert L.nicp_cloud_download(N, N, N, N, N, N, N) == 1
    assert L.nicp_cloud_download_stats(N, N, N, N, N) == 1
    assert L.nicp_cloud_transform(N, N, N) == 1
    assert L.nicp_cloud_append(N, N, N, N) == 1
    assert L.nicp_cloud_compute_gaussians(N, N, N, N, f0, f0, N) == 1
    assert L.nicp_cloud_has_gaussians(N) == 0
    assert L.nicp_cloud_download_gaussians(N, N, N, N) == 1
    assert L.nicp_cloud_upload_gaussians(N, N, N, N) == 1
    assert L.nicp_merge(N, N, N, N, N, N, N) == 1
    assert L.nicp_voxelize(N, N, C.c_float(0.01), N, N) == 1
    assert L.nicp_depth_prepare(N, N, 4, 4, C.c_float(0.001), 1, C.c_float(0.01), N) == 1
    assert L.nicp_unproject(N, N, 4, 4, N, f0, f0, N, N) == 1
    assert L.nicp_project_intervals(N, N, N, f0, N) == 1
    assert L.nicp_depth_to_cloud(N, N, N, N, N, 0, N, N) == 1
    assert L.nicp_raw_depth_to_cloud(N, N, 4, 4, C.c_float(0.001), 1, C.c_float(0.01), N, N, N, 0, N, N) == 1
    assert L.nicp_raw_depth_to_cloud_batch(N, 2, N, 4, 4, C.c_float(0.001), 1, C.c_float(0.01), N, N, N, 0, N) == 1
    assert L.nicp_stats_compute(N, N, 0, N, N, 4, 4, N, N, N, N, N, N) == 1
    assert L.nicp_information_compute(N, 0, N, N, N, N, N, N, N) == 1
    assert L.nicp_last_integral_image(N, N) == 1
    assert L.nicp_last_interval_image(N, N) == 1
    assert L.nicp_project(N, N, N, 4, 4, f0, f0, N, N) == 1
    assert L.nicp_correspond_linearize(N, N, N, N, N, 4, 4, N, N, N, N, N, N, N, N) == 1
    assert L.nicp_linearize(N, N, N, N, 0, N, N, N, N, N, N) == 1
    assert L.nicp_align(N, N, N, N, N, N, N, N, N, 0, f0, N) == 1
    assert L.nicp_align_get_state(N, N, N, N, N, N, N, N) == 1
    assert L.nicp_align_get_trace(N, N, 0) == 1
    assert L.nicp_statistics_tail(N, 1, N, N, N, N) == 1
    assert L.nicp_statistics_tail_host(1, N, N, N, N) == 1
    assert L.nicp_statistics_tail_host(-1, N, N, N, N) == 1
    assert L.nicp_statistics_tail_host(0, N, N, N, N) == 0
    assert L.nicp_align_batch(N, 0, N, N, N, N, N, N, N, f0, N) == 1
    assert L.nicp_align_batch_priors(N, 0, N, N, N, N, N, N, N, N, N, f0, N) == 1
    assert L.nicp_multi_depth_to_cloud(N, N, N, N, N, 0, N, N) == 1
    assert L.nicp_multi_project(N, N, N, N, N, N) == 1
    assert L.nicp_multi_align(N, N, N, N, N, N, N, N, N, 0, f0, N) == 1
    assert L.nicp_shard_pool_create(N, 0, N) == 1
    assert L.nicp_shard_pool_size(N) == 0
    assert L.nicp_align_frames_sharded(N, 0, N, 4, 4, C.c_float(0.001), 1, C.c_float(0.01), N, N, N, 0, N, N, N, N, f0, N) == 1
    L.nicp_shard_pool_destroy(N)
    L.nicp_destroy(N)
    L.nicp_cloud_destroy(N)
    rows, cols = C.c_int(7), C.c_int(7)
    L.nicp_multi_image_size(N, C.byref(rows), C.byref(cols))
    assert (rows.value, cols.value) == (0, 0)


@pytest.mark.skipif(not os.path.isdir("/root/reference/g2o_frontend/pwn_core"), reason="no reference tree (GPU box)")
def test_reference_artifacts_are_built_where_the_reference_exists():
    """where /root/reference exists (the build container) __graft_entry__.build() must have produced every compiled copy of
    the reference under oracle/_ref -- the tests that use them skip when they are absent, and a silent skip here would hide a
    broken reference build"""
    ref = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(ref) or not os.listdir(ref):
        pytest.skip("oracle/_ref is empty: __graft_entry__.build() has not run in this tree")
    for name in ("libpwn_core_ref.so", "libpwn_core_ref_fast.so", "libpwn_cuda_ref.so", "pwn_simple_aligner_ref", "pwn_aligner_ref",
                 "drop_in_demo"):
        assert os.path.exists(os.path.join(ref, name)), "oracle/_ref/%s missing: run __graft_entry__.build()" % name
    # and nothing but compiled artefacts: no reference source is copied into the repository
    for f in os.listdir(ref):
        assert not f.endswith((".cpp", ".h", ".hpp", ".cu", ".cuh", ".c")), f

"""ctypes binding of the C-ABI in include/nicp_b200.h (the CUDA library built from csrc/).

This is the thin Python face used by tests/, bench.py and __graft_entry__.py.  It never falls
back to a CPU implementation: if the shared library is missing, or no CUDA device works,
calls raise.  (The C++ host classes mirroring pwn:: live in include/pwn/.)
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_DIR = os.path.join(_HERE, "lib")

NICP_OK = 0

# every symbol include/nicp_b200.h declares (checked by tests/test_abi.py)
SYMBOLS = [
    "nicp_create", "nicp_destroy", "nicp_last_error", "nicp_synchronize", "nicp_is_verification_build",
    "nicp_launch_count", "nicp_stream", "nicp_set_kernel_timing", "nicp_get_kernel_timing",
    "nicp_update_matrices", "nicp_v2t", "nicp_t2v",
    "nicp_cloud_create", "nicp_cloud_destroy", "nicp_cloud_size", "nicp_cloud_upload", "nicp_cloud_download",
    "nicp_cloud_download_stats", "nicp_cloud_transform", "nicp_cloud_append",
    "nicp_depth_prepare", "nicp_unproject", "nicp_project_intervals", "nicp_depth_to_cloud",
    "nicp_raw_depth_to_cloud", "nicp_raw_depth_to_cloud_batch", "nicp_last_integral_image", "nicp_last_interval_image",
    "nicp_stats_compute", "nicp_information_compute",
    "nicp_project", "nicp_correspond_linearize", "nicp_linearize",
    "nicp_align", "nicp_align_get_state", "nicp_align_get_trace", "nicp_align_batch", "nicp_align_batch_priors",
    "nicp_statistics_tail", "nicp_statistics_tail_host",
    "nicp_multi_image_size", "nicp_multi_depth_to_cloud", "nicp_multi_project", "nicp_multi_align",
    "nicp_multi_raw_depth_to_cloud_batch", "nicp_multi_align_batch",
    "nicp_cloud_compute_gaussians", "nicp_multi_cloud_compute_gaussians", "nicp_cloud_has_gaussians",
    "nicp_cloud_download_gaussians", "nicp_cloud_upload_gaussians", "nicp_merge", "nicp_voxelize",
    "nicp_raw_depth_to_local_map", "nicp_multi_raw_depth_to_local_map",
    "nicp_shard_pool_create", "nicp_shard_pool_destroy", "nicp_shard_pool_size", "nicp_align_frames_sharded",
    "nicp_multi_align_frames_sharded",
    "nicp_frame_store_create", "nicp_multi_frame_store_create", "nicp_frame_store_destroy", "nicp_frame_store_add",
    "nicp_frame_store_remove", "nicp_frame_store_size", "nicp_frame_store_align", "nicp_frame_store_counters",
    "nicp_tracker_create", "nicp_multi_tracker_create", "nicp_tracker_destroy", "nicp_tracker_size", "nicp_tracker_step",
    "nicp_tracker_reset",
]

GAUSS_FLOATS = 24
GAUSS_MOMENTS, GAUSS_INFO = 1, 2


class Projector(C.Structure):
    _fields_ = [("K", C.c_float * 9), ("rows", C.c_int), ("cols", C.c_int),
                ("min_distance", C.c_float), ("max_distance", C.c_float)]


MAX_CAMERAS = 8


class MultiProjector(C.Structure):
    _fields_ = [("num_cameras", C.c_int), ("camera", Projector * MAX_CAMERAS),
                ("sensor_offset", (C.c_float * 16) * MAX_CAMERAS)]


class StatsParams(C.Structure):
    _fields_ = [("world_radius", C.c_float), ("min_image_radius", C.c_int), ("max_image_radius", C.c_int),
                ("min_points", C.c_int), ("curvature_threshold", C.c_float),
                ("omega_curvature_threshold", C.c_float), ("flat_omega_p", C.c_float * 3),
                ("flat_omega_n", C.c_float * 3), ("nonflat_omega_n", C.c_float * 3)]


class MergeParams(C.Structure):
    """Merger defaults (merger.cpp:5-13)"""
    _fields_ = [("distance_threshold", C.c_float), ("normal_threshold", C.c_float), ("max_point_depth", C.c_float)]


def make_merge_params(distance_threshold=0.1, normal_threshold=None, max_point_depth=10.0):
    if normal_threshold is None:
        normal_threshold = float(np.cos(np.float32(10 * np.pi / 180.0)))  # cosf(10 * M_PI / 180.0f)
    return MergeParams(distance_threshold, normal_threshold, max_point_depth)


class AlignParams(C.Structure):
    _fields_ = [("inlier_distance_threshold", C.c_float), ("inlier_normal_angular_threshold", C.c_float),
                ("flat_curvature_threshold", C.c_float), ("inlier_curvature_ratio_threshold", C.c_float),
                ("inlier_max_chi2", C.c_float), ("robust_kernel", C.c_int), ("outer_iterations", C.c_int),
                ("inner_iterations", C.c_int)]


class Prior(C.Structure):
    _fields_ = [("kind", C.c_int), ("mean", C.c_float * 16), ("reference", C.c_float * 16),
                ("information", C.c_float * 36)]


class AlignResult(C.Structure):
    _fields_ = [("T", C.c_float * 16), ("omega", C.c_float * 36), ("error", C.c_float), ("inliers", C.c_int),
                ("num_correspondences", C.c_int), ("image_non_zeros", C.c_int), ("image_inliers", C.c_int),
                ("image_outliers", C.c_int), ("image_reprojection_distance", C.c_float), ("status", C.c_int),
                ("translational_eigen_ratio", C.c_float), ("rotational_eigen_ratio", C.c_float),
                ("reserved", C.c_float * 2)]


assert C.sizeof(AlignResult) == 256

RESULT_DTYPE = np.dtype([("T", np.float32, 16), ("omega", np.float32, 36), ("error", np.float32),
                         ("inliers", np.int32), ("num_correspondences", np.int32), ("image_non_zeros", np.int32),
                         ("image_inliers", np.int32), ("image_outliers", np.int32),
                         ("image_reprojection_distance", np.float32), ("status", np.int32),
                         ("translational_eigen_ratio", np.float32), ("rotational_eigen_ratio", np.float32),
                         ("reserved", np.float32, 2)])
assert RESULT_DTYPE.itemsize == 256


class TrackResult(C.Structure):
    _fields_ = [("global_T", C.c_float * 16), ("relative_T", C.c_float * 16), ("guess", C.c_float * 16),
                ("frame", C.c_int), ("aligned", C.c_int), ("keyframe", C.c_int), ("num_keyframes", C.c_int),
                ("record", AlignResult)]


assert C.sizeof(TrackResult) == 464

TRACK_DTYPE = np.dtype([("global_T", np.float32, 16), ("relative_T", np.float32, 16), ("guess", np.float32, 16),
                        ("frame", np.int32), ("aligned", np.int32), ("keyframe", np.int32), ("num_keyframes", np.int32),
                        ("record", RESULT_DTYPE)])
assert TRACK_DTYPE.itemsize == 464


def lib_path(verify=False):
    return os.path.join(LIB_DIR, "libnicp_b200_verify.so" if verify else "libnicp_b200.so")


_LIBS = {}


def load(verify=False):
    """dlopen the CUDA library; raises if it has not been built (no fallback)."""
    key = bool(verify)
    if key in _LIBS:
        return _LIBS[key]
    path = lib_path(verify)
    if not os.path.exists(path):
        raise RuntimeError("%s is missing: build it with `make -C g2o_frontend_b200/csrc` "
                           "(or __graft_entry__.build()); there is no CPU fallback" % path)
    L = C.CDLL(path)
    L.nicp_last_error.restype = C.c_char_p
    L.nicp_launch_count.restype = C.c_longlong
    L.nicp_stream.restype = C.c_void_p
    L.nicp_destroy.restype = None
    L.nicp_cloud_destroy.restype = None
    L.nicp_update_matrices.restype = None
    L.nicp_v2t.restype = None
    L.nicp_t2v.restype = None
    L.nicp_multi_image_size.restype = None
    L.nicp_frame_store_destroy.restype = None
    L.nicp_tracker_destroy.restype = None
    for name in SYMBOLS:
        fn = getattr(L, name)
        if fn.restype is C.c_int:
            pass
    _LIBS[key] = L
    return L


class NicpError(RuntimeError):
    pass


def _check(L, rc):
    if rc != NICP_OK:
        raise NicpError("nicp error %d: %s" % (rc, L.nicp_last_error().decode()))


def colmajor(M):
    return np.ascontiguousarray(np.asarray(M, dtype=np.float32).T).reshape(-1)


def from_colmajor(v, n):
    return np.asarray(v, dtype=np.float32).reshape(n, n).T.copy()


def _fptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _iptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


def _guesses(guesses, n):
    """n (4, 4) poses -> pointer to n x 16 column-major floats (the pointer keeps the array alive); None -> NULL (identity)"""
    if guesses is None:
        return None
    return _fptr(np.ascontiguousarray(np.asarray(guesses, np.float32).transpose(0, 2, 1)).reshape(n, 16))


def _priors(priors, n):
    """None or n lists of Prior -> (priors, prior_offsets) arguments: pair i owns priors[offs[i] .. offs[i + 1])"""
    if priors is None:
        return None, None
    assert len(priors) == n
    flat = [p for ps in priors for p in ps]
    offs = np.zeros(n + 1, np.int32)
    offs[1:] = np.cumsum([len(ps) for ps in priors])
    return (Prior * max(len(flat), 1))(*flat), _iptr(offs)


def _rig_frames(frames, nc):
    """n rig frames of nc raw uint16 images each -> (the n * nc images, frame-major, as C-contiguous arrays, raw_rows,
    raw_cols); camera i must have the same shape in every frame"""
    imgs = []
    for fr in frames:
        assert len(fr) == nc, "a frame needs one raw image per camera"
        imgs += [np.ascontiguousarray(r, np.uint16) for r in fr]
    shapes = [im.shape for im in imgs[:nc]] if imgs else [(0, 0)] * nc
    for k, im in enumerate(imgs):
        assert im.shape == shapes[k % nc], "camera %d has a different raw size in frame %d" % (k % nc, k // nc)
    return imgs, np.array([s[0] for s in shapes], np.int32), np.array([s[1] for s in shapes], np.int32)


def _per_camera(v, mp):
    """a scalar for every camera of the rig, or one value per camera -> mp.num_cameras float32"""
    a = np.asarray(v, np.float32)
    a = np.full(mp.num_cameras, a, np.float32) if a.ndim == 0 else np.ascontiguousarray(a)
    assert a.shape == (mp.num_cameras,), "one value per camera"
    return a


def make_projector(K, rows, cols, min_distance=0.01, max_distance=6.0):
    p = Projector()
    p.K[:] = colmajor(K).tolist()
    p.rows, p.cols = int(rows), int(cols)
    p.min_distance, p.max_distance = min_distance, max_distance
    return p


def make_multi_projector(cameras):
    """cameras: list of dicts {K, width, height, minD, maxD, offset} (addPointProjector(p, offset, width, height))"""
    m = MultiProjector()
    m.num_cameras = len(cameras)
    for i, c in enumerate(cameras):
        m.camera[i] = make_projector(c["K"], c["width"], c["height"], c["minD"], c["maxD"])
        m.sensor_offset[i][:] = colmajor(c["offset"]).tolist()
    return m


def multi_image_size(mp, verify=False):
    r, c = C.c_int(0), C.c_int(0)
    load(verify).nicp_multi_image_size(C.byref(mp), C.byref(r), C.byref(c))
    return r.value, c.value


def make_stats_params(world_radius=0.1, min_image_radius=10, max_image_radius=30, min_points=50,
                      curvature_threshold=0.02, omega_curvature_threshold=0.02,
                      flat_omega_p=(1000.0, 1.0, 1.0), flat_omega_n=(100.0, 100.0, 100.0),
                      nonflat_omega_n=(1.0, 1.0, 1.0)):
    s = StatsParams()
    s.world_radius = world_radius
    s.min_image_radius, s.max_image_radius, s.min_points = min_image_radius, max_image_radius, min_points
    s.curvature_threshold, s.omega_curvature_threshold = curvature_threshold, omega_curvature_threshold
    s.flat_omega_p[:] = list(flat_omega_p)
    s.flat_omega_n[:] = list(flat_omega_n)
    s.nonflat_omega_n[:] = list(nonflat_omega_n)
    return s


def make_prior(kind, mean, information, reference=None):
    """kind 0 = SE3RelativePrior(mean, information), 1 = SE3AbsolutePrior(reference, mean, information)"""
    p = Prior()
    p.kind = int(kind)
    p.mean[:] = colmajor(mean).tolist()
    p.reference[:] = colmajor(np.eye(4) if reference is None else reference).tolist()
    p.information[:] = colmajor(information).tolist()
    return p


def make_align_params(inlier_distance_threshold=0.5, inlier_normal_angular_threshold=float(np.cos(np.pi / 6)),
                      flat_curvature_threshold=0.02, inlier_curvature_ratio_threshold=1.3, inlier_max_chi2=9e3,
                      robust_kernel=True, outer_iterations=10, inner_iterations=1):
    a = AlignParams()
    a.inlier_distance_threshold = inlier_distance_threshold
    a.inlier_normal_angular_threshold = inlier_normal_angular_threshold
    a.flat_curvature_threshold = flat_curvature_threshold
    a.inlier_curvature_ratio_threshold = inlier_curvature_ratio_threshold
    a.inlier_max_chi2 = inlier_max_chi2
    a.robust_kernel = int(robust_kernel)
    a.outer_iterations, a.inner_iterations = outer_iterations, inner_iterations
    return a


class Cloud:
    def __init__(self, ctx, capacity):
        self.ctx = ctx
        self.capacity = int(capacity)
        self.handle = C.c_void_p()
        _check(ctx.L, ctx.L.nicp_cloud_create(ctx.handle, self.capacity, C.byref(self.handle)))

    def close(self):
        if self.handle:
            self.ctx.L.nicp_cloud_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def size(self):
        return self.ctx.L.nicp_cloud_size(self.handle)

    def upload(self, points4, normals4=None, curvature=None, omega_p6=None, omega_n6=None):
        pts = np.ascontiguousarray(points4, np.float32)
        n = pts.shape[0]
        keep = [pts]

        def opt(a, w):
            if a is None:
                return None
            a = np.ascontiguousarray(a, np.float32)
            assert a.size == n * w
            keep.append(a)
            return _fptr(a)

        _check(self.ctx.L, self.ctx.L.nicp_cloud_upload(self.ctx.handle, self.handle, n, _fptr(pts), opt(normals4, 4),
                                                         opt(curvature, 1), opt(omega_p6, 6), opt(omega_n6, 6)))
        return self

    def download(self):
        n = self.size()
        out = {"points": np.zeros((n, 4), np.float32), "normals": np.zeros((n, 4), np.float32),
               "curvature": np.zeros(n, np.float32), "omega_p": np.zeros((n, 6), np.float32),
               "omega_n": np.zeros((n, 6), np.float32)}
        _check(self.ctx.L, self.ctx.L.nicp_cloud_download(self.ctx.handle, self.handle, _fptr(out["points"]),
                                                           _fptr(out["normals"]), _fptr(out["curvature"]),
                                                           _fptr(out["omega_p"]), _fptr(out["omega_n"])))
        return out

    def download_stats(self):
        n = self.size()
        s16 = np.zeros((n, 16), np.float32)
        ev = np.zeros((n, 3), np.float32)
        cnt = np.zeros(n, np.int32)
        _check(self.ctx.L, self.ctx.L.nicp_cloud_download_stats(self.ctx.handle, self.handle, _fptr(s16), _fptr(ev),
                                                                 _iptr(cnt)))
        return s16, ev, cnt

    def transform(self, T):
        t = colmajor(T)
        _check(self.ctx.L, self.ctx.L.nicp_cloud_transform(self.ctx.handle, self.handle, _fptr(t)))

    # ---- local-map maintenance (Gaussian3f sensor model, Merger, VoxelCalculator) ----
    def compute_gaussians(self, depth, proj, baseline=0.075, alpha=0.1, sensor_offset=None):
        """gaussians of PinholePointProjector::unProject for the depth image this cloud was built from"""
        d = np.ascontiguousarray(depth, np.float32)
        so = colmajor(np.eye(4) if sensor_offset is None else sensor_offset)
        _check(self.ctx.L, self.ctx.L.nicp_cloud_compute_gaussians(self.ctx.handle, self.handle, _fptr(d), C.byref(proj),
                                                                    C.c_float(baseline), C.c_float(alpha), _fptr(so)))

    def multi_compute_gaussians(self, depth, mp, baseline=0.075, alpha=0.1, sensor_offset=None):
        """the rig gaussians (nicp_multi_cloud_compute_gaussians) for the composite depth image this cloud was built from;
        baseline / alpha: a scalar for every camera or one value per camera"""
        d = np.ascontiguousarray(depth, np.float32)
        so = colmajor(np.eye(4) if sensor_offset is None else sensor_offset)
        b, a = _per_camera(baseline, mp), _per_camera(alpha, mp)
        _check(self.ctx.L, self.ctx.L.nicp_multi_cloud_compute_gaussians(self.ctx.handle, self.handle, _fptr(d), C.byref(mp),
                                                                          _fptr(b), _fptr(a), _fptr(so)))

    def has_gaussians(self):
        return bool(self.ctx.L.nicp_cloud_has_gaussians(self.handle))

    def download_gaussians(self):
        n = self.size()
        g = np.zeros((n, GAUSS_FLOATS), np.float32)
        f = np.zeros(n, np.int32)
        _check(self.ctx.L, self.ctx.L.nicp_cloud_download_gaussians(self.ctx.handle, self.handle, _fptr(g), _iptr(f)))
        return g, f

    def upload_gaussians(self, gauss, flags):
        g = np.ascontiguousarray(gauss, np.float32)
        f = np.ascontiguousarray(flags, np.int32)
        assert g.shape == (self.size(), GAUSS_FLOATS) and f.shape == (self.size(),)
        _check(self.ctx.L, self.ctx.L.nicp_cloud_upload_gaussians(self.ctx.handle, self.handle, _fptr(g), _iptr(f)))

    def merge(self, proj, T=None, params=None):
        """Merger::merge(cloud, T) -> (new size, _collapsedIndices of the input points)"""
        n = self.size()
        t = colmajor(np.eye(4) if T is None else T)
        mp = params if params is not None else make_merge_params()
        collapsed = np.zeros(max(n, 1), np.int32)
        new_size = C.c_int(0)
        _check(self.ctx.L, self.ctx.L.nicp_merge(self.ctx.handle, self.handle, C.byref(proj), _fptr(t), C.byref(mp),
                                                  _iptr(collapsed), C.byref(new_size)))
        return new_size.value, collapsed[:n]

    def voxelize(self, resolution=0.01):
        """VoxelCalculator::compute(cloud, resolution) -> (new size, indices of the kept input points in output order)"""
        n = self.size()
        rep = np.zeros(max(n, 1), np.int32)
        new_size = C.c_int(0)
        _check(self.ctx.L, self.ctx.L.nicp_voxelize(self.ctx.handle, self.handle, C.c_float(resolution), _iptr(rep),
                                                     C.byref(new_size)))
        return new_size.value, rep[:new_size.value].copy()

    def append(self, other, T=None):
        """Cloud::add(other, T): append a transformed copy of `other`"""
        t = colmajor(np.eye(4) if T is None else T)
        _check(self.ctx.L, self.ctx.L.nicp_cloud_append(self.ctx.handle, self.handle, other.handle, _fptr(t)))


class Context:
    """One nicp_context (one GPU, one stream)."""

    def __init__(self, device=0, verify=False):
        self.L = load(verify)
        self.verify = verify
        self.device = int(device)
        self.handle = C.c_void_p()
        _check(self.L, self.L.nicp_create(int(device), C.byref(self.handle)))

    def close(self):
        if self.handle:
            self.L.nicp_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def synchronize(self):
        _check(self.L, self.L.nicp_synchronize(self.handle))

    def launch_count(self):
        return int(self.L.nicp_launch_count(self.handle))

    def stream(self):
        return self.L.nicp_stream(self.handle)

    def set_kernel_timing(self, enable=True):
        _check(self.L, self.L.nicp_set_kernel_timing(self.handle, int(enable)))

    def kernel_timing(self):
        """{'corr_lin_ms', 'corr_lin_launches', 'project_ms', 'project_launches'} since the last enable"""
        a, b = C.c_double(0), C.c_double(0)
        na, nb = C.c_longlong(0), C.c_longlong(0)
        _check(self.L, self.L.nicp_get_kernel_timing(self.handle, C.byref(a), C.byref(na), C.byref(b), C.byref(nb)))
        return {"corr_lin_ms": a.value, "corr_lin_launches": na.value, "project_ms": b.value,
                "project_launches": nb.value}

    def new_cloud(self, capacity):
        return Cloud(self, capacity)

    # ---- depth helpers
    def depth_prepare(self, raw, depth_scale=0.001, step=1, max_depth_cov=0.01):
        raw = np.ascontiguousarray(raw, np.uint16)
        rows, cols = raw.shape
        out = np.zeros((rows // max(step, 1), cols // max(step, 1)), np.float32)
        _check(self.L, self.L.nicp_depth_prepare(self.handle, raw.ctypes.data_as(C.POINTER(C.c_uint16)), rows, cols,
                                                 C.c_float(depth_scale), int(step), C.c_float(max_depth_cov), _fptr(out)))
        return out

    # ---- frame preparation
    def unproject(self, depth, iKRt, min_distance, max_distance, cloud=None):
        depth = np.ascontiguousarray(depth, np.float32)
        rows, cols = depth.shape
        cloud = cloud or self.new_cloud(rows * cols)
        index = np.zeros((rows, cols), np.int32)
        m = colmajor(iKRt)
        _check(self.L, self.L.nicp_unproject(self.handle, _fptr(depth), rows, cols, _fptr(m), C.c_float(min_distance),
                                             C.c_float(max_distance), cloud.handle, _iptr(index)))
        return cloud, index

    def project_intervals(self, depth, proj, world_radius):
        depth = np.ascontiguousarray(depth, np.float32)
        out = np.zeros(depth.shape, np.int32)
        _check(self.L, self.L.nicp_project_intervals(self.handle, _fptr(depth), C.byref(proj), C.c_float(world_radius),
                                                     _iptr(out)))
        return out

    def depth_to_cloud(self, depth, proj, sp, sensor_offset=None, keep_stats=False, cloud=None, want_index=True):
        depth = np.ascontiguousarray(depth, np.float32)
        assert depth.shape == (proj.rows, proj.cols)
        cloud = cloud or self.new_cloud(proj.rows * proj.cols)
        index = np.zeros(depth.shape, np.int32) if want_index else None
        so = colmajor(np.eye(4) if sensor_offset is None else sensor_offset)
        _check(self.L, self.L.nicp_depth_to_cloud(self.handle, _fptr(depth), C.byref(proj), C.byref(sp), _fptr(so),
                                                  int(keep_stats), cloud.handle,
                                                  _iptr(index) if want_index else None))
        return cloud, index

    def raw_depth_to_cloud(self, raw, proj, sp, depth_scale=0.001, step=1, max_depth_cov=0.01, sensor_offset=None,
                           keep_stats=False, cloud=None, want_index=False):
        """raw may be a numpy uint16 array or an integer host address (pinned buffer) with raw_shape."""
        raw = np.ascontiguousarray(raw, np.uint16)
        rows, cols = raw.shape
        cloud = cloud or self.new_cloud(proj.rows * proj.cols)
        index = np.zeros((proj.rows, proj.cols), np.int32) if want_index else None
        so = colmajor(np.eye(4) if sensor_offset is None else sensor_offset)
        _check(self.L, self.L.nicp_raw_depth_to_cloud(self.handle, raw.ctypes.data_as(C.POINTER(C.c_uint16)), rows, cols,
                                                      C.c_float(depth_scale), int(step), C.c_float(max_depth_cov),
                                                      C.byref(proj), C.byref(sp), _fptr(so), int(keep_stats),
                                                      cloud.handle, _iptr(index) if want_index else None))
        return cloud, index

    def raw_depth_to_cloud_batch(self, raws, proj, sp, depth_scale=0.001, step=1, max_depth_cov=0.01, sensor_offset=None,
                                 keep_stats=False, clouds=None):
        """n raw frames (uint16 arrays of one shape, or rows of one 3-D array -- e.g. a pinned staging buffer) -> n clouds
        with one launch set per sub-batch (nicp_raw_depth_to_cloud_batch).  Asynchronous like raw_depth_to_cloud."""
        n = len(raws)
        frames = [r if (isinstance(r, np.ndarray) and r.dtype == np.uint16 and r.flags.c_contiguous)
                  else np.ascontiguousarray(r, np.uint16) for r in raws]
        rows, cols = frames[0].shape
        clouds = clouds or [self.new_cloud(proj.rows * proj.cols) for _ in range(n)]
        so = colmajor(np.eye(4) if sensor_offset is None else sensor_offset)
        RA = (C.c_void_p * n)(*[f.ctypes.data for f in frames])
        CA = (C.c_void_p * n)(*[c.handle for c in clouds])
        _check(self.L, self.L.nicp_raw_depth_to_cloud_batch(self.handle, n, RA, rows, cols, C.c_float(depth_scale), int(step),
                                                            C.c_float(max_depth_cov), C.byref(proj), C.byref(sp), _fptr(so),
                                                            int(keep_stats), CA))
        self._keepalive = frames  # the copies are asynchronous: keep the host frames alive until the next call
        return clouds

    def raw_depth_to_local_map(self, raws, proj, sp, poses, map_cloud, depth_scale=0.001, step=1, max_depth_cov=0.01,
                               sensor_offset=None, baseline=0.075, alpha=0.1, merge_params=None, merge_transform=None,
                               voxel_resolution=0.0):
        """n raw frames (uint16 arrays of one shape) with n (4, 4) poses -> appended to map_cloud with their sensor-model
        gaussians, then Merger::merge(merge_params, merge_transform; identity if None) if merge_params is given, then
        VoxelCalculator::compute(voxel_resolution) if it is > 0 (nicp_raw_depth_to_local_map).  Synchronous.  Returns
        (appended points, new size, collapsed indices of the merged points or None, voxel representatives or None).  A map
        too small raises NicpError with `needed_size` (the size the map would need); the map is left as it was."""
        n = len(raws)
        frames = [r if (isinstance(r, np.ndarray) and r.dtype == np.uint16 and r.flags.c_contiguous)
                  else np.ascontiguousarray(r, np.uint16) for r in raws]
        rows, cols = frames[0].shape
        assert all(f.shape == (rows, cols) for f in frames), "every raw frame needs the same shape"
        P = np.asarray(poses, np.float32)
        assert P.shape == (n, 4, 4), "one (4, 4) pose per frame"
        pp = np.ascontiguousarray(P.transpose(0, 2, 1)).reshape(n, 16)
        so = colmajor(np.eye(4) if sensor_offset is None else sensor_offset)
        mt = colmajor(np.eye(4) if merge_transform is None else merge_transform)
        RA = (C.c_void_p * max(n, 1))(*[f.ctypes.data for f in frames])
        return self._local_map_call(
            map_cloud, merge_params, voxel_resolution,
            lambda outs: self.L.nicp_raw_depth_to_local_map(
                self.handle, n, RA, rows, cols, C.c_float(depth_scale), int(step), C.c_float(max_depth_cov), C.byref(proj),
                C.byref(sp), _fptr(so), C.c_float(baseline), C.c_float(alpha), _fptr(pp),
                C.byref(merge_params) if merge_params is not None else None, _fptr(mt), C.c_float(voxel_resolution),
                map_cloud.handle, *outs))

    def multi_raw_depth_to_local_map(self, frames, mp, sp, poses, map_cloud, depth_scale=0.001, step=1, max_depth_cov=0.01,
                                     sensor_offset=None, baseline=0.075, alpha=0.1, merge_proj=None, merge_params=None,
                                     merge_transform=None, voxel_resolution=0.0):
        """raw_depth_to_local_map for rig frames (nicp_multi_raw_depth_to_local_map): frames as in
        multi_raw_depth_to_cloud_batch, baseline / alpha a scalar or one value per camera; the merge runs through the
        pinhole view merge_proj, which merge_params needs.  Returns what raw_depth_to_local_map returns."""
        n = len(frames)
        imgs, rr, rc = _rig_frames(frames, mp.num_cameras)
        P = np.asarray(poses, np.float32)
        assert P.shape == (n, 4, 4), "one (4, 4) pose per frame"
        assert merge_params is None or merge_proj is not None, "a merge needs merge_proj (a pinhole merge view)"
        pp = np.ascontiguousarray(P.transpose(0, 2, 1)).reshape(n, 16)
        so = colmajor(np.eye(4) if sensor_offset is None else sensor_offset)
        mt = colmajor(np.eye(4) if merge_transform is None else merge_transform)
        b, a = _per_camera(baseline, mp), _per_camera(alpha, mp)
        RA = (C.c_void_p * max(len(imgs), 1))(*[im.ctypes.data for im in imgs])
        return self._local_map_call(
            map_cloud, merge_params, voxel_resolution,
            lambda outs: self.L.nicp_multi_raw_depth_to_local_map(
                self.handle, n, RA, _iptr(rr), _iptr(rc), C.c_float(depth_scale), int(step), C.c_float(max_depth_cov),
                C.byref(mp), C.byref(sp), _fptr(so), _fptr(b), _fptr(a), _fptr(pp),
                C.byref(merge_proj) if merge_proj is not None else None,
                C.byref(merge_params) if merge_params is not None else None, _fptr(mt), C.c_float(voxel_resolution),
                map_cloud.handle, *outs))

    def _local_map_call(self, map_cloud, merge_params, voxel_resolution, call):
        """runs call((appended_size, new_size, collapsed, representatives)) of a local-map entry -> its Python results"""
        before = map_cloud.size()
        collapsed = np.zeros(map_cloud.capacity, np.int32) if merge_params is not None else None
        reps = np.zeros(map_cloud.capacity, np.int32) if voxel_resolution > 0 else None
        appended, new_size = C.c_int(0), C.c_int(0)
        rc = call((C.byref(appended), C.byref(new_size), _iptr(collapsed) if collapsed is not None else None,
                   _iptr(reps) if reps is not None else None))
        if rc != NICP_OK:
            err = NicpError("nicp error %d: %s" % (rc, self.L.nicp_last_error().decode()))
            err.needed_size = new_size.value
            raise err
        merged = before + appended.value
        if collapsed is not None:
            collapsed = collapsed[:merged].copy()
        if reps is not None:
            reps = reps[:new_size.value].copy()
        return appended.value, new_size.value, collapsed, reps

    def stats_compute(self, points, index, interval, sp):
        """StatsCalculatorIntegralImage::compute(normals, stats, points, indexImage) with its interval image"""
        pts = np.ascontiguousarray(points, np.float32)
        n = pts.shape[0]
        idx = np.ascontiguousarray(index, np.int32)
        itv = np.ascontiguousarray(interval, np.int32)
        rows, cols = idx.shape
        out = {"normals": np.zeros((n, 4), np.float32), "stats16": np.zeros((n, 16), np.float32),
               "eigenvalues": np.zeros((n, 3), np.float32), "n": np.zeros(n, np.int32), "curvature": np.zeros(n, np.float32)}
        _check(self.L, self.L.nicp_stats_compute(self.handle, _fptr(pts), n, _iptr(idx), _iptr(itv), rows, cols, C.byref(sp),
                                                 _fptr(out["normals"]), _fptr(out["stats16"]), _fptr(out["eigenvalues"]),
                                                 _iptr(out["n"]), _fptr(out["curvature"])))
        return out

    def information_compute(self, normals, stats16, eigenvalues, curvature, sp):
        """Point / NormalInformationMatrixCalculator::compute: (n, 6) upper triangles"""
        n = normals.shape[0]
        op, on = np.zeros((n, 6), np.float32), np.zeros((n, 6), np.float32)
        _check(self.L, self.L.nicp_information_compute(self.handle, n, _fptr(np.ascontiguousarray(normals, np.float32)),
                                                       _fptr(np.ascontiguousarray(stats16, np.float32)),
                                                       _fptr(np.ascontiguousarray(eigenvalues, np.float32)),
                                                       _fptr(np.ascontiguousarray(curvature, np.float32)), C.byref(sp),
                                                       _fptr(op), _fptr(on)))
        return op, on

    def last_integral_image(self, rows, cols):
        out = np.zeros((rows, cols, 10), np.float32)
        _check(self.L, self.L.nicp_last_integral_image(self.handle, _fptr(out)))
        return out

    def last_interval_image(self, rows, cols):
        out = np.zeros((rows, cols), np.int32)
        _check(self.L, self.L.nicp_last_interval_image(self.handle, _iptr(out)))
        return out

    # ---- projection
    def project(self, cloud, KRt, rows, cols, min_distance, max_distance):
        index = np.zeros((rows, cols), np.int32)
        depth = np.zeros((rows, cols), np.float32)
        m = colmajor(KRt)
        _check(self.L, self.L.nicp_project(self.handle, cloud.handle, _fptr(m), rows, cols, C.c_float(min_distance),
                                           C.c_float(max_distance), _iptr(index), _fptr(depth)))
        return index, depth

    # ---- stage-level finder + lineariser
    def correspond_linearize(self, ref, cur, ref_index, cur_index, T, ap):
        ri = np.ascontiguousarray(ref_index, np.int32)
        ci = np.ascontiguousarray(cur_index, np.int32)
        rows, cols = ri.shape
        t = colmajor(T)
        H = np.zeros(36, np.float32)
        b = np.zeros(6, np.float32)
        err, inl, nc = C.c_float(0), C.c_int(0), C.c_int(0)
        cimg = np.zeros((rows, cols), np.int32)
        _check(self.L, self.L.nicp_correspond_linearize(self.handle, ref.handle, cur.handle, _iptr(ri), _iptr(ci), rows,
                                                        cols, _fptr(t), C.byref(ap), _fptr(H), _fptr(b), C.byref(err),
                                                        C.byref(inl), C.byref(nc), _iptr(cimg)))
        return from_colmajor(H, 6), b, err.value, inl.value, nc.value, cimg

    def linearize(self, ref, cur, corr, T, ap):
        corr = np.ascontiguousarray(corr, np.int32)
        t = colmajor(T)
        H = np.zeros(36, np.float32)
        b = np.zeros(6, np.float32)
        err, inl = C.c_float(0), C.c_int(0)
        _check(self.L, self.L.nicp_linearize(self.handle, ref.handle, cur.handle, _iptr(corr), corr.shape[0], _fptr(t),
                                             C.byref(ap), _fptr(H), _fptr(b), C.byref(err), C.byref(inl)))
        return from_colmajor(H, 6), b, err.value, inl.value

    # ---- alignment
    def align(self, ref, cur, proj, ap, ref_offset=None, cur_offset=None, guess=None, img_threshold=50.0, priors=()):
        """priors: sequence of Prior (make_prior) -- Aligner::addRelativePrior / addAbsolutePrior"""
        eye = np.eye(4, dtype=np.float32)
        ro = colmajor(eye if ref_offset is None else ref_offset)
        co = colmajor(eye if cur_offset is None else cur_offset)
        g = colmajor(eye if guess is None else guess)
        res = AlignResult()
        parr = (Prior * len(priors))(*priors) if len(priors) else None
        _check(self.L, self.L.nicp_align(self.handle, ref.handle, cur.handle, C.byref(proj), C.byref(ap), _fptr(ro),
                                         _fptr(co), _fptr(g), parr, len(priors), C.c_float(img_threshold), C.byref(res)))
        return res

    # ---- MultiPointProjector
    def multi_depth_to_cloud(self, depth, mp, sp, sensor_offset=None, keep_stats=False, cloud=None):
        depth = np.ascontiguousarray(depth, np.float32)
        rows, cols = multi_image_size(mp, self.verify)
        assert depth.shape == (rows, cols)
        cloud = cloud or self.new_cloud(rows * cols)
        index = np.zeros((rows, cols), np.int32)
        so = colmajor(np.eye(4) if sensor_offset is None else sensor_offset)
        _check(self.L, self.L.nicp_multi_depth_to_cloud(self.handle, _fptr(depth), C.byref(mp), C.byref(sp), _fptr(so),
                                                        int(keep_stats), cloud.handle, _iptr(index)))
        return cloud, index

    def multi_project(self, cloud, mp, T):
        rows, cols = multi_image_size(mp, self.verify)
        index = np.zeros((rows, cols), np.int32)
        depth = np.zeros((rows, cols), np.float32)
        t = colmajor(T)
        _check(self.L, self.L.nicp_multi_project(self.handle, cloud.handle, C.byref(mp), _fptr(t), _iptr(index), _fptr(depth)))
        return index, depth

    def multi_align(self, ref, cur, mp, ap, ref_offset=None, cur_offset=None, guess=None, img_threshold=50.0, priors=()):
        eye = np.eye(4, dtype=np.float32)
        ro = colmajor(eye if ref_offset is None else ref_offset)
        co = colmajor(eye if cur_offset is None else cur_offset)
        g = colmajor(eye if guess is None else guess)
        res = AlignResult()
        parr = (Prior * len(priors))(*priors) if len(priors) else None
        _check(self.L, self.L.nicp_multi_align(self.handle, ref.handle, cur.handle, C.byref(mp), C.byref(ap), _fptr(ro),
                                               _fptr(co), _fptr(g), parr, len(priors), C.c_float(img_threshold), C.byref(res)))
        return res

    def multi_raw_depth_to_cloud_batch(self, frames, mp, sp, depth_scale=0.001, step=1, max_depth_cov=0.01, sensor_offset=None,
                                       keep_stats=False, clouds=None):
        """n rig frames -> n clouds (nicp_multi_raw_depth_to_cloud_batch).  frames: n sequences of mp.num_cameras raw uint16
        images in sensor orientation (camera i: (height_i * step) x (width_i * step), the same shape in every frame), numpy
        arrays or numpy views of pinned buffers.  Asynchronous like raw_depth_to_cloud_batch."""
        n = len(frames)
        imgs, rr, rc = _rig_frames(frames, mp.num_cameras)
        rows, cols = multi_image_size(mp, self.verify)
        clouds = clouds or [self.new_cloud(rows * cols) for _ in range(n)]
        so = colmajor(np.eye(4) if sensor_offset is None else sensor_offset)
        RA = (C.c_void_p * max(len(imgs), 1))(*[im.ctypes.data for im in imgs])
        CA = (C.c_void_p * max(n, 1))(*[c.handle for c in clouds])
        _check(self.L, self.L.nicp_multi_raw_depth_to_cloud_batch(self.handle, n, RA, _iptr(rr), _iptr(rc), C.c_float(depth_scale),
                                                                  int(step), C.c_float(max_depth_cov), C.byref(mp), C.byref(sp),
                                                                  _fptr(so), int(keep_stats), CA))
        self._keepalive = imgs  # the copies are asynchronous: keep the host frames alive until the next call
        return clouds

    def multi_align_batch(self, refs, curs, mp, ap, guesses=None, ref_offset=None, cur_offset=None, img_threshold=50.0,
                          results=None, priors=None):
        """align_batch with a MultiPointProjector (nicp_multi_align_batch): record i equals multi_align on pair i.
        priors: None or n lists of Prior.  Returns a numpy structured array (RESULT_DTYPE) of n records."""
        n = len(refs)
        assert len(curs) == n
        eye = np.eye(4, dtype=np.float32)
        ro = colmajor(eye if ref_offset is None else ref_offset)
        co = colmajor(eye if cur_offset is None else cur_offset)
        RA = (C.c_void_p * max(n, 1))(*[r.handle for r in refs])
        CA = (C.c_void_p * max(n, 1))(*[c.handle for c in curs])
        if results is None:
            results = np.zeros(n, RESULT_DTYPE)
        parr, offs = _priors(priors, n)
        _check(self.L, self.L.nicp_multi_align_batch(self.handle, n, RA, CA, C.byref(mp), C.byref(ap), _fptr(ro), _fptr(co),
                                                     _guesses(guesses, n), parr, offs, C.c_float(img_threshold),
                                                     results.ctypes.data_as(C.POINTER(AlignResult))))
        return results

    def align_state(self, rows, cols, max_corr=None):
        ri = np.zeros((rows, cols), np.int32)
        rd = np.zeros((rows, cols), np.float32)
        ci = np.zeros((rows, cols), np.int32)
        cd = np.zeros((rows, cols), np.float32)
        corr = np.full((rows * cols, 2), -1, np.int32)
        H = np.zeros(36, np.float32)
        b = np.zeros(6, np.float32)
        _check(self.L, self.L.nicp_align_get_state(self.handle, _iptr(ri), _fptr(rd), _iptr(ci), _fptr(cd), _iptr(corr),
                                                   _fptr(H), _fptr(b)))
        n = int((corr[:, 0] >= 0).sum())
        return {"ref_index": ri, "ref_depth": rd, "cur_index": ci, "cur_depth": cd, "corr": corr[:n],
                "H": from_colmajor(H, 6), "b": b}

    def align_trace(self, iters):
        tr = np.zeros((iters, 61), np.float32)
        _check(self.L, self.L.nicp_align_get_trace(self.handle, _fptr(tr), iters))
        return tr

    def statistics_tail(self, H, T):
        """the batch's _computeStatistics tail kernel on n caller-given linearisations (test hook): H (n, 36) and T (n, 16)
        column-major -> omega (n, 36) column-major, ratios (n, 2) = (translational, rotational)"""
        H, T, omega, ratios = _tail_args(H, T)
        _check(self.L, self.L.nicp_statistics_tail(self.handle, H.shape[0], _fptr(H), _fptr(T), _fptr(omega), _fptr(ratios)))
        return omega, ratios

    def align_batch(self, refs, curs, proj, ap, guesses=None, ref_offset=None, cur_offset=None, img_threshold=50.0,
                    results=None, priors=None):
        """refs/curs: sequences of Cloud.  guesses: (n,4,4) row/col matrices or None.  priors: None or a sequence of
        n lists of Prior (nicp_align_batch_priors).  Returns a numpy structured array (RESULT_DTYPE) of n 256-byte records."""
        n = len(refs)
        assert len(curs) == n
        eye = np.eye(4, dtype=np.float32)
        ro = colmajor(eye if ref_offset is None else ref_offset)
        co = colmajor(eye if cur_offset is None else cur_offset)
        RA = (C.c_void_p * n)(*[r.handle for r in refs])
        CA = (C.c_void_p * n)(*[c.handle for c in curs])
        if results is None:
            results = np.zeros(n, RESULT_DTYPE)
        parr, offs = _priors(priors, n)
        _check(self.L, self.L.nicp_align_batch_priors(self.handle, n, RA, CA, C.byref(proj), C.byref(ap), _fptr(ro), _fptr(co),
                                                      _guesses(guesses, n), parr, offs, C.c_float(img_threshold),
                                                      results.ctypes.data_as(C.POINTER(AlignResult))))
        return results


def update_matrices(K, T, verify=False):
    """PinholePointProjector::_updateMatrices through the library (host-side, no GPU needed)."""
    L = load(verify)
    k, t = colmajor(K), colmajor(T)
    KRt, iKRt = np.zeros(16, np.float32), np.zeros(16, np.float32)
    L.nicp_update_matrices(_fptr(k), _fptr(t), _fptr(KRt), _fptr(iKRt))
    return from_colmajor(KRt, 4), from_colmajor(iKRt, 4)


def _tail_args(H, T):
    H = np.ascontiguousarray(H, np.float32).reshape(-1, 36)
    T = np.ascontiguousarray(T, np.float32).reshape(-1, 16)
    assert H.shape[0] == T.shape[0]
    return H, T, np.zeros((H.shape[0], 36), np.float32), np.zeros((H.shape[0], 2), np.float32)


def statistics_tail_host(H, T, verify=False):
    """the host function that finishes a single alignment's record (test hook, no GPU needed): Context.statistics_tail's
    arguments and results"""
    L = load(verify)
    H, T, omega, ratios = _tail_args(H, T)
    _check(L, L.nicp_statistics_tail_host(H.shape[0], _fptr(H), _fptr(T), _fptr(omega), _fptr(ratios)))
    return omega, ratios


def result_T(res):
    return from_colmajor(np.array(res.T[:], np.float32), 4)


def result_omega(res):
    return from_colmajor(np.array(res.omega[:], np.float32), 6)


class ShardPool:
    """nicp_shard_pool: one worker thread + context per listed device (a device may be listed twice)"""

    def __init__(self, devices, verify=False):
        self.L = load(verify)
        self.handle = C.c_void_p()
        arr = (C.c_int * len(devices))(*devices)
        rc = self.L.nicp_shard_pool_create(arr, len(devices), C.byref(self.handle))
        if rc != NICP_OK:
            raise NicpError("nicp_shard_pool_create failed (%d): %s" % (rc, self.L.nicp_last_error().decode()))

    def size(self):
        return int(self.L.nicp_shard_pool_size(self.handle))

    def align_frames(self, raws, proj, sp, ref_frame, cur_frame, guesses, ap, depth_scale=0.001, step=1, max_depth_cov=0.01,
                     sensor_offset=None, img_threshold=50.0):
        """raws: list of uint16 frames; pair i = (ref_frame[i], cur_frame[i]); returns RESULT_DTYPE records"""
        frames = [np.ascontiguousarray(r, np.uint16) for r in raws]
        rows, cols = frames[0].shape
        n = len(ref_frame)
        RA = (C.c_void_p * len(frames))(*[f.ctypes.data for f in frames])
        rf = np.ascontiguousarray(ref_frame, np.int32)
        cf = np.ascontiguousarray(cur_frame, np.int32)
        so = colmajor(np.eye(4) if sensor_offset is None else sensor_offset)
        results = np.zeros(n, RESULT_DTYPE)
        _check(self.L, self.L.nicp_align_frames_sharded(self.handle, len(frames), RA, rows, cols, C.c_float(depth_scale), int(step),
                                                        C.c_float(max_depth_cov), C.byref(proj), C.byref(sp), _fptr(so), n,
                                                        _iptr(rf), _iptr(cf), _guesses(guesses, n), C.byref(ap),
                                                        C.c_float(img_threshold),
                                                        results.ctypes.data_as(C.POINTER(AlignResult))))
        return results

    def multi_align_frames(self, frames, mp, sp, ref_frame, cur_frame, guesses, ap, priors=None, depth_scale=0.001, step=1,
                           max_depth_cov=0.01, sensor_offset=None, img_threshold=50.0):
        """rig frames in, records out (nicp_multi_align_frames_sharded).  frames: n sequences of mp.num_cameras raw uint16
        images, as in Context.multi_raw_depth_to_cloud_batch; pair i = (ref_frame[i], cur_frame[i]) with guesses[i] (None:
        identity); priors: None or one list of Prior per pair.  Returns RESULT_DTYPE records."""
        imgs, rr, rc = _rig_frames(frames, mp.num_cameras)
        n = len(ref_frame)
        assert len(cur_frame) == n
        RA = (C.c_void_p * max(len(imgs), 1))(*[im.ctypes.data for im in imgs])
        rf = np.ascontiguousarray(ref_frame, np.int32)
        cf = np.ascontiguousarray(cur_frame, np.int32)
        so = colmajor(np.eye(4) if sensor_offset is None else sensor_offset)
        parr, offs = _priors(priors, n)
        results = np.zeros(n, RESULT_DTYPE)
        _check(self.L, self.L.nicp_multi_align_frames_sharded(
            self.handle, len(frames), RA, _iptr(rr), _iptr(rc), C.c_float(depth_scale), int(step), C.c_float(max_depth_cov),
            C.byref(mp), C.byref(sp), _fptr(so), n, _iptr(rf), _iptr(cf), _guesses(guesses, n), parr, offs, C.byref(ap),
            C.c_float(img_threshold), results.ctypes.data_as(C.POINTER(AlignResult))))
        return results

    def close(self):
        if self.handle:
            self.L.nicp_shard_pool_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _ids(ids):
    return np.ascontiguousarray(ids, np.int64)


def _llptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_longlong))


class FrameStore:
    """nicp_frame_store: the raw frames of one pinhole camera or one rig on a shard pool, under caller-chosen int64 ids.
    Each worker keeps the clouds of the frames it aligned across calls and prepares a frame only when it does not hold it.

    camera is a Projector (pinhole; raw_shape = (rows, cols) of every raw frame) or a MultiProjector (rig; raw_shape = one
    (rows, cols) per camera, as the sensor delivers it).  The other arguments are those of ShardPool.align_frames /
    multi_align_frames and are fixed for the store's lifetime."""

    def __init__(self, pool, camera, sp, raw_shape, depth_scale=0.001, step=1, max_depth_cov=0.01, sensor_offset=None):
        self.pool = pool  # the store's clouds live on the pool's workers
        self.L = pool.L
        self.rig = isinstance(camera, MultiProjector)
        self.num_cameras = camera.num_cameras if self.rig else 1
        self.handle = C.c_void_p()
        so = None if sensor_offset is None else _fptr(colmajor(sensor_offset))
        # the C call copies raw_rows x raw_cols pixels of every camera from whatever pointer it is given, so add() checks
        # each image against these shapes
        self.raw_shapes = [tuple(int(x) for x in s) for s in (raw_shape if self.rig else [raw_shape])]
        if self.rig:
            shapes = np.array(raw_shape, np.int32).reshape(self.num_cameras, 2)
            rr, rc = np.ascontiguousarray(shapes[:, 0]), np.ascontiguousarray(shapes[:, 1])
            _check(self.L, self.L.nicp_multi_frame_store_create(
                pool.handle, _iptr(rr), _iptr(rc), C.c_float(depth_scale), int(step), C.c_float(max_depth_cov),
                C.byref(camera), C.byref(sp), so, C.byref(self.handle)))
        else:
            rows, cols = raw_shape
            _check(self.L, self.L.nicp_frame_store_create(pool.handle, int(rows), int(cols), C.c_float(depth_scale), int(step),
                                                          C.c_float(max_depth_cov), C.byref(camera), C.byref(sp), so,
                                                          C.byref(self.handle)))

    def add(self, ids, frames):
        """frames[k] gets id ids[k]: a uint16 image (pinhole) or a sequence of one uint16 image per camera (rig), each of
        exactly the raw shape the store was created with for its camera; any other shape raises ValueError and adds
        nothing"""
        ids = _ids(ids)
        n = len(ids)
        if len(frames) != n:
            raise ValueError("%d ids for %d frames" % (n, len(frames)))
        nc = self.num_cameras
        imgs = []
        for k, fr in enumerate(frames):
            cams = fr if self.rig else [fr]
            if len(cams) != nc:
                raise ValueError("frame %d has %d images for %d cameras" % (k, len(cams), nc))
            for i, im in enumerate(cams):
                im = np.ascontiguousarray(im, np.uint16)
                if im.shape != self.raw_shapes[i]:
                    raise ValueError("frame %d, camera %d: raw image of shape %s, the store takes %s"
                                     % (k, i, im.shape, self.raw_shapes[i]))
                imgs.append(im)
        RA = (C.c_void_p * max(len(imgs), 1))(*[im.ctypes.data for im in imgs])
        _check(self.L, self.L.nicp_frame_store_add(self.handle, n, _llptr(ids), RA))

    def remove(self, ids):
        ids = _ids(ids)
        _check(self.L, self.L.nicp_frame_store_remove(self.handle, len(ids), _llptr(ids)))

    def size(self):
        return int(self.L.nicp_frame_store_size(self.handle))

    def align(self, ref_ids, cur_ids, guesses, ap, priors=None, img_threshold=50.0):
        """pair i = (ref_ids[i], cur_ids[i]) with guesses[i] (None: identity); priors: None or one list of Prior per pair.
        Returns RESULT_DTYPE records."""
        rf, cf = _ids(ref_ids), _ids(cur_ids)
        n = len(rf)
        assert len(cf) == n
        parr, offs = _priors(priors, n)
        results = np.zeros(n, RESULT_DTYPE)
        _check(self.L, self.L.nicp_frame_store_align(self.handle, n, _llptr(rf), _llptr(cf), _guesses(guesses, n), parr, offs,
                                                     C.byref(ap), C.c_float(img_threshold),
                                                     results.ctypes.data_as(C.POINTER(AlignResult))))
        return results

    def counters(self):
        """(frames built, frames found resident) since creation, summed over the workers and the windows of every call"""
        b, r = C.c_longlong(0), C.c_longlong(0)
        _check(self.L, self.L.nicp_frame_store_counters(self.handle, C.byref(b), C.byref(r)))
        return b.value, r.value

    def close(self):
        if self.handle:
            self.L.nicp_frame_store_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Tracker:
    """nicp_tracker: S independent depth sequences tracked as pwn::SequentialTracker::processFrame tracks one, with their
    keyframes resident on the workers of a shard pool (sequence s on worker s * G // S).  One step takes one frame of each
    listed sequence: one batched prep and one batched alignment per worker.

    camera is a Projector (pinhole, describing the image after scaling; raw_shape = (rows, cols) of every raw frame) or a
    MultiProjector (rig; raw_shape = one (rows, cols) per camera, as the sensor delivers it), as for FrameStore.  sp and ap
    are the statistics and alignment parameters, img_threshold the frame inlier depth threshold of every record, and
    new_frame_inliers_fraction the keyframe threshold of SequentialTracker::setNewFrameInliersFraction.  Every argument is
    fixed for the tracker's lifetime."""

    def __init__(self, pool, camera, sp, ap, raw_shape, n_sequences, depth_scale=0.001, step=1, max_depth_cov=0.01,
                 sensor_offset=None, img_threshold=50.0, new_frame_inliers_fraction=0.4):
        self.pool = pool  # the tracker's clouds live on the pool's workers
        self.L = pool.L
        self.rig = isinstance(camera, MultiProjector)
        self.num_cameras = camera.num_cameras if self.rig else 1
        self.handle = C.c_void_p()
        so = None if sensor_offset is None else _fptr(colmajor(sensor_offset))
        # the C call reads raw_rows x raw_cols pixels of every camera from whatever pointer it is given, so step() checks
        # each image against these shapes
        self.raw_shapes = [tuple(int(x) for x in s) for s in (raw_shape if self.rig else [raw_shape])]
        common = (C.c_float(depth_scale), int(step), C.c_float(max_depth_cov))
        tail = (C.byref(sp), so, C.byref(ap), C.c_float(img_threshold), C.c_float(new_frame_inliers_fraction),
                C.byref(self.handle))
        if self.rig:
            shapes = np.array(raw_shape, np.int32).reshape(self.num_cameras, 2)
            rr, rc = np.ascontiguousarray(shapes[:, 0]), np.ascontiguousarray(shapes[:, 1])
            _check(self.L, self.L.nicp_multi_tracker_create(pool.handle, int(n_sequences), _iptr(rr), _iptr(rc), *common,
                                                            C.byref(camera), *tail))
        else:
            rows, cols = raw_shape
            _check(self.L, self.L.nicp_tracker_create(pool.handle, int(n_sequences), int(rows), int(cols), *common,
                                                      C.byref(camera), *tail))

    def step(self, sequences, frames, odometry=None):
        """frames[k] is the next frame of sequence sequences[k]: a uint16 image (pinhole) or one uint16 image per camera
        (rig), each of exactly the raw shape given at creation (any other shape raises ValueError and the library is not
        called).  odometry: None (identity) or one (4, 4) initial guess per frame.  Returns TRACK_DTYPE results."""
        seqs = np.ascontiguousarray(sequences, np.int32)
        n = len(seqs)
        if len(frames) != n:
            raise ValueError("%d sequences for %d frames" % (n, len(frames)))
        nc = self.num_cameras
        imgs = []
        for k, fr in enumerate(frames):
            cams = fr if self.rig else [fr]
            if len(cams) != nc:
                raise ValueError("frame %d has %d images for %d cameras" % (k, len(cams), nc))
            for i, im in enumerate(cams):
                im = np.ascontiguousarray(im, np.uint16)
                if im.shape != self.raw_shapes[i]:
                    raise ValueError("frame %d, camera %d: raw image of shape %s, the tracker takes %s"
                                     % (k, i, im.shape, self.raw_shapes[i]))
                imgs.append(im)
        if odometry is not None and len(odometry) != n:
            raise ValueError("%d odometry guesses for %d frames" % (len(odometry), n))
        RA = (C.c_void_p * max(len(imgs), 1))(*[im.ctypes.data for im in imgs])
        results = np.zeros(n, TRACK_DTYPE)
        _check(self.L, self.L.nicp_tracker_step(self.handle, n, _iptr(seqs), RA, _guesses(odometry, n),
                                                results.ctypes.data_as(C.POINTER(TrackResult))))
        return results

    def reset(self, sequences):
        """the listed sequences start over: no keyframe, global pose identity, counters 0"""
        seqs = np.ascontiguousarray(sequences, np.int32)
        _check(self.L, self.L.nicp_tracker_reset(self.handle, len(seqs), _iptr(seqs)))

    def size(self):
        return int(self.L.nicp_tracker_size(self.handle))

    def close(self):
        if self.handle:
            self.L.nicp_tracker_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

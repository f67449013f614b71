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
    "nicp_multi_image_size", "nicp_multi_depth_to_cloud", "nicp_multi_project", "nicp_multi_align",
    "nicp_multi_raw_depth_to_cloud_batch", "nicp_multi_align_batch",
    "nicp_cloud_compute_gaussians", "nicp_cloud_has_gaussians", "nicp_cloud_download_gaussians",
    "nicp_cloud_upload_gaussians", "nicp_merge", "nicp_voxelize",
    "nicp_shard_pool_create", "nicp_shard_pool_destroy", "nicp_shard_pool_size", "nicp_align_frames_sharded",
    "nicp_multi_align_frames_sharded",
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
        n, nc = len(frames), mp.num_cameras
        imgs = []
        for fr in frames:
            assert len(fr) == nc, "a frame needs one raw image per camera"
            imgs += [r if (isinstance(r, np.ndarray) and r.dtype == np.uint16 and r.flags.c_contiguous)
                     else np.ascontiguousarray(r, np.uint16) for r in fr]
        shapes = [imgs[i].shape for i in range(nc)] if n else []
        for k, im in enumerate(imgs):
            assert im.shape == shapes[k % nc], "camera %d has a different raw size in frame %d" % (k % nc, k // nc)
        rr = np.array([s[0] for s in shapes] or [0], np.int32)
        rc = np.array([s[1] for s in shapes] or [0], np.int32)
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
        if guesses is None:
            g = np.tile(colmajor(eye), (n, 1))
        else:
            g = np.asarray(guesses, np.float32).transpose(0, 2, 1).reshape(n, 16)
        g = np.ascontiguousarray(g, np.float32)
        RA = (C.c_void_p * max(n, 1))(*[r.handle for r in refs])
        CA = (C.c_void_p * max(n, 1))(*[c.handle for c in curs])
        if results is None:
            results = np.zeros(n, RESULT_DTYPE)
        parr, offs = None, None
        if priors is not None:
            assert len(priors) == n
            flat = [p for ps in priors for p in ps]
            offs = np.zeros(n + 1, np.int32)
            offs[1:] = np.cumsum([len(ps) for ps in priors])
            parr = (Prior * max(len(flat), 1))(*flat)
        _check(self.L, self.L.nicp_multi_align_batch(self.handle, n, RA, CA, C.byref(mp), C.byref(ap), _fptr(ro), _fptr(co),
                                                     _fptr(g), parr, None if offs is None else _iptr(offs),
                                                     C.c_float(img_threshold), results.ctypes.data_as(C.POINTER(AlignResult))))
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

    def align_batch(self, refs, curs, proj, ap, guesses=None, ref_offset=None, cur_offset=None, img_threshold=50.0,
                    results=None, priors=None):
        """refs/curs: sequences of Cloud.  guesses: (n,4,4) row/col matrices or None.  priors: None or a sequence of
        n lists of Prior (nicp_align_batch_priors).  Returns a numpy structured array (RESULT_DTYPE) of n 256-byte records."""
        n = len(refs)
        assert len(curs) == n
        eye = np.eye(4, dtype=np.float32)
        ro = colmajor(eye if ref_offset is None else ref_offset)
        co = colmajor(eye if cur_offset is None else cur_offset)
        if guesses is None:
            g = np.tile(colmajor(eye), (n, 1))
        else:
            g = np.ascontiguousarray(np.asarray(guesses, np.float32).transpose(0, 2, 1)).reshape(n, 16)
        g = np.ascontiguousarray(g, np.float32)
        RA = (C.c_void_p * n)(*[r.handle for r in refs])
        CA = (C.c_void_p * n)(*[c.handle for c in curs])
        if results is None:
            results = np.zeros(n, RESULT_DTYPE)
        if priors is not None:
            assert len(priors) == n
            flat = [p for ps in priors for p in ps]
            offs = np.zeros(n + 1, np.int32)
            offs[1:] = np.cumsum([len(ps) for ps in priors])
            parr = (Prior * max(len(flat), 1))(*flat)
            _check(self.L, self.L.nicp_align_batch_priors(self.handle, n, RA, CA, C.byref(proj), C.byref(ap), _fptr(ro),
                                                          _fptr(co), _fptr(g), parr, _iptr(offs), C.c_float(img_threshold),
                                                          results.ctypes.data_as(C.POINTER(AlignResult))))
            return results
        _check(self.L, self.L.nicp_align_batch(self.handle, n, RA, CA, C.byref(proj), C.byref(ap), _fptr(ro), _fptr(co),
                                               _fptr(g), C.c_float(img_threshold),
                                               results.ctypes.data_as(C.POINTER(AlignResult))))
        return results


def update_matrices(K, T, verify=False):
    """PinholePointProjector::_updateMatrices through the library (host-side, no GPU needed)."""
    L = load(verify)
    k, t = colmajor(K), colmajor(T)
    KRt, iKRt = np.zeros(16, np.float32), np.zeros(16, np.float32)
    L.nicp_update_matrices(_fptr(k), _fptr(t), _fptr(KRt), _fptr(iKRt))
    return from_colmajor(KRt, 4), from_colmajor(iKRt, 4)


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
        g = np.ascontiguousarray(np.asarray(guesses, np.float32).transpose(0, 2, 1)).reshape(n, 16)
        so = colmajor(np.eye(4) if sensor_offset is None else sensor_offset)
        results = np.zeros(n, RESULT_DTYPE)
        _check(self.L, self.L.nicp_align_frames_sharded(self.handle, len(frames), RA, rows, cols, C.c_float(depth_scale), int(step),
                                                        C.c_float(max_depth_cov), C.byref(proj), C.byref(sp), _fptr(so), n,
                                                        _iptr(rf), _iptr(cf), _fptr(g), C.byref(ap), C.c_float(img_threshold),
                                                        results.ctypes.data_as(C.POINTER(AlignResult))))
        return results

    def multi_align_frames(self, frames, mp, sp, ref_frame, cur_frame, guesses, ap, priors=None, depth_scale=0.001, step=1,
                           max_depth_cov=0.01, sensor_offset=None, img_threshold=50.0):
        """rig frames in, records out (nicp_multi_align_frames_sharded).  frames: n sequences of mp.num_cameras raw uint16
        images, as in Context.multi_raw_depth_to_cloud_batch; pair i = (ref_frame[i], cur_frame[i]) with guesses[i] (None:
        identity); priors: None or one list of Prior per pair.  Returns RESULT_DTYPE records."""
        nc = mp.num_cameras
        imgs = []
        for fr in frames:
            assert len(fr) == nc, "a frame needs one raw image per camera"
            imgs += [r if (isinstance(r, np.ndarray) and r.dtype == np.uint16 and r.flags.c_contiguous)
                     else np.ascontiguousarray(r, np.uint16) for r in fr]
        shapes = [imgs[i].shape for i in range(nc)] if frames else [(0, 0)] * nc
        for k, im in enumerate(imgs):
            assert im.shape == shapes[k % nc], "camera %d has a different raw size in frame %d" % (k % nc, k // nc)
        rr = np.array([s[0] for s in shapes], np.int32)
        rc = np.array([s[1] for s in shapes], np.int32)
        n = len(ref_frame)
        assert len(cur_frame) == n
        RA = (C.c_void_p * max(len(imgs), 1))(*[im.ctypes.data for im in imgs])
        rf = np.ascontiguousarray(ref_frame, np.int32)
        cf = np.ascontiguousarray(cur_frame, np.int32)
        g = None
        if guesses is not None:
            g = np.ascontiguousarray(np.asarray(guesses, np.float32).transpose(0, 2, 1)).reshape(n, 16)
        so = colmajor(np.eye(4) if sensor_offset is None else sensor_offset)
        parr, offs = None, None
        if priors is not None:
            assert len(priors) == n
            flat = [p for ps in priors for p in ps]
            offs = np.zeros(n + 1, np.int32)
            offs[1:] = np.cumsum([len(ps) for ps in priors])
            parr = (Prior * max(len(flat), 1))(*flat)
        results = np.zeros(n, RESULT_DTYPE)
        _check(self.L, self.L.nicp_multi_align_frames_sharded(
            self.handle, len(frames), RA, _iptr(rr), _iptr(rc), C.c_float(depth_scale), int(step), C.c_float(max_depth_cov),
            C.byref(mp), C.byref(sp), _fptr(so), n, _iptr(rf), _iptr(cf), None if g is None else _fptr(g), parr,
            None if offs is None else _iptr(offs), C.byref(ap), C.c_float(img_threshold),
            results.ctypes.data_as(C.POINTER(AlignResult))))
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

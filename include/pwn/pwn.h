// pwn/pwn.h -- the pwn:: class surface of g2o_frontend's NICP core, implemented over the C-ABI of
// the B200-native library (include/nicp_b200.h).  Same class names, setter/getter names and
// constructor defaults as the reference so that trackers and mappers (PwnMatcherBase::makeCloud /
// matchClouds, pwn_tracker2/pwn_matcher_base.cpp:46-196; pwn_simple_aligner.cpp:28-188) compile
// against it unchanged apart from the Eigen/OpenCV stand-in types of pwn/compat.h.
//
// Reference headers mirrored (g2o_frontend/pwn_core/): pointprojector.h, pinholepointprojector.h,
// statscalculator.h, statscalculatorintegralimage.h, informationmatrixcalculator.h, cloud.h,
// depthimageconverter.h, depthimageconverterintegralimage.h, correspondencefinder.h, linearizer.h,
// aligner.h, pwn_static.h.
//
// Differences that follow from the data living on the GPU:
//   * pwn::Cloud owns a device handle; its host vectors (points(), normals(), stats(), ...) are
//     mirrors materialised on first access.  Non-const access marks the host copy as the truth and
//     the cloud is re-uploaded before its next use on the device.
//   * All calls are made on the calling thread's context (pwn::Context::current(); one GPU, one
//     stream) -- like pwn_core, the classes are not thread-safe.
//   * Errors: the reference only asserts; here a failing CUDA call throws std::runtime_error with
//     nicp_last_error().  There is no CPU fallback.
#pragma once
#include <cfloat>
#include <cmath>
#include <fstream>
#include <iostream>
#include <sstream>
#include <stdexcept>
#include <string>
#include <sys/time.h>
#include <vector>

#include "../nicp_b200.h"
#include "compat.h"

namespace pwn {

inline void nicpCheck(int rc, const char *what) {
  if (rc != NICP_OK) throw std::runtime_error(std::string(what) + ": " + nicp_last_error());
}

// one nicp_context per host thread
class Context {
 public:
  static Context &current(int device = 0) {
    static thread_local Context ctx(device);
    return ctx;
  }
  nicp_context *handle() { return _ctx; }
  ~Context() { nicp_destroy(_ctx); }

 private:
  explicit Context(int device) : _ctx(0) { nicpCheck(nicp_create(device, &_ctx), "nicp_create"); }
  Context(const Context &);
  nicp_context *_ctx;
};

// ---- pwn_static.h ------------------------------------------------------------------------------
inline void DepthImage_convert_16UC1_to_32FC1(DepthImage &dest, const RawDepthImage &src, float scale = 0.001f) {
  dest.create(src.rows, src.cols);
  nicpCheck(nicp_depth_prepare(Context::current().handle(), src.data(), src.rows, src.cols, scale, 1, 0.01f, dest.data()),
            "DepthImage_convert_16UC1_to_32FC1");
}
// raw -> metres -> box down-sample in one device pass (pwn_static.cpp:5-36 after :54-68)
inline void DepthImage_convertAndScale(DepthImage &dest, const RawDepthImage &src, int step, float scale = 0.001f,
                                       float maxDepthCov = 0.01f) {
  dest.create(src.rows / step, src.cols / step);
  nicpCheck(nicp_depth_prepare(Context::current().handle(), src.data(), src.rows, src.cols, scale, step, maxDepthCov,
                               dest.data()),
            "DepthImage_scale");
}

// ---- bm_se3.h ------------------------------------------------------------------------------------
inline Isometry3f v2t(const Vector6f &v) {
  Isometry3f T;
  nicp_v2t(v.data(), T.data());
  return T;
}
inline Vector6f t2v(const Isometry3f &T) {
  Vector6f v;
  nicp_t2v(T.data(), v.data());
  return v;
}

// ---- cloud.h -------------------------------------------------------------------------------------
// basemath/gaussian.h Gaussian<float, 3>: both forms with the reference's lazy conversion (host view)
struct Gaussian3f {
  Vector3f _mean, _informationVector;
  Matrix3f _covarianceMatrix, _informationMatrix;
  bool _momentsUpdated, _infoUpdated;
  Gaussian3f() : _momentsUpdated(false), _infoUpdated(false) {}
  const Vector3f &mean() const { return _mean; }
  const Matrix3f &covarianceMatrix() const { return _covarianceMatrix; }
  const Vector3f &informationVector() const { return _informationVector; }
  const Matrix3f &informationMatrix() const { return _informationMatrix; }
};
typedef std::vector<Gaussian3f> Gaussian3fVector;

class Cloud {
 public:
  Cloud() : _dev(0), _capacity(0), _deviceValid(false), _hostValid(true), _hasStats(false) {}
  virtual ~Cloud() { release(); }
  // The reference copies clouds by value (Cloud::add(Cloud cloud, ...), cloud.cpp:145; `pwn::Cloud cloud = *cloud_;`,
  // pwn_tracker2/manifold_voronoi_extractor.cpp:82): a copy owns its own device cloud (device-to-device append with the
  // identity; Stats and gaussians are carried through the host mirror / are not carried, like Cloud::add).
  Cloud(const Cloud &o) : _dev(0), _capacity(0), _deviceValid(false), _hostValid(true), _hasStats(false) { copyFrom(o); }
  Cloud &operator=(const Cloud &o) {
    if (this != &o) copyFrom(o);
    return *this;
  }

  const PointVector &points() const { ensureHost(); return _points; }
  PointVector &points() { ensureHost(); _deviceValid = false; return _points; }
  const NormalVector &normals() const { ensureHost(); return _normals; }
  NormalVector &normals() { ensureHost(); _deviceValid = false; return _normals; }
  const StatsVector &stats() const { ensureHost(); return _stats; }
  StatsVector &stats() { ensureHost(); _deviceValid = false; return _stats; }
  const InformationMatrixVector &pointInformationMatrix() const { ensureHost(); return _pointInformationMatrix; }
  InformationMatrixVector &pointInformationMatrix() { ensureHost(); _deviceValid = false; return _pointInformationMatrix; }
  const InformationMatrixVector &normalInformationMatrix() const { ensureHost(); return _normalInformationMatrix; }
  InformationMatrixVector &normalInformationMatrix() { ensureHost(); _deviceValid = false; return _normalInformationMatrix; }
  // cloud.h:99-105: host-only side channel of the traversability analysis (never read by the NICP path)
  const std::vector<int> &traversabilityVector() const { return _traversabilityVector; }
  std::vector<int> &traversabilityVector() { return _traversabilityVector; }

  size_t size() const {
    if (_deviceValid) return (size_t)nicp_cloud_size(_dev);
    return _points.size();
  }

  void clear() {
    _points.clear(); _normals.clear(); _stats.clear();
    _pointInformationMatrix.clear(); _normalInformationMatrix.clear();
    _traversabilityVector.clear();
    _hostValid = true;
    _deviceValid = false;
  }

  // Cloud::add (cloud.cpp:145-171): append a copy of `cloud` transformed by T.  Stats are not carried over on
  // the device (they are only materialised on request); everything the aligner reads is.
  void add(const Cloud &cloud, const Isometry3f &T = Isometry3f::Identity()) {
    nicp_context *ctx = Context::current().handle();
    const int n0 = (int)size(), n1 = (int)cloud.size();
    nicp_cloud *src = cloud.device();
    nicp_cloud *old = n0 > 0 ? device() : 0;
    if (old && _capacity >= n0 + n1) {  // room left: append in place
      nicpCheck(nicp_cloud_append(ctx, old, src, T.data()), "Cloud::add");
    } else {  // grow geometrically so that a local map is not reallocated for every frame
      const int cap = n0 + n1 > 0 ? (old ? 2 * (n0 + n1) : n0 + n1) : 1;
      nicp_cloud *merged = 0;
      nicpCheck(nicp_cloud_create(ctx, cap, &merged), "nicp_cloud_create");
      Isometry3f I;
      if (old) nicpCheck(nicp_cloud_append(ctx, merged, old, I.data()), "Cloud::add");
      nicpCheck(nicp_cloud_append(ctx, merged, src, T.data()), "Cloud::add");
      release();
      _dev = merged;
      _capacity = cap;
    }
    _deviceValid = true;
    _hostValid = false;
    _hasStats = false;
  }

  // Cloud::save / Cloud::load (cloud.cpp:25-133): "PWNCLOUD n binary" + pose 6-vector + one record per point.
  // ASCII records ("POINTWITHSTATS x y z nx ny nz <16 stats>") are written exactly like the reference.  The
  // reference's binary mode dumps its C++ objects raw (os.write(&point, sizeof(Point)) ...), i.e. including each
  // object's vptr and padding: on LP64 / Itanium ABI that is 32 B per Point (8 vptr, 8 pad, 4 floats), 32 B per
  // Normal, 112 B per Stats (8 vptr, 8 pad, 16 floats column-major, int n, 3 eigenvalues, bool, float curvature,
  // pad).  We write zeros into the vptr/padding bytes and ignore them on load.
  bool save(std::ostream &os, Isometry3f T = Isometry3f::Identity(), int step = 1, bool binary = true) const {
    ensureHost();
    os << "PWNCLOUD " << _points.size() / step << " " << binary << std::endl;
    Vector6f transform = t2v(T);
    os << transform[0] << " " << transform[1] << " " << transform[2] << " " << transform[3] << " " << transform[4] << " "
       << transform[5] << " " << std::endl;
    for (size_t i = 0; i < _points.size(); i += step) {
      const Point &point = _points[i];
      const Normal &normal = _normals[i];
      const Stats &stats = _stats[i];
      if (!binary) {
        os << "POINTWITHSTATS ";
        for (int k = 0; k < 3; k++) os << point[k] << " ";
        for (int k = 0; k < 3; k++) os << normal[k] << " ";
        for (int r = 0; r < 4; r++)
          for (int c = 0; c < 4; c++) os << stats(r, c) << " ";
        os << std::endl;
      } else {
        unsigned char rec[32 + 32 + 112];
        std::memset(rec, 0, sizeof rec);
        std::memcpy(rec + 16, point.m, 16);
        std::memcpy(rec + 32 + 16, normal.m, 16);
        std::memcpy(rec + 64 + 16, stats.m, 64);
        int n = stats._n;
        float curv = stats.curvature();
        std::memcpy(rec + 64 + 80, &n, 4);
        std::memcpy(rec + 64 + 84, stats._eigenValues.m, 12);
        rec[64 + 96] = 1;  // _curvatureComputed
        std::memcpy(rec + 64 + 100, &curv, 4);
        os.write((const char *)rec, sizeof rec);
      }
    }
    return os.good();
  }
  bool save(const char *filename, Isometry3f T = Isometry3f::Identity(), int step = 1, bool binary = true) const {
    std::ofstream os(filename);
    if (!os) return false;
    return save(os, T, step, binary);
  }
  bool load(Isometry3f &T, std::istream &is) {
    clear();
    char buf[1024];
    is.getline(buf, 1024);
    std::istringstream ls(buf);
    std::string tag;
    size_t numPoints = 0;
    bool binary = false;
    ls >> tag;
    if (tag != "PWNCLOUD") return false;
    ls >> numPoints >> binary;
    _points.resize(numPoints);
    _normals.resize(numPoints);
    _stats.assign(numPoints, Stats());
    _pointInformationMatrix.assign(numPoints, InformationMatrix());
    _normalInformationMatrix.assign(numPoints, InformationMatrix());
    is.getline(buf, 1024);
    std::istringstream lst(buf);
    Vector6f transform;
    lst >> transform[0] >> transform[1] >> transform[2] >> transform[3] >> transform[4] >> transform[5];
    T = v2t(transform);
    size_t k = 0;
    while (k < _points.size() && is.good()) {
      Point &point = _points[k];
      Normal &normal = _normals[k];
      Stats &stats = _stats[k];
      if (!binary) {
        is.getline(buf, 1024);
        std::istringstream l2(buf);
        std::string s;
        l2 >> s;
        if (s != "POINTWITHSTATS") continue;
        for (int i = 0; i < 3 && l2; i++) l2 >> point[i];
        for (int i = 0; i < 3 && l2; i++) l2 >> normal[i];
        for (int r = 0; r < 4 && l2; r++)
          for (int c = 0; c < 4 && l2; c++) l2 >> stats(r, c);
      } else {
        unsigned char rec[32 + 32 + 112];
        is.read((char *)rec, sizeof rec);
        std::memcpy(point.m, rec + 16, 16);
        std::memcpy(normal.m, rec + 32 + 16, 16);
        std::memcpy(stats.m, rec + 64 + 16, 64);
        std::memcpy(&stats._n, rec + 64 + 80, 4);
        std::memcpy(stats._eigenValues.m, rec + 64 + 84, 12);
        if (rec[64 + 96]) {  // _curvatureComputed, _curvature (stats.h:117-118)
          float curv;
          std::memcpy(&curv, rec + 64 + 100, 4);
          stats.setCurvature(curv);
        }
      }
      point[3] = 1.0f;
      normal[3] = 0.0f;
      k++;
    }
    _hostValid = true;
    _deviceValid = false;
    return is.good() || is.eof();
  }
  bool load(Isometry3f &T, const char *filename) {
    std::ifstream is(filename);
    if (!is) return false;
    return load(T, is);
  }

  // Cloud::transformInPlace (cloud.cpp:173-186)
  void transformInPlace(const Isometry3f &T) {
    nicp_cloud *d = device();
    nicpCheck(nicp_cloud_transform(Context::current().handle(), d, T.data()), "Cloud::transformInPlace");
    _hostValid = false;
  }

  // Gaussian3f per point (basemath/gaussian.h), read-only host view: mean, covariance, information vector / matrix
  // and which of the two forms is valid.  Present when the converter ran with setKeepGaussians(true).
  bool hasGaussians() const { return _deviceValid && _dev && nicp_cloud_has_gaussians(_dev); }
  Gaussian3fVector gaussians() const {
    Gaussian3fVector out;
    if (!hasGaussians()) return out;
    const int n = nicp_cloud_size(_dev);
    std::vector<float> g((size_t)NICP_GAUSS_FLOATS * n);
    std::vector<int> f(n);
    nicpCheck(nicp_cloud_download_gaussians(Context::current().handle(), _dev, g.data(), f.data()), "Cloud::gaussians");
    out.resize(n);
    for (int i = 0; i < n; i++) {
      const float *q = &g[(size_t)NICP_GAUSS_FLOATS * i];
      for (int k = 0; k < 3; k++) { out[i]._mean(k) = q[k]; out[i]._informationVector(k) = q[12 + k]; }
      for (int k = 0; k < 9; k++) { out[i]._covarianceMatrix.m[k] = q[3 + k]; out[i]._informationMatrix.m[k] = q[15 + k]; }
      out[i]._momentsUpdated = (f[i] & NICP_GAUSS_MOMENTS) != 0;
      out[i]._infoUpdated = (f[i] & NICP_GAUSS_INFO) != 0;
    }
    return out;
  }
  // after a device-side operation changed the cloud (Merger, VoxelCalculator)
  void deviceChanged() { _hostValid = false; _deviceValid = true; }

  // device side (used by the converter / aligner)
  nicp_cloud *deviceForWrite(int capacity) {
    if (!_dev || _capacity < capacity) {
      release();
      nicpCheck(nicp_cloud_create(Context::current().handle(), capacity, &_dev), "nicp_cloud_create");
      _capacity = capacity;
    }
    _deviceValid = true;
    _hostValid = false;
    return _dev;
  }
  nicp_cloud *device() const {
    Cloud *self = const_cast<Cloud *>(this);
    if (!_deviceValid) self->upload();
    return _dev;
  }
  void setHasStats(bool v) { _hasStats = v; }

 protected:
  void release() {
    if (_dev) nicp_cloud_destroy(_dev);
    _dev = 0;
    _capacity = 0;
  }
  void copyFrom(const Cloud &o) {
    _traversabilityVector = o._traversabilityVector;
    if (o._hostValid) {  // the host vectors are the truth (or as good as the device): copy them, upload on demand
      _points = o._points; _normals = o._normals; _stats = o._stats;
      _pointInformationMatrix = o._pointInformationMatrix; _normalInformationMatrix = o._normalInformationMatrix;
      _hostValid = true;
      _deviceValid = false;
      _hasStats = false;
      return;
    }
    // device-resident source: a device-to-device copy into a cloud of our own
    nicp_context *ctx = Context::current().handle();
    const int n = (int)o.size();
    nicp_cloud *fresh = 0;
    nicpCheck(nicp_cloud_create(ctx, n > 0 ? n : 1, &fresh), "nicp_cloud_create");
    Isometry3f I;
    int rc = nicp_cloud_append(ctx, fresh, o._dev, I.data());
    if (rc != NICP_OK) { nicp_cloud_destroy(fresh); nicpCheck(rc, "Cloud copy"); }
    release();
    _dev = fresh;
    _capacity = n > 0 ? n : 1;
    _points.clear(); _normals.clear(); _stats.clear();
    _pointInformationMatrix.clear(); _normalInformationMatrix.clear();
    _deviceValid = true;
    _hostValid = false;
    _hasStats = false;
  }
  void upload() {
    const int n = (int)_points.size();
    if (!_dev || _capacity < n || _capacity == 0) {
      release();
      nicpCheck(nicp_cloud_create(Context::current().handle(), n > 0 ? n : 1, &_dev), "nicp_cloud_create");
      _capacity = n > 0 ? n : 1;
    }
    std::vector<float> p(4 * (size_t)n), nr(4 * (size_t)n), cv(n), op(6 * (size_t)n), on(6 * (size_t)n);
    for (int i = 0; i < n; i++) {
      for (int k = 0; k < 4; k++) p[4 * (size_t)i + k] = _points[i][k];
      if ((size_t)i < _normals.size())
        for (int k = 0; k < 4; k++) nr[4 * (size_t)i + k] = _normals[i][k];
      cv[i] = (size_t)i < _stats.size() ? _stats[i].curvature() : 0.0f;
      if ((size_t)i < _pointInformationMatrix.size()) sym6(_pointInformationMatrix[i], &op[6 * (size_t)i]);
      if ((size_t)i < _normalInformationMatrix.size()) sym6(_normalInformationMatrix[i], &on[6 * (size_t)i]);
    }
    static const float dummy[4] = {0, 0, 0, 1};
    nicpCheck(nicp_cloud_upload(Context::current().handle(), _dev, n, n ? p.data() : dummy, nr.data(), cv.data(), op.data(),
                                on.data()),
              "nicp_cloud_upload");
    _deviceValid = true;
    _hasStats = false;
  }
  static void sym6(const Matrix4f &m, float *o) {
    o[0] = m(0, 0); o[1] = m(0, 1); o[2] = m(0, 2); o[3] = m(1, 1); o[4] = m(1, 2); o[5] = m(2, 2);
  }
  static void unsym6(const float *o, InformationMatrix &m) {
    m.setZero();
    m(0, 0) = o[0]; m(0, 1) = m(1, 0) = o[1]; m(0, 2) = m(2, 0) = o[2];
    m(1, 1) = o[3]; m(1, 2) = m(2, 1) = o[4]; m(2, 2) = o[5];
  }
  void ensureHost() const {
    if (_hostValid) return;
    Cloud *self = const_cast<Cloud *>(this);
    nicp_context *ctx = Context::current().handle();
    const int n = nicp_cloud_size(_dev);
    std::vector<float> p(4 * (size_t)n), nr(4 * (size_t)n), cv(n), op(6 * (size_t)n), on(6 * (size_t)n);
    nicpCheck(nicp_cloud_download(ctx, _dev, p.data(), nr.data(), cv.data(), op.data(), on.data()), "nicp_cloud_download");
    self->_points.resize(n);
    self->_normals.resize(n);
    self->_stats.assign(n, Stats());
    self->_pointInformationMatrix.resize(n);
    self->_normalInformationMatrix.resize(n);
    std::vector<float> s16, ev;
    std::vector<int> cnt;
    if (_hasStats && n) {
      s16.resize(16 * (size_t)n); ev.resize(3 * (size_t)n); cnt.resize(n);
      nicpCheck(nicp_cloud_download_stats(ctx, _dev, s16.data(), ev.data(), cnt.data()), "nicp_cloud_download_stats");
    }
    for (int i = 0; i < n; i++) {
      for (int k = 0; k < 4; k++) { self->_points[i][k] = p[4 * (size_t)i + k]; self->_normals[i][k] = nr[4 * (size_t)i + k]; }
      unsym6(&op[6 * (size_t)i], self->_pointInformationMatrix[i]);
      unsym6(&on[6 * (size_t)i], self->_normalInformationMatrix[i]);
      if (!s16.empty()) {
        for (int k = 0; k < 16; k++) self->_stats[i].m[k] = s16[16 * (size_t)i + k];
        for (int k = 0; k < 3; k++) self->_stats[i]._eigenValues(k) = ev[3 * (size_t)i + k];
        self->_stats[i]._n = cnt[i];
      }
      // the curvature lives with the normals on the device and is always mirrored (stats.h:98-119 caches it in Stats)
      self->_stats[i].setCurvature(cv[i]);
    }
    self->_hostValid = true;
  }

  nicp_cloud *_dev;
  int _capacity;
  bool _deviceValid, _hostValid, _hasStats;
  PointVector _points;
  NormalVector _normals;
  StatsVector _stats;
  InformationMatrixVector _pointInformationMatrix, _normalInformationMatrix;
  std::vector<int> _traversabilityVector;
};

// ---- pointprojector.h / pinholepointprojector.h ---------------------------------------------------
class PointProjector {
 public:
  PointProjector() : _minDistance(0.01f), _maxDistance(6.0f), _imageRows(0), _imageCols(0) {}  // pointprojector.cpp:6-13
  virtual ~PointProjector() {}
  virtual const Isometry3f &transform() const { return _transform; }
  virtual void setTransform(const Isometry3f &transform_) { _transform = transform_; _transform.fixLastRow(); }
  float minDistance() const { return _minDistance; }
  void setMinDistance(const float minDistance_) { _minDistance = minDistance_; }
  float maxDistance() const { return _maxDistance; }
  void setMaxDistance(const float maxDistance_) { _maxDistance = maxDistance_; }
  int imageRows() const { return _imageRows; }
  int imageCols() const { return _imageCols; }
  void setImageSize(const int imageRows_, const int imageCols_) { _imageRows = imageRows_; _imageCols = imageCols_; }
  virtual void project(IntImage &indexImage, DepthImage &depthImage, const Cloud &cloud) const = 0;
  virtual void unProject(Cloud &cloud, IntImage &indexImage, const DepthImage &depthImage) const = 0;
  virtual void projectIntervals(IntImage &intervalImage, const DepthImage &depthImage, const float worldRadius) const = 0;
  // pointprojector.h:228-233: the base class answers 0
  virtual int projectInterval(const int, const int, const float, const float) const { return 0; }
  virtual void scale(float scalingFactor) = 0;

 protected:
  Isometry3f _transform;
  float _minDistance, _maxDistance;
  int _imageRows, _imageCols;
};

class PinholePointProjector : public PointProjector {
 public:
  PinholePointProjector() : PointProjector(), _baseline(0.075f), _alpha(0.1f) {  // pinholepointprojector.cpp:5-13
    _cameraMatrix.setIdentity();
    _cameraMatrix(0, 2) = 0.5f;
    _cameraMatrix(1, 2) = 0.5f;
    _updateMatrices();
  }
  virtual void setTransform(const Isometry3f &transform_) { PointProjector::setTransform(transform_); _updateMatrices(); }
  const Matrix3f &cameraMatrix() const { return _cameraMatrix; }
  void setCameraMatrix(const Matrix3f &cameraMatrix_) { _cameraMatrix = cameraMatrix_; _updateMatrices(); }
  float baseline() const { return _baseline; }
  void setBaseline(float baseline_) { _baseline = baseline_; }
  float alpha() const { return _alpha; }
  void setAlpha(float alpha_) { _alpha = alpha_; }
  const Matrix4f &KRt() const { return _KRt; }
  const Matrix4f &iKRt() const { return _iKRt; }
  // pinholepointprojector.h:61: K^-1 (closed form for the upper-triangular camera matrix [fx s cx; 0 fy cy; 0 0 1])
  Matrix3f inverseCameraMatrix() const {
    Matrix3f iK;
    const float fx = _cameraMatrix(0, 0), fy = _cameraMatrix(1, 1), sk = _cameraMatrix(0, 1), cx = _cameraMatrix(0, 2),
                cy = _cameraMatrix(1, 2), w = _cameraMatrix(2, 2);
    iK(0, 0) = 1.0f / fx;
    iK(0, 1) = -sk / (fx * fy);
    iK(0, 2) = (sk * cy - cx * fy) / (fx * fy * w);
    iK(1, 1) = 1.0f / fy;
    iK(1, 2) = -cy / (fy * w);
    iK(2, 2) = 1.0f / w;
    return iK;
  }

  // pinholepointprojector.cpp:33-66
  virtual void project(IntImage &indexImage, DepthImage &depthImage, const Cloud &cloud) const {
    indexImage.create(_imageRows, _imageCols);
    depthImage.create(_imageRows, _imageCols);
    nicpCheck(nicp_project(Context::current().handle(), cloud.device(), _KRt.data(), _imageRows, _imageCols, _minDistance,
                           _maxDistance, indexImage.data(), depthImage.data()),
              "PinholePointProjector::project");
  }
  // pinholepointprojector.cpp:68-91
  virtual void unProject(Cloud &cloud, IntImage &indexImage, const DepthImage &depthImage) const {
    indexImage.create(depthImage.rows, depthImage.cols);
    nicp_cloud *d = cloud.deviceForWrite(depthImage.rows * depthImage.cols);
    nicpCheck(nicp_unproject(Context::current().handle(), depthImage.data(), depthImage.rows, depthImage.cols, _iKRt.data(),
                             _minDistance, _maxDistance, d, indexImage.data()),
              "PinholePointProjector::unProject");
    cloud.setHasStats(false);
  }
  // pinholepointprojector.cpp:135-147
  virtual void projectIntervals(IntImage &intervalImage, const DepthImage &depthImage, const float worldRadius) const {
    intervalImage.create(depthImage.rows, depthImage.cols);
    nicp_projector p = abiProjector();
    p.rows = depthImage.rows;
    p.cols = depthImage.cols;
    nicpCheck(nicp_project_intervals(Context::current().handle(), depthImage.data(), &p, worldRadius, intervalImage.data()),
              "PinholePointProjector::projectIntervals");
  }
  // pinholepointprojector.cpp:149-154
  virtual void scale(float scalingFactor) {
    for (int c = 0; c < 3; c++) { _cameraMatrix(0, c) *= scalingFactor; _cameraMatrix(1, c) *= scalingFactor; }
    _imageRows = (int)(_imageRows * scalingFactor);
    _imageCols = (int)(_imageCols * scalingFactor);
    _updateMatrices();
  }
  // per-point forms (pinholepointprojector.h:224-251), host side
  bool project(int &x, int &y, float &d, const Point &p) const {
    float ip[3];
    for (int i = 0; i < 3; i++) ip[i] = ((_KRt(i, 0) * p[0] + _KRt(i, 1) * p[1]) + _KRt(i, 2) * p[2]) + _KRt(i, 3) * p[3];
    d = ip[2];
    if (d < _minDistance || d > _maxDistance) return false;
    float s = 1.0f / d;
    x = (int)roundf(ip[0] * s);
    y = (int)roundf(ip[1] * s);
    return true;
  }
  bool unProject(Point &p, const int x, const int y, const float d) const {
    if (d < _minDistance || d > _maxDistance) return false;
    float v[4] = {x * d, y * d, d, 1.0f};
    for (int i = 0; i < 3; i++) p[i] = ((_iKRt(i, 0) * v[0] + _iKRt(i, 1) * v[1]) + _iKRt(i, 2) * v[2]) + _iKRt(i, 3) * v[3];
    p[3] = 1.0f;
    return true;
  }
  // _projectInterval (pinholepointprojector.h:264-274): p = K (r, r, 0) / d, the larger component truncated
  virtual int projectInterval(const int, const int, const float d, const float worldRadius) const {
    if (d < _minDistance || d > _maxDistance) return -1;
    const float p0 = (_cameraMatrix(0, 0) * worldRadius + _cameraMatrix(0, 1) * worldRadius) + _cameraMatrix(0, 2) * 0.0f;
    const float p1 = (_cameraMatrix(1, 0) * worldRadius + _cameraMatrix(1, 1) * worldRadius) + _cameraMatrix(1, 2) * 0.0f;
    const float s = 1.0f / d;
    const float a = p0 * s, b = p1 * s;
    return a > b ? (int)a : (int)b;
  }
  nicp_projector abiProjector() const {
    nicp_projector p;
    for (int i = 0; i < 9; i++) p.K[i] = _cameraMatrix.m[i];
    p.rows = _imageRows;
    p.cols = _imageCols;
    p.min_distance = _minDistance;
    p.max_distance = _maxDistance;
    return p;
  }

 protected:
  void _updateMatrices() { nicp_update_matrices(_cameraMatrix.data(), _transform.data(), _KRt.data(), _iKRt.data()); }
  float _baseline, _alpha;
  Matrix3f _cameraMatrix;
  Matrix4f _KRt, _iKRt;
};

// ---- multipointprojector.h ----------------------------------------------------------------------------
// Composite image layout and unProject order: see nicp_multi_projector in nicp_b200.h.
class MultiPointProjector : public PointProjector {
 public:
  MultiPointProjector() : PointProjector() {}
  virtual ~MultiPointProjector() {}
  // multipointprojector.h:23-27: the child is remembered with transform() * sensorOffset_
  void addPointProjector(PinholePointProjector *pointProjector_, Isometry3f sensorOffset_, int width_, int height_) {
    ChildProjectorInfo c;
    c.pointProjector = pointProjector_;
    c.sensorOffset = transform() * sensorOffset_;
    c.width = width_;
    c.height = height_;
    pointProjector_->setImageSize(width_, height_);
    _pointProjectors.push_back(c);
  }
  // multipointprojector.h:20-27 (like the reference it leaves the remembered width / height of the slot alone)
  void setPointProjector(PinholePointProjector *pointProjector_, Isometry3f sensorOffset_, int width_, int height_, int position) {
    _pointProjectors.at(position).pointProjector = pointProjector_;
    _pointProjectors.at(position).sensorOffset = sensorOffset_;
    pointProjector_->setImageSize(width_, height_);
  }
  void clearProjectors() { _pointProjectors.clear(); }
  size_t numProjectors() const { return _pointProjectors.size(); }
  // baseline() / alpha() of every child: the per-camera sensor model of the rig's gaussians
  // (nicp_multi_cloud_compute_gaussians); every child must be a PinholePointProjector
  void childSensorModels(std::vector<float> &baseline, std::vector<float> &alpha) const {
    baseline.clear();
    alpha.clear();
    for (size_t i = 0; i < _pointProjectors.size(); i++) {
      const PinholePointProjector *pp = _pointProjectors[i].pointProjector;
      if (!pp) throw std::runtime_error("MultiPointProjector: the sensor model needs a PinholePointProjector per child");
      baseline.push_back(pp->baseline());
      alpha.push_back(pp->alpha());
    }
  }
  // multipointprojector.cpp:7-18
  void computeImageSize(int &rows, int &cols) const {
    nicp_multi_projector mp = abiMultiProjector();
    nicp_multi_image_size(&mp, &rows, &cols);
  }
  // multipointprojector.cpp:207-215
  virtual void setTransform(const Isometry3f &transform_) {
    PointProjector::setTransform(transform_);
    for (size_t i = 0; i < _pointProjectors.size(); i++)
      _pointProjectors[i].pointProjector->setTransform(transform_ * _pointProjectors[i].sensorOffset);
  }
  // what Aligner executes for this projector: pointprojector.cpp:17-40 over multipointprojector.cpp:157-205
  virtual void project(IntImage &indexImage, DepthImage &depthImage, const Cloud &cloud) const {
    nicp_multi_projector mp = abiMultiProjector();
    int rows, cols;
    nicp_multi_image_size(&mp, &rows, &cols);
    indexImage.create(rows, cols);
    depthImage.create(rows, cols);
    nicpCheck(nicp_multi_project(Context::current().handle(), cloud.device(), &mp, _transform.data(), indexImage.data(),
                                 depthImage.data()),
              "MultiPointProjector::project");
  }
  virtual void unProject(Cloud &, IntImage &, const DepthImage &) const {
    throw std::runtime_error("MultiPointProjector::unProject: use DepthImageConverterIntegralImage::compute");
  }
  virtual void projectIntervals(IntImage &, const DepthImage &, const float) const {
    throw std::runtime_error("MultiPointProjector::projectIntervals: use DepthImageConverterIntegralImage::compute");
  }
  // multipointprojector.cpp:226-234
  virtual void scale(float scalingFactor) {
    for (size_t i = 0; i < _pointProjectors.size(); i++) {
      _pointProjectors[i].pointProjector->scale(scalingFactor);
      _pointProjectors[i].width = _pointProjectors[i].pointProjector->imageRows();
      _pointProjectors[i].height = _pointProjectors[i].pointProjector->imageCols();
    }
    int r, c;
    computeImageSize(r, c);
    setImageSize(r, c);
  }
  nicp_multi_projector abiMultiProjector() const {
    nicp_multi_projector mp;
    std::memset(&mp, 0, sizeof mp);
    mp.num_cameras = (int)_pointProjectors.size();
    for (int i = 0; i < mp.num_cameras && i < NICP_MAX_CAMERAS; i++) {
      const ChildProjectorInfo &c = _pointProjectors[i];
      mp.camera[i] = c.pointProjector->abiProjector();
      mp.camera[i].rows = c.width;
      mp.camera[i].cols = c.height;
      for (int k = 0; k < 16; k++) mp.sensor_offset[i][k] = c.sensorOffset.data()[k];
    }
    return mp;
  }

 protected:
  struct ChildProjectorInfo {
    PinholePointProjector *pointProjector;
    Isometry3f sensorOffset;
    int width, height;
  };
  std::vector<ChildProjectorInfo> _pointProjectors;
};

// ---- statscalculator.h / statscalculatorintegralimage.h ---------------------------------------------
class StatsCalculator {
 public:
  virtual ~StatsCalculator() {}
  // statscalculator.h:36: the base class computes nothing
  virtual void compute(NormalVector &, StatsVector &, const PointVector &, const IntImage &) {}
};
class StatsCalculatorIntegralImage : public StatsCalculator {
 public:
  StatsCalculatorIntegralImage()  // statscalculatorintegralimage.cpp:6-12
      : _worldRadius(0.1f), _maxImageRadius(30), _minImageRadius(10), _minPoints(50), _curvatureThreshold(0.02f) {}
  void setWorldRadius(const float worldRadius_) { _worldRadius = worldRadius_; }
  void setMaxImageRadius(const int maxImageRadius_) { _maxImageRadius = maxImageRadius_; }
  void setMinImageRadius(const int minImageRadius_) { _minImageRadius = minImageRadius_; }
  void setMinPoints(const int minPoints_) { _minPoints = minPoints_; }
  void setCurvatureThreshold(float curvatureThreshold_) { _curvatureThreshold = curvatureThreshold_; }
  float worldRadius() const { return _worldRadius; }
  int maxImageRadius() const { return _maxImageRadius; }
  int minImageRadius() const { return _minImageRadius; }
  int minPoints() const { return _minPoints; }
  float curvatureThreshold() const { return _curvatureThreshold; }
  IntImage &intervalImage() { return _intervalImage; }

  // statscalculatorintegralimage.h:37 / .cpp:14-82: normals and Stats of `points` from the integral image over
  // (indexImage, points) and the interval image set through intervalImage() (nicp_stats_compute)
  virtual void compute(NormalVector &normals, StatsVector &statsVector, const PointVector &points, const IntImage &indexImage) {
    const int n = (int)points.size();
    if (_intervalImage.rows != indexImage.rows || _intervalImage.cols != indexImage.cols)
      throw std::runtime_error("StatsCalculatorIntegralImage::compute: the interval image does not match the index image");
    std::vector<float> p(4 * (size_t)n), nr(4 * (size_t)n), s16(16 * (size_t)n), ev(3 * (size_t)n), cv(n);
    std::vector<int> cnt(n);
    for (int i = 0; i < n; i++)
      for (int k = 0; k < 4; k++) p[4 * (size_t)i + k] = points[i][k];
    nicp_stats_params sp = abiParams();
    nicpCheck(nicp_stats_compute(Context::current().handle(), p.data(), n, indexImage.data(), _intervalImage.data(), indexImage.rows,
                                 indexImage.cols, &sp, nr.data(), s16.data(), ev.data(), cnt.data(), cv.data()),
              "StatsCalculatorIntegralImage::compute");
    normals.resize(n);
    statsVector.assign(n, Stats());
    for (int i = 0; i < n; i++) {
      for (int k = 0; k < 4; k++) normals[i][k] = nr[4 * (size_t)i + k];
      for (int k = 0; k < 16; k++) statsVector[i].m[k] = s16[16 * (size_t)i + k];
      for (int k = 0; k < 3; k++) statsVector[i]._eigenValues(k) = ev[3 * (size_t)i + k];
      statsVector[i]._n = cnt[i];
      statsVector[i].setCurvature(cv[i]);
    }
  }
  // the statistics half of nicp_stats_params (the information-matrix half keeps its defaults)
  nicp_stats_params abiParams() const {
    nicp_stats_params sp;
    sp.world_radius = _worldRadius;
    sp.min_image_radius = _minImageRadius;
    sp.max_image_radius = _maxImageRadius;
    sp.min_points = _minPoints;
    sp.curvature_threshold = _curvatureThreshold;
    sp.omega_curvature_threshold = 0.02f;
    const float fp[3] = {1000.0f, 1.0f, 1.0f}, fn[3] = {100.0f, 100.0f, 100.0f}, nn[3] = {1.0f, 1.0f, 1.0f};
    for (int i = 0; i < 3; i++) { sp.flat_omega_p[i] = fp[i]; sp.flat_omega_n[i] = fn[i]; sp.nonflat_omega_n[i] = nn[i]; }
    return sp;
  }

 protected:
  float _worldRadius;
  int _maxImageRadius, _minImageRadius, _minPoints;
  float _curvatureThreshold;
  IntImage _intervalImage;
};

// ---- informationmatrixcalculator.h ---------------------------------------------------------------------
class InformationMatrixCalculator {
 public:
  InformationMatrixCalculator() : _curvatureThreshold(0.0f) {
    _flatInformationMatrix.setDiagonal(1.0f, 1.0f, 1.0f);
    _nonFlatInformationMatrix.setDiagonal(1.0f, 1.0f, 1.0f);
  }
  virtual ~InformationMatrixCalculator() {}
  InformationMatrix flatInformationMatrix() const { return _flatInformationMatrix; }
  // only the diagonal is used (the reference's configs only ever set diagonals)
  void setFlatInformationMatrix(const InformationMatrix flatInformationMatrix_) { _flatInformationMatrix = flatInformationMatrix_; }
  InformationMatrix nonFlatInformationMatrix() const { return _nonFlatInformationMatrix; }
  void setNonFlatInformationMatrix(const InformationMatrix nonFlatInformationMatrix_) { _nonFlatInformationMatrix = nonFlatInformationMatrix_; }
  float curvatureThreshold() const { return _curvatureThreshold; }
  void setCurvatureThreshold(const float curvatureThreshold_) { _curvatureThreshold = curvatureThreshold_; }
  // informationmatrixcalculator.h:83: pure virtual in the reference
  virtual void compute(InformationMatrixVector &informationMatrix, const StatsVector &statsVector,
                       const NormalVector &imageNormals) = 0;

 protected:
  // nicp_information_compute with this calculator's matrices in the point (which = 0) or the normal (1) slot
  void computeOnDevice(int which, InformationMatrixVector &informationMatrix, const StatsVector &statsVector,
                       const NormalVector &imageNormals) const {
    const int n = (int)statsVector.size();
    if ((int)imageNormals.size() != n) throw std::runtime_error("InformationMatrixCalculator::compute: size mismatch");
    std::vector<float> nr(4 * (size_t)n), s16(16 * (size_t)n), ev(3 * (size_t)n), cv(n), out(6 * (size_t)n);
    for (int i = 0; i < n; i++) {
      for (int k = 0; k < 4; k++) nr[4 * (size_t)i + k] = imageNormals[i][k];
      for (int k = 0; k < 16; k++) s16[16 * (size_t)i + k] = statsVector[i].m[k];
      for (int k = 0; k < 3; k++) ev[3 * (size_t)i + k] = statsVector[i]._eigenValues(k);
      cv[i] = statsVector[i].curvature();
    }
    nicp_stats_params sp;
    std::memset(&sp, 0, sizeof sp);
    sp.omega_curvature_threshold = _curvatureThreshold;
    for (int i = 0; i < 3; i++) {
      sp.flat_omega_p[i] = sp.flat_omega_n[i] = _flatInformationMatrix(i, i);
      sp.nonflat_omega_n[i] = _nonFlatInformationMatrix(i, i);
    }
    nicpCheck(nicp_information_compute(Context::current().handle(), n, nr.data(), s16.data(), ev.data(), cv.data(), &sp,
                                       which == 0 ? out.data() : 0, which == 1 ? out.data() : 0),
              "InformationMatrixCalculator::compute");
    informationMatrix.resize(n);
    for (int i = 0; i < n; i++) {
      const float *o = &out[6 * (size_t)i];
      InformationMatrix &m = informationMatrix[i];
      m.setZero();
      m(0, 0) = o[0]; m(0, 1) = m(1, 0) = o[1]; m(0, 2) = m(2, 0) = o[2];
      m(1, 1) = o[3]; m(1, 2) = m(2, 1) = o[4]; m(2, 2) = o[5];
    }
  }
  InformationMatrix _flatInformationMatrix, _nonFlatInformationMatrix;
  float _curvatureThreshold;
};
class PointInformationMatrixCalculator : public InformationMatrixCalculator {
 public:
  PointInformationMatrixCalculator() {  // informationmatrixcalculator.h:105-110
    _flatInformationMatrix.setDiagonal(1000.0f, 1.0f, 1.0f);
    _nonFlatInformationMatrix.setDiagonal(1.0f, 1.0f, 1.0f);
    _curvatureThreshold = 0.02f;
  }
  // informationmatrixcalculator.h:123 / .cpp:9-36: flat -> U diag(flat) U^T, else U diag(1 / eigenvalues) U^T
  virtual void compute(InformationMatrixVector &informationMatrix, const StatsVector &statsVector, const NormalVector &imageNormals) {
    computeOnDevice(0, informationMatrix, statsVector, imageNormals);
  }
};
class NormalInformationMatrixCalculator : public InformationMatrixCalculator {
 public:
  NormalInformationMatrixCalculator() {  // informationmatrixcalculator.h:140-145
    _flatInformationMatrix.setDiagonal(100.0f, 100.0f, 100.0f);
    _nonFlatInformationMatrix.setDiagonal(1.0f, 1.0f, 1.0f);
    _curvatureThreshold = 0.02f;
  }
  // informationmatrixcalculator.h:158 / .cpp:38-58
  virtual void compute(InformationMatrixVector &informationMatrix, const StatsVector &statsVector, const NormalVector &imageNormals) {
    computeOnDevice(1, informationMatrix, statsVector, imageNormals);
  }
};

// ---- depthimageconverter.h / depthimageconverterintegralimage.h -------------------------------------
class DepthImageConverter {
 public:
  DepthImageConverter(PointProjector *projector_ = 0, StatsCalculator *statsCalculator_ = 0,
                      PointInformationMatrixCalculator *pointInformationMatrixCalculator_ = 0,
                      NormalInformationMatrixCalculator *normalInformationMatrixCalculator_ = 0)
      : _projector(projector_), _statsCalculator(statsCalculator_),
        _pointInformationMatrixCalculator(pointInformationMatrixCalculator_),
        _normalInformationMatrixCalculator(normalInformationMatrixCalculator_), _keepStats(false), _keepGaussians(false) {}
  virtual ~DepthImageConverter() {}
  virtual void compute(Cloud &cloud, const DepthImage &depthImage, const Isometry3f &sensorOffset = Isometry3f::Identity()) = 0;
  PointProjector *projector() { return _projector; }
  void setProjector(PointProjector *projector_) { _projector = projector_; }
  StatsCalculator *statsCalculator() { return _statsCalculator; }
  void setStatsCalculator(StatsCalculator *statsCalculator_) { _statsCalculator = statsCalculator_; }
  PointInformationMatrixCalculator *pointInformationMatrixCalculator() { return _pointInformationMatrixCalculator; }
  void setPointInformationMatrixCalculator(PointInformationMatrixCalculator *c) { _pointInformationMatrixCalculator = c; }
  NormalInformationMatrixCalculator *normalInformationMatrixCalculator() { return _normalInformationMatrixCalculator; }
  void setNormalInformationMatrixCalculator(NormalInformationMatrixCalculator *c) { _normalInformationMatrixCalculator = c; }
  IntImage &indexImage() { return _indexImage; }
  // pwn::Stats (eigenvectors, mean, eigenvalues, n) are only materialised on request
  void setKeepStats(bool v) { _keepStats = v; }
  // the sensor-model gaussians of unProject(points, gaussians, ...) (pinholepointprojector.cpp:93-133) are only needed
  // by the Merger; the reference always computes them, here they are opt-in
  void setKeepGaussians(bool v) { _keepGaussians = v; }

 protected:
  PointProjector *_projector;
  StatsCalculator *_statsCalculator;
  PointInformationMatrixCalculator *_pointInformationMatrixCalculator;
  NormalInformationMatrixCalculator *_normalInformationMatrixCalculator;
  IntImage _indexImage;
  bool _keepStats, _keepGaussians;
};

class DepthImageConverterIntegralImage : public DepthImageConverter {
 public:
  DepthImageConverterIntegralImage(PointProjector *projector_ = 0, StatsCalculator *statsCalculator_ = 0,
                                   PointInformationMatrixCalculator *pointInformationMatrixCalculator_ = 0,
                                   NormalInformationMatrixCalculator *normalInformationMatrixCalculator_ = 0)
      : DepthImageConverter(projector_, statsCalculator_, pointInformationMatrixCalculator_, normalInformationMatrixCalculator_) {}

  nicp_stats_params abiStatsParams() const {
    StatsCalculatorIntegralImage *sc = dynamic_cast<StatsCalculatorIntegralImage *>(_statsCalculator);
    if (!sc || !_pointInformationMatrixCalculator || !_normalInformationMatrixCalculator)
      throw std::runtime_error("DepthImageConverterIntegralImage: missing statsCalculator / information matrix calculators");
    nicp_stats_params sp;
    sp.world_radius = sc->worldRadius();
    sp.min_image_radius = sc->minImageRadius();
    sp.max_image_radius = sc->maxImageRadius();
    sp.min_points = sc->minPoints();
    sp.curvature_threshold = sc->curvatureThreshold();
    sp.omega_curvature_threshold = _pointInformationMatrixCalculator->curvatureThreshold();
    InformationMatrix fp = _pointInformationMatrixCalculator->flatInformationMatrix();
    InformationMatrix fn = _normalInformationMatrixCalculator->flatInformationMatrix();
    InformationMatrix nn = _normalInformationMatrixCalculator->nonFlatInformationMatrix();
    for (int i = 0; i < 3; i++) { sp.flat_omega_p[i] = fp(i, i); sp.flat_omega_n[i] = fn(i, i); sp.nonflat_omega_n[i] = nn(i, i); }
    return sp;
  }

  // depthimageconverterintegralimage.cpp:15-55
  virtual void compute(Cloud &cloud, const DepthImage &depthImage, const Isometry3f &sensorOffset = Isometry3f::Identity()) {
    nicp_stats_params sp = abiStatsParams();
    if (MultiPointProjector *mpp = dynamic_cast<MultiPointProjector *>(_projector)) {
      mpp->setTransform(Isometry3f::Identity());
      nicp_multi_projector mp = mpp->abiMultiProjector();
      _indexImage.create(depthImage.rows, depthImage.cols);
      nicp_cloud *d = cloud.deviceForWrite(depthImage.rows * depthImage.cols);
      nicpCheck(nicp_multi_depth_to_cloud(Context::current().handle(), depthImage.data(), &mp, &sp, sensorOffset.data(),
                                          _keepStats ? 1 : 0, d, _indexImage.data()),
                "DepthImageConverterIntegralImage::compute (MultiPointProjector)");
      cloud.setHasStats(_keepStats);
      if (_keepGaussians) {
        std::vector<float> baseline, alpha;
        mpp->childSensorModels(baseline, alpha);
        nicpCheck(nicp_multi_cloud_compute_gaussians(Context::current().handle(), d, depthImage.data(), &mp, baseline.data(),
                                                     alpha.data(), sensorOffset.data()),
                  "DepthImageConverterIntegralImage::compute (MultiPointProjector gaussians)");
      }
      return;
    }
    PinholePointProjector *pp = dynamic_cast<PinholePointProjector *>(_projector);
    if (!pp) throw std::runtime_error("DepthImageConverterIntegralImage: unsupported projector type");
    pp->setImageSize(depthImage.rows, depthImage.cols);
    pp->setTransform(Isometry3f::Identity());
    _indexImage.create(depthImage.rows, depthImage.cols);
    nicp_projector p = pp->abiProjector();
    nicp_cloud *d = cloud.deviceForWrite(depthImage.rows * depthImage.cols);
    nicpCheck(nicp_depth_to_cloud(Context::current().handle(), depthImage.data(), &p, &sp, sensorOffset.data(), _keepStats ? 1 : 0,
                                  d, _indexImage.data()),
              "DepthImageConverterIntegralImage::compute");
    cloud.setHasStats(_keepStats);
    if (_keepGaussians)
      nicpCheck(nicp_cloud_compute_gaussians(Context::current().handle(), d, depthImage.data(), &p, pp->baseline(), pp->alpha(),
                                             sensorOffset.data()),
                "DepthImageConverterIntegralImage::compute (gaussians)");
    StatsCalculatorIntegralImage *sc = dynamic_cast<StatsCalculatorIntegralImage *>(_statsCalculator);
    sc->intervalImage().create(depthImage.rows, depthImage.cols);
    nicpCheck(nicp_last_interval_image(Context::current().handle(), sc->intervalImage().data()), "interval image");
  }
};

// ---- merger.h ----------------------------------------------------------------------------------------
class Merger {
 public:
  Merger() : _distanceThreshold(0.1f), _normalThreshold(cosf(10 * M_PI / 180.0f)), _maxPointDepth(10.0f),  // merger.cpp:5-13
             _depthImageConverter(0), _rows(0), _cols(0) {}
  virtual ~Merger() {}
  float distanceThreshold() const { return _distanceThreshold; }
  void setDistanceThreshold(float v) { _distanceThreshold = v; }
  float normalThreshold() const { return _normalThreshold; }
  void setNormalThreshold(float v) { _normalThreshold = v; }
  float maxPointDepth() const { return _maxPointDepth; }
  void setMaxPointDepth(float v) { _maxPointDepth = v; }
  DepthImageConverter *depthImageConverter() const { return _depthImageConverter; }
  void setDepthImageConverter(DepthImageConverter *c) { _depthImageConverter = c; }
  void setImageSize(int r, int c) { _rows = r; _cols = c; }
  int imageRows() const { return _rows; }
  int imageCols() const { return _cols; }
  // merger.h:95: (rows, cols) of the Merger's index image
  struct Size2i { int r, c; int x() const { return r; } int y() const { return c; } int operator[](int i) const { return i ? c : r; } };
  Size2i imageSize() const { Size2i s = {_rows, _cols}; return s; }
  const std::vector<int> &collapsedIndices() const { return _collapsedIndices; }

  // merger.cpp:15-119.  The Merger's projector must be a PinholePointProjector: a rig cloud (a MultiPointProjector
  // converter with setKeepGaussians(true)) is merged through a pinhole view of the Merger's image size.
  void merge(Cloud *cloud, Isometry3f transform = Isometry3f::Identity()) {
    if (_rows <= 0 || _cols <= 0) throw std::runtime_error("Merger: _indexImage has zero size");
    if (!_depthImageConverter || !_depthImageConverter->projector()) throw std::runtime_error("Merger: missing _depthImageConverter / projector");
    PinholePointProjector *pp = dynamic_cast<PinholePointProjector *>(_depthImageConverter->projector());
    if (!pp) throw std::runtime_error("Merger: the projector must be a PinholePointProjector");
    pp->setTransform(transform);
    nicp_projector p = pp->abiProjector();
    p.rows = _rows;
    p.cols = _cols;
    nicp_merge_params mp = {_distanceThreshold, _normalThreshold, _maxPointDepth};
    nicp_cloud *d = cloud->device();
    _collapsedIndices.assign(cloud->size(), -1);
    int k = 0;
    nicpCheck(nicp_merge(Context::current().handle(), d, &p, transform.data(), &mp,
                         _collapsedIndices.empty() ? 0 : _collapsedIndices.data(), &k),
              "Merger::merge");
    cloud->deviceChanged();
  }

 protected:
  float _distanceThreshold, _normalThreshold, _maxPointDepth;
  DepthImageConverter *_depthImageConverter;
  int _rows, _cols;
  std::vector<int> _collapsedIndices;
};

// ---- voxelcalculator.h ---------------------------------------------------------------------------------
class VoxelCalculator {
 public:
  VoxelCalculator() : _resolution(0.01f) {}
  virtual ~VoxelCalculator() {}
  float resolution() const { return _resolution; }
  void setResolution(float r) { _resolution = r; }
  void compute(Cloud &cloud, float res) {
    float old = _resolution;
    _resolution = res;
    compute(cloud);
    _resolution = old;
  }
  // voxelcalculator.cpp:15-73 (first point of every occupied voxel, lexicographic voxel order; see nicp_voxelize)
  void compute(Cloud &cloud) {
    int k = 0;
    nicpCheck(nicp_voxelize(Context::current().handle(), cloud.device(), _resolution, 0, &k), "VoxelCalculator::compute");
    cloud.deviceChanged();
  }

 protected:
  float _resolution;
};

// ---- correspondencefinder.h ----------------------------------------------------------------------------
class CorrespondenceFinder {
 public:
  CorrespondenceFinder()  // correspondencefinder.cpp:9-18
      : _inlierDistanceThreshold(0.5f), _flatCurvatureThreshold(0.02f), _inlierCurvatureRatioThreshold(1.3f),
        _inlierNormalAngularThreshold(cosf((float)M_PI / 6)), _numCorrespondences(0), _rows(0), _cols(0) {
    _squaredThreshold = _inlierDistanceThreshold * _inlierDistanceThreshold;
  }
  virtual ~CorrespondenceFinder() {}
  const CorrespondenceVector &correspondences() const { return _correspondences; }
  CorrespondenceVector &correspondences() { return _correspondences; }
  const IntImage &currentIndexImage() const { return _currentIndexImage; }
  IntImage &currentIndexImage() { return _currentIndexImage; }
  const IntImage &referenceIndexImage() const { return _referenceIndexImage; }
  IntImage &referenceIndexImage() { return _referenceIndexImage; }
  const DepthImage &currentDepthImage() const { return _currentDepthImage; }
  DepthImage &currentDepthImage() { return _currentDepthImage; }
  const DepthImage &referenceDepthImage() const { return _referenceDepthImage; }
  DepthImage &referenceDepthImage() { return _referenceDepthImage; }
  float squaredThreshold() const { return _squaredThreshold; }
  float inlierDistanceThreshold() const { return _inlierDistanceThreshold; }
  void setInlierDistanceThreshold(const float v) { _inlierDistanceThreshold = v; _squaredThreshold = v * v; }
  float flatCurvatureThreshold() const { return _flatCurvatureThreshold; }
  void setFlatCurvatureThreshold(const float v) { _flatCurvatureThreshold = v; }
  float inlierCurvatureRatioThreshold() const { return _inlierCurvatureRatioThreshold; }
  void setInlierCurvatureRatioThreshold(const float v) { _inlierCurvatureRatioThreshold = v; }
  float inlierNormalAngularThreshold() const { return _inlierNormalAngularThreshold; }
  void setInlierNormalAngularThreshold(const float v) { _inlierNormalAngularThreshold = v; }
  int imageRows() const { return _rows; }
  int imageCols() const { return _cols; }
  void setImageSize(const int rows_, const int cols_) {
    if (_rows != rows_ || _cols != cols_) {
      _rows = rows_;
      _cols = cols_;
      _referenceIndexImage.create(_rows, _cols);
      _currentIndexImage.create(_rows, _cols);
    }
  }
  int numCorrespondences() const { return _numCorrespondences; }

  void fillAbi(nicp_align_params &ap) const {
    ap.inlier_distance_threshold = _inlierDistanceThreshold;
    ap.inlier_normal_angular_threshold = _inlierNormalAngularThreshold;
    ap.flat_curvature_threshold = _flatCurvatureThreshold;
    ap.inlier_curvature_ratio_threshold = _inlierCurvatureRatioThreshold;
  }

  // correspondencefinder.cpp:20-118, on the finder's own index images.  The fused kernel also
  // linearises at T; those sums are discarded here.
  void compute(const Cloud &referenceScene, const Cloud &currentScene, Isometry3f T) {
    T.fixLastRow();
    nicp_align_params ap;
    fillAbi(ap);
    ap.inlier_max_chi2 = 9e3f; ap.robust_kernel = 1; ap.outer_iterations = 1; ap.inner_iterations = 1;
    const int rows = _referenceIndexImage.rows, cols = _referenceIndexImage.cols;
    IntImage corrImage(rows, cols);
    float H[36], b[6], err;
    int inl, nc;
    nicpCheck(nicp_correspond_linearize(Context::current().handle(), referenceScene.device(), currentScene.device(),
                                        _referenceIndexImage.data(), _currentIndexImage.data(), rows, cols, T.data(), &ap, H, b,
                                        &err, &inl, &nc, corrImage.data()),
              "CorrespondenceFinder::compute");
    _correspondences.assign((size_t)rows * cols, Correspondence());
    int k = 0;
    for (size_t p = 0; p < corrImage.total(); p++)
      if (corrImage.buf[p] >= 0) _correspondences[k++] = Correspondence(corrImage.buf[p], _currentIndexImage.buf[p]);
    _numCorrespondences = k;
  }
  // used by Aligner::align to publish the state of the last iteration
  void setNumCorrespondences(int n) { _numCorrespondences = n; }

 protected:
  float _inlierDistanceThreshold, _squaredThreshold, _flatCurvatureThreshold, _inlierCurvatureRatioThreshold,
      _inlierNormalAngularThreshold;
  int _numCorrespondences, _rows, _cols;
  CorrespondenceVector _correspondences;
  IntImage _referenceIndexImage, _currentIndexImage;
  DepthImage _referenceDepthImage, _currentDepthImage;
};

// ---- linearizer.h ------------------------------------------------------------------------------------------
class Aligner;
class Linearizer {
 public:
  Linearizer() : _aligner(0), _inlierMaxChi2(9e3f), _robustKernel(true), _error(0), _inliers(0) {}  // linearizer.cpp:9-15
  virtual ~Linearizer() {}
  Aligner *aligner() const { return _aligner; }
  void setAligner(Aligner *const aligner_) { _aligner = aligner_; }
  Isometry3f T() const { return _T; }
  void setT(const Isometry3f T_) { _T = T_; _T.fixLastRow(); }
  float inlierMaxChi2() const { return _inlierMaxChi2; }
  void setInlierMaxChi2(const float v) { _inlierMaxChi2 = v; }
  bool robustKernel() const { return _robustKernel; }
  void setRobustKernel(bool v) { _robustKernel = v; }
  Matrix6f H() const { return _H; }
  Vector6f b() const { return _b; }
  float error() const { return _error; }
  int inliers() const { return _inliers; }
  inline void update();  // linearizer.cpp:17-115 (defined after Aligner)
  void setResult(const float *H, const float *b, float error, int inliers) {
    for (int i = 0; i < 36; i++) _H.m[i] = H[i];
    for (int i = 0; i < 6; i++) _b.m[i] = b[i];
    _error = error;
    _inliers = inliers;
  }

 protected:
  Aligner *_aligner;
  Isometry3f _T;
  float _inlierMaxChi2;
  bool _robustKernel;
  Matrix6f _H;
  Vector6f _b;
  float _error;
  int _inliers;
};

// ---- aligner.h ----------------------------------------------------------------------------------------------
class Aligner {
 public:
  Aligner()  // aligner.cpp:13-32
      : _projector(0), _linearizer(0), _correspondenceFinder(0), _referenceCloud(0), _currentCloud(0), _outerIterations(10),
        _innerIterations(1), _totalTime(0), _error(0), _inliers(0), _minInliers(100), _rotationalMinEigenRatio(50),
        _translationalMinEigenRatio(50), _rotationalEigenRatio(0), _translationalEigenRatio(0), _debug(false),
        _frameInlierDepthThreshold(50.0f) {}
  virtual ~Aligner() {}

  PointProjector *projector() { return _projector; }
  void setProjector(PointProjector *projector_) { _projector = projector_; }
  const Cloud *referenceCloud() const { return _referenceCloud; }
  void setReferenceCloud(Cloud *referenceCloud_) { _referenceCloud = referenceCloud_; clearPriors(); }
  const Cloud *currentCloud() const { return _currentCloud; }
  void setCurrentCloud(Cloud *currentCloud_) { _currentCloud = currentCloud_; clearPriors(); }
  int outerIterations() const { return _outerIterations; }
  void setOuterIterations(const int v) { _outerIterations = v; }
  int innerIterations() const { return _innerIterations; }
  void setInnerIterations(const int v) { _innerIterations = v; }
  const Isometry3f &T() const { return _T; }
  const Isometry3f &initialGuess() const { return _initialGuess; }
  void setInitialGuess(const Isometry3f initialGuess_) { _initialGuess = initialGuess_; _initialGuess.fixLastRow(); }
  const Isometry3f &sensorOffset() const { return _referenceSensorOffset; }
  void setSensorOffset(const Isometry3f sensorOffset_) { setReferenceSensorOffset(sensorOffset_); setCurrentSensorOffset(sensorOffset_); }
  const Isometry3f &referenceSensorOffset() const { return _referenceSensorOffset; }
  void setReferenceSensorOffset(const Isometry3f v) { _referenceSensorOffset = v; _referenceSensorOffset.fixLastRow(); }
  const Isometry3f &currentSensorOffset() const { return _currentSensorOffset; }
  void setCurrentSensorOffset(const Isometry3f v) { _currentSensorOffset = v; _currentSensorOffset.fixLastRow(); }
  Linearizer *linearizer() { return _linearizer; }
  void setLinearizer(Linearizer *linearizer_) { _linearizer = linearizer_; if (_linearizer) _linearizer->setAligner(this); }
  bool debug() const { return _debug; }
  void setDebug(const bool debug_) { _debug = debug_; }
  int minInliers() const { return _minInliers; }
  void setMinInliers(const int v) { _minInliers = v; }
  float translationalMinEigenRatio() { return _translationalMinEigenRatio; }
  void setTranslationalMinEigenRatio(const float v) { _translationalMinEigenRatio = v; }
  float rotationalMinEigenRatio() { return _rotationalMinEigenRatio; }
  void setRotationalMinEigenRatio(const float v) { _rotationalMinEigenRatio = v; }
  float translationalEigenRatio() { return _translationalEigenRatio; }
  float rotationalEigenRatio() { return _rotationalEigenRatio; }
  CorrespondenceFinder *correspondenceFinder() { return _correspondenceFinder; }
  void setCorrespondenceFinder(CorrespondenceFinder *c) { _correspondenceFinder = c; }
  const Matrix6f &omega() const { return _omega; }
  float error() const { return _error; }
  int inliers() const { return _inliers; }
  double totalTime() const { return _totalTime; }
  void addRelativePrior(const Isometry3f &mean, const Matrix6f &informationMatrix) {
    nicp_prior p;
    p.kind = 0;
    for (int i = 0; i < 16; i++) { p.mean[i] = mean.data()[i]; p.reference[i] = Isometry3f().data()[i]; }
    for (int i = 0; i < 36; i++) p.information[i] = informationMatrix.m[i];
    _priors.push_back(p);
  }
  void addAbsolutePrior(const Isometry3f &referenceTransform, const Isometry3f &mean, const Matrix6f &informationMatrix) {
    nicp_prior p;
    p.kind = 1;
    for (int i = 0; i < 16; i++) { p.mean[i] = mean.data()[i]; p.reference[i] = referenceTransform.data()[i]; }
    for (int i = 0; i < 36; i++) p.information[i] = informationMatrix.m[i];
    _priors.push_back(p);
  }
  void clearPriors() { _priors.clear(); }
  // PwnMatcherBase::_frameInlierDepthThreshold (pwn_matcher_base.cpp:15): threshold of the image statistics
  void setFrameInlierDepthThreshold(float v) { _frameInlierDepthThreshold = v; }
  const nicp_align_result &lastResult() const { return _last; }

  nicp_align_params abiAlignParams() const {
    nicp_align_params ap;
    _correspondenceFinder->fillAbi(ap);
    ap.inlier_max_chi2 = _linearizer->inlierMaxChi2();
    ap.robust_kernel = _linearizer->robustKernel() ? 1 : 0;
    ap.outer_iterations = _outerIterations;
    ap.inner_iterations = _innerIterations;
    return ap;
  }

  // aligner.cpp:49-150: all iterations run on the device; the finder's images / correspondences and the
  // lineariser's H/b are fetched afterwards (what matchClouds reads, pwn_matcher_base.cpp:156-171).
  virtual void align() {
    if (!_projector || !_linearizer || !_correspondenceFinder || !_referenceCloud || !_currentCloud)
      throw std::runtime_error("Aligner: missing projector / linearizer / correspondenceFinder / clouds");
    PinholePointProjector *pp = dynamic_cast<PinholePointProjector *>(_projector);
    MultiPointProjector *mpp = dynamic_cast<MultiPointProjector *>(_projector);
    if (!pp && !mpp) throw std::runtime_error("Aligner: unsupported projector type");
    struct timeval tvStart, tvEnd;
    gettimeofday(&tvStart, 0);
    nicp_context *ctx = Context::current().handle();
    nicp_projector p;
    nicp_align_params ap = abiAlignParams();
    if (mpp) {
      nicp_multi_projector mp = mpp->abiMultiProjector();
      nicp_multi_image_size(&mp, &p.rows, &p.cols);
      nicpCheck(nicp_multi_align(ctx, _referenceCloud->device(), _currentCloud->device(), &mp, &ap, _referenceSensorOffset.data(),
                                 _currentSensorOffset.data(), _initialGuess.data(), _priors.empty() ? 0 : &_priors[0],
                                 (int)_priors.size(), _frameInlierDepthThreshold, &_last),
                "Aligner::align (MultiPointProjector)");
    } else {
      p = pp->abiProjector();
      nicpCheck(nicp_align(ctx, _referenceCloud->device(), _currentCloud->device(), &p, &ap, _referenceSensorOffset.data(),
                           _currentSensorOffset.data(), _initialGuess.data(), _priors.empty() ? 0 : &_priors[0],
                           (int)_priors.size(), _frameInlierDepthThreshold, &_last),
                "Aligner::align");
    }
    for (int i = 0; i < 16; i++) _T.data()[i] = _last.T[i];
    for (int i = 0; i < 36; i++) _omega.m[i] = _last.omega[i];
    _error = _last.error;
    _inliers = _last.inliers;
    _translationalEigenRatio = _last.translational_eigen_ratio;
    _rotationalEigenRatio = _last.rotational_eigen_ratio;
    gettimeofday(&tvEnd, 0);
    _totalTime = (tvEnd.tv_sec - tvStart.tv_sec) * 1000.0 + (tvEnd.tv_usec - tvStart.tv_usec) * 0.001;
    // publish the state the callers read after align()
    CorrespondenceFinder *cf = _correspondenceFinder;
    cf->referenceIndexImage().create(p.rows, p.cols);
    cf->currentIndexImage().create(p.rows, p.cols);
    cf->referenceDepthImage().create(p.rows, p.cols);
    cf->currentDepthImage().create(p.rows, p.cols);
    std::vector<int> corr(2 * (size_t)p.rows * p.cols, -1);
    float H[36], b[6];
    nicpCheck(nicp_align_get_state(ctx, cf->referenceIndexImage().data(), cf->referenceDepthImage().data(),
                                   cf->currentIndexImage().data(), cf->currentDepthImage().data(), corr.data(), H, b),
              "Aligner::align state");
    cf->correspondences().assign((size_t)p.rows * p.cols, Correspondence());
    int k = 0;
    while ((size_t)k < (size_t)p.rows * p.cols && corr[2 * (size_t)k] >= 0) {
      cf->correspondences()[k] = Correspondence(corr[2 * (size_t)k], corr[2 * (size_t)k + 1]);
      k++;
    }
    cf->setNumCorrespondences(k);
    Isometry3f invT = _T.inverse();
    _linearizer->setT(invT);
    _linearizer->setResult(H, b, _last.error, _last.inliers);
    _projector->setTransform(_T * _referenceSensorOffset);
  }

 protected:
  PointProjector *_projector;
  Linearizer *_linearizer;
  CorrespondenceFinder *_correspondenceFinder;
  Cloud *_referenceCloud, *_currentCloud;
  int _outerIterations, _innerIterations;
  Isometry3f _T, _initialGuess, _referenceSensorOffset, _currentSensorOffset;
  double _totalTime;
  float _error;
  int _inliers, _minInliers;
  float _rotationalMinEigenRatio, _translationalMinEigenRatio, _rotationalEigenRatio, _translationalEigenRatio;
  bool _debug;
  float _frameInlierDepthThreshold;
  Matrix6f _omega;
  std::vector<nicp_prior> _priors;
  nicp_align_result _last;
};

inline void Linearizer::update() {
  if (!_aligner) throw std::runtime_error("Linearizer: missing _aligner");
  CorrespondenceFinder *cf = _aligner->correspondenceFinder();
  const int n = cf->numCorrespondences();
  std::vector<int> corr(2 * (size_t)(n > 0 ? n : 1));
  for (int i = 0; i < n; i++) {
    corr[2 * (size_t)i] = cf->correspondences()[i].referenceIndex;
    corr[2 * (size_t)i + 1] = cf->correspondences()[i].currentIndex;
  }
  nicp_align_params ap;
  cf->fillAbi(ap);
  ap.inlier_max_chi2 = _inlierMaxChi2;
  ap.robust_kernel = _robustKernel ? 1 : 0;
  ap.outer_iterations = 1;
  ap.inner_iterations = 1;
  float H[36], b[6];
  nicpCheck(nicp_linearize(Context::current().handle(), _aligner->referenceCloud()->device(), _aligner->currentCloud()->device(),
                           corr.data(), n, _T.data(), &ap, H, b, &_error, &_inliers),
            "Linearizer::update");
  for (int i = 0; i < 36; i++) _H.m[i] = H[i];
  for (int i = 0; i < 6; i++) _b.m[i] = b[i];
}

}  // namespace pwn

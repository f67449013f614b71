// map_ops.cu -- local-map maintenance on the device (SURVEY.md section 8f rank 3).
//
// Replaces
//   PinholePointProjector::unProject(points, gaussians, ...)   pinholepointprojector.cpp:93-133  -> k_gaussians
//   Gaussian3fVector::transformInPlace                          gaussian3.h:26-36                 -> k_gauss_transform
//   Gaussian::addInformation / _updateInfo / _updateMoments     basemath/gaussian.h:49-90          -> gauss_* device functions
//   Merger::merge                                               merger.cpp:15-119                 -> k_merge_* + compaction
//   VoxelCalculator::compute                                    voxelcalculator.cpp:15-73         -> k_voxel_* + radix sort
//
// Merger::merge is a sequential loop in the reference; what makes it order-sensitive is the float32 accumulation of
// information matrices into the z-buffer winner of a pixel.  Here every point classifies itself in parallel, the
// contributors of a target are binned (count -> exclusive scan -> fill), each target sorts its (short) list by point
// index and adds the contributions in exactly the reference's order.  The surviving points are compacted in
// index order with a scan, as the reference's second loop does.
//
// VoxelCalculator keeps the first point (lowest index) of every occupied voxel and emits them in the order of its
// std::map.  The reference's key comparator (voxelcalculator.h:40-46) is not a strict weak ordering, so the content of
// that map depends on the C++ library's tree; the device path implements the lexicographic order the comparator
// evidently intends: voxel keys are packed into 64 bits, a stable LSD radix sort orders (key, index), segment heads are
// the representatives.  tests/ quantify the difference against a libstdc++ std::map with the comparator as written.
#include "nicp_internal.cuh"
#include <climits>

namespace nicp {

// ---------------------------------------------------------------------------------------------
// scratch: one grow-only device buffer per context, carved by a bump pointer
// ---------------------------------------------------------------------------------------------
struct Bump {
  unsigned char *base;
  size_t used, cap;
  template <typename T>
  T *take(size_t count) {
    size_t bytes = (count * sizeof(T) + 255) & ~(size_t)255;
    T *p = reinterpret_cast<T *>(base + used);
    used += bytes;
    return used <= cap ? p : nullptr;
  }
};
static int map_scratch(nicp_context *ctx, size_t bytes, Bump *b) {
  if (ctx->mapScratchBytes < bytes) {
    NICP_CUDA(cudaStreamSynchronize(ctx->stream));
    if (ctx->d_mapScratch) cudaFree(ctx->d_mapScratch);
    ctx->d_mapScratch = nullptr;
    ctx->mapScratchBytes = 0;
    size_t want = bytes + bytes / 4;
    cudaError_t e = cudaMalloc(&ctx->d_mapScratch, want);
    if (e != cudaSuccess) {
      set_error("cudaMalloc(%zu bytes) of the map scratch failed: %s", want, cudaGetErrorString(e));
      return NICP_ERR_ALLOC;
    }
    ctx->mapScratchBytes = want;
  }
  b->base = static_cast<unsigned char *>(ctx->d_mapScratch);
  b->used = 0;
  b->cap = ctx->mapScratchBytes;
  return NICP_OK;
}
static size_t pad256(size_t bytes) { return (bytes + 255) & ~(size_t)255; }

// ---------------------------------------------------------------------------------------------
// exclusive scan of an int array (2048 items per CTA, recursive over the CTA totals)
// ---------------------------------------------------------------------------------------------
constexpr int kScanThreads = 256, kScanItems = 8, kScanTile = kScanThreads * kScanItems;

__global__ void __launch_bounds__(kScanThreads) k_scan_block(const int *__restrict__ in, int *__restrict__ out, int n,
                                                            int *__restrict__ blockSums) {
  __shared__ int warpSums[kScanThreads / 32];
  const int base = blockIdx.x * kScanTile + threadIdx.x * kScanItems;
  int v[kScanItems], s = 0;
#pragma unroll
  for (int k = 0; k < kScanItems; k++) {
    v[k] = (base + k < n) ? in[base + k] : 0;
    s += v[k];
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) warpSums[warp] = incl;
  __syncthreads();
  int warpPrefix = 0;
  for (int w = 0; w < warp; w++) warpPrefix += warpSums[w];
  int running = warpPrefix + incl - s;
#pragma unroll
  for (int k = 0; k < kScanItems; k++) {
    if (base + k < n) out[base + k] = running;
    running += v[k];
  }
  if (threadIdx.x == kScanThreads - 1) blockSums[blockIdx.x] = running;
}
__global__ void __launch_bounds__(kScanThreads) k_scan_add(int *__restrict__ out, const int *__restrict__ blockOffsets, int n) {
  const int off = blockOffsets[blockIdx.x];
  const int base = blockIdx.x * kScanTile + threadIdx.x * kScanItems;
#pragma unroll
  for (int k = 0; k < kScanItems; k++)
    if (base + k < n) out[base + k] += off;
}
__global__ void k_scan_total(const int *__restrict__ in, const int *__restrict__ out, int n, int *__restrict__ total) {
  *total = n > 0 ? out[n - 1] + in[n - 1] : 0;
}
static size_t scan_scratch_ints(int n) {
  size_t tot = 0;
  while (n > 1) {
    int nb = (n + kScanTile - 1) / kScanTile;
    tot += 2 * (size_t)nb + 64;
    n = nb;
  }
  return tot + 64;
}
// in != out; scratch holds scan_scratch_ints(n) ints
static int scan_rec(nicp_context *ctx, const int *in, int *out, int n, int *scratch) {
  if (n <= 0) return NICP_OK;
  const int nb = (n + kScanTile - 1) / kScanTile;
  k_scan_block<<<nb, kScanThreads, 0, ctx->stream>>>(in, out, n, scratch);
  NICP_CHECK_LAUNCH(ctx);
  if (nb > 1) {
    int *sums = scratch, *offsets = scratch + nb;
    int rc = scan_rec(ctx, sums, offsets, nb, scratch + 2 * (size_t)nb + 64);
    if (rc) return rc;
    k_scan_add<<<nb, kScanThreads, 0, ctx->stream>>>(out, offsets, n);
    NICP_CHECK_LAUNCH(ctx);
  }
  return NICP_OK;
}
static int exclusive_scan(nicp_context *ctx, const int *in, int *out, int n, int *scratch, int *d_total) {
  int rc = scan_rec(ctx, in, out, n, scratch);
  if (rc) return rc;
  if (d_total) {
    k_scan_total<<<1, 1, 0, ctx->stream>>>(in, out, n, d_total);
    NICP_CHECK_LAUNCH(ctx);
  }
  return NICP_OK;
}

// ---------------------------------------------------------------------------------------------
// Gaussian3f: 24 floats (mean 3, covariance 9, information vector 3, information matrix 9) + flags
// ---------------------------------------------------------------------------------------------
constexpr int kGF = NICP_GAUSS_FLOATS;
__device__ __forceinline__ void gauss_load(const float *__restrict__ src, float *g) {
  const float4 *s = reinterpret_cast<const float4 *>(src);
#pragma unroll
  for (int k = 0; k < kGF / 4; k++) {
    float4 v = s[k];
    g[4 * k] = v.x; g[4 * k + 1] = v.y; g[4 * k + 2] = v.z; g[4 * k + 3] = v.w;
  }
}
__device__ __forceinline__ void gauss_store(float *__restrict__ dst, const float *g) {
  float4 *d = reinterpret_cast<float4 *>(dst);
#pragma unroll
  for (int k = 0; k < kGF / 4; k++) d[k] = make_float4(g[4 * k], g[4 * k + 1], g[4 * k + 2], g[4 * k + 3]);
}
__device__ __forceinline__ void mat3_vec(const float *A, const float *v, float *o) {
  float t0 = dot3(NM3(A, 0, 0), NM3(A, 0, 1), NM3(A, 0, 2), v[0], v[1], v[2]);
  float t1 = dot3(NM3(A, 1, 0), NM3(A, 1, 1), NM3(A, 1, 2), v[0], v[1], v[2]);
  float t2 = dot3(NM3(A, 2, 0), NM3(A, 2, 1), NM3(A, 2, 2), v[0], v[1], v[2]);
  o[0] = t0; o[1] = t1; o[2] = t2;
}
__device__ __forceinline__ void mat3_mul(const float *A, const float *B, float *C) {  // C = A*B (C may alias neither)
  for (int c = 0; c < 3; c++)
    for (int r = 0; r < 3; r++)
      NM3(C, r, c) = dot3(NM3(A, r, 0), NM3(A, r, 1), NM3(A, r, 2), NM3(B, 0, c), NM3(B, 1, c), NM3(B, 2, c));
}
__device__ __forceinline__ void mat3_mul_bt(const float *A, const float *B, float *C) {  // C = A*B^T
  for (int c = 0; c < 3; c++)
    for (int r = 0; r < 3; r++)
      NM3(C, r, c) = dot3(NM3(A, r, 0), NM3(A, r, 1), NM3(A, r, 2), NM3(B, c, 0), NM3(B, c, 1), NM3(B, c, 2));
}
// Gaussian::_updateMoments / _updateInfo (gaussian.h:76-90)
__device__ __forceinline__ void gauss_update_moments(float *g, int &f) {
  if (f & NICP_GAUSS_MOMENTS) return;
  mat3_inverse(g + 15, g + 3);
  mat3_vec(g + 3, g + 12, g);
  f |= NICP_GAUSS_MOMENTS;
}
__device__ __forceinline__ void gauss_update_info(float *g, int &f) {
  if (f & NICP_GAUSS_INFO) return;
  mat3_inverse(g + 3, g + 15);
  mat3_vec(g + 15, g, g + 12);
  f |= NICP_GAUSS_INFO;
}

__global__ void k_valid_flags(const float *__restrict__ depth, int n, float minD, float maxD, int *__restrict__ flags) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float d = depth[i];
  flags[i] = (d < minD || d > maxD) ? 0 : 1;
}

struct Mat3 { float m[9]; };
// pinholepointprojector.cpp:104-123 for the valid pixel of image coordinates (x, y) and depth z (a pinhole image: x = c,
// y = r): g = the gaussian in the moments form
__device__ __forceinline__ void gauss_sensor_model(float x, float y, float z, const Mat3 &iK, const Affine &iKRt, float fB,
                                                   float alpha, float *g) {
#pragma unroll
  for (int k = 0; k < kGF; k++) g[k] = 0.0f;
  xform_point(iKRt, fmul(x, z), fmul(y, z), z, g[0], g[1], g[2]);
  const float zVariation = fdiv(fmul(fmul(alpha, z), z), fadd(fB, fmul(z, alpha)));
  float J0[9] = {z, 0.0f, 0.0f, 0.0f, z, 0.0f, x, y, 1.0f}, J[9], JD[9];
  mat3_mul(iK.m, J0, J);
  const float dg[3] = {3.0f, 3.0f, zVariation};
  for (int j = 0; j < 3; j++)
    for (int i = 0; i < 3; i++) NM3(JD, i, j) = fmul(NM3(J, i, j), dg[j]);
  mat3_mul_bt(JD, J, g + 3);
}
// cov' = (R cov) R^T in place
__device__ __forceinline__ void gauss_rotate_cov(const float *R, float *cov) {
  float RC[9], out[9];
  mat3_mul(R, cov, RC);
  mat3_mul_bt(RC, R, out);
  for (int k = 0; k < 9; k++) cov[k] = out[k];
}
// gaussian3.h:26-36 for one gaussian whose moments are up to date: mean' = R mean + t, cov' = (R cov) R^T
__device__ __forceinline__ void gauss_xform_moments(const Affine &M, float *g) {
  float R[9];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) NM3(R, r, c) = M.r[r][c];
  float mean[3];
  mat3_vec(R, g, mean);
  g[0] = fadd(mean[0], M.r[0][3]);
  g[1] = fadd(mean[1], M.r[1][3]);
  g[2] = fadd(mean[2], M.r[2][3]);
  gauss_rotate_cov(R, g + 3);
}

// the valid pixels of one depth image; slot = raster rank of the pixel
__global__ void k_gaussians(const float *__restrict__ depth, const int *__restrict__ rank, int rows, int cols, float minD,
                            float maxD, Mat3 iK, Affine iKRt, float fB, float alpha, int capacity,
                            float *__restrict__ gauss, int *__restrict__ gflags) {
  int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= rows * cols) return;
  const float z = depth[pix];
  if (z < minD || z > maxD) return;
  const int slot = rank[pix];
  if (slot >= capacity) return;
  const int r = pix / cols, c = pix - r * cols;
  float g[kGF];
  gauss_sensor_model((float)c, (float)r, z, iK, iKRt, fB, alpha, g);
  gauss_store(gauss + (size_t)kGF * slot, g);
  gflags[slot] = NICP_GAUSS_MOMENTS;
}

// gaussian3.h:26-36 for entries [first, first + *count) (count read on the device)
__global__ void k_gauss_transform(float *__restrict__ gauss, int *__restrict__ gflags, const int *__restrict__ firstPtr,
                                  int firstConst, const int *__restrict__ countPtr, int capacity, Affine M) {
  const int first = firstPtr ? *firstPtr : firstConst;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= *countPtr) return;
  i += first;
  if (i >= capacity) return;
  float g[kGF];
  gauss_load(gauss + (size_t)kGF * i, g);
  int f = gflags[i];
  gauss_update_moments(g, f);
  gauss_xform_moments(M, g);
  gauss_store(gauss + (size_t)kGF * i, g);
  gflags[i] = NICP_GAUSS_MOMENTS;
}

static bool is_identity16(const float *m) {
  for (int r = 0; r < 4; r++)
    for (int c = 0; c < 4; c++)
      if (NM4(m, r, c) != (r == c ? 1.0f : 0.0f)) return false;
  return true;
}

int cloud_ensure_gaussians(nicp_context *ctx, nicp_cloud *cloud) {
  if (cloud->gauss) return NICP_OK;
  NICP_CUDA(cudaSetDevice(ctx->device));
  cudaError_t e = cudaMalloc(&cloud->gauss, (size_t)cloud->capacity * kGF * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&cloud->gflags, (size_t)cloud->capacity * sizeof(int));
  if (e != cudaSuccess) {
    set_error("cudaMalloc of the gaussians (%d points) failed: %s", cloud->capacity, cudaGetErrorString(e));
    return NICP_ERR_ALLOC;
  }
  return NICP_OK;
}

int launch_gauss_transform(nicp_context *ctx, nicp_cloud *cloud, const int *d_first, int first, const int *d_count,
                           int maxCount, const float T[16]) {
  float m[16];
  for (int i = 0; i < 16; i++) m[i] = T[i];
  fix_last_row(m);
  if (is_identity16(m) || maxCount <= 0) return NICP_OK;
  k_gauss_transform<<<(maxCount + 127) / 128, 128, 0, ctx->stream>>>(cloud->gauss, cloud->gflags, d_first, first, d_count,
                                                                     cloud->capacity, affine_from(m));
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

// Cloud::add (cloud.cpp:145-171) for the gaussians: copies of src's gaussians, transformed, behind dst's *dstN entries
__global__ void k_gauss_append(const float *__restrict__ sg, const int *__restrict__ sf, const int *__restrict__ srcN,
                               int srcCapacity, float *__restrict__ dg, int *__restrict__ df, const int *__restrict__ dstN,
                               int dstCapacity, Affine M, int identity) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= *srcN || i >= srcCapacity) return;
  const size_t o = (size_t)*dstN + i;
  if (o >= (size_t)dstCapacity) return;
  float g[kGF];
  gauss_load(sg + (size_t)kGF * i, g);
  int f = sf[i];
  if (!identity) {
    gauss_update_moments(g, f);
    gauss_xform_moments(M, g);
    f = NICP_GAUSS_MOMENTS;
  }
  gauss_store(dg + kGF * o, g);
  df[o] = f;
}
// must run before the destination count is advanced
int launch_gauss_append(nicp_context *ctx, nicp_cloud *dst, const nicp_cloud *src, const float T[16]) {
  if (!src->has_gauss) return NICP_OK;
  int rc = cloud_ensure_gaussians(ctx, dst);
  if (rc) return rc;
  if (!dst->has_gauss) {  // points that were already there get default (all-zero) gaussians, like vector::resize
    NICP_CUDA(cudaMemsetAsync(dst->gauss, 0, sizeof(float) * kGF * (size_t)dst->capacity, ctx->stream));
    NICP_CUDA(cudaMemsetAsync(dst->gflags, 0, sizeof(int) * (size_t)dst->capacity, ctx->stream));
    dst->has_gauss = true;
  }
  float m[16];
  for (int i = 0; i < 16; i++) m[i] = T[i];
  fix_last_row(m);
  k_gauss_append<<<(src->capacity + 127) / 128, 128, 0, ctx->stream>>>(src->gauss, src->gflags, src->d_n, src->capacity,
                                                                      dst->gauss, dst->gflags, dst->d_n, dst->capacity,
                                                                      affine_from(m), is_identity16(m) ? 1 : 0);
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

// host-side constants of the sensor model: unProject matrix with the projector at identity, K^-1, baseline * fx
struct SensorModel {
  Affine iKRt;
  Mat3 iK;
  float fB;
};
static SensorModel sensor_model(const nicp_projector *proj, float baseline) {
  SensorModel s;
  float I4[16], iKRt[16];
  mat4_identity(I4);
  compute_iKRt(proj->K, I4, iKRt);
  s.iKRt = affine_from(iKRt);
  mat3_inverse(proj->K, s.iK.m);
  s.fB = fmul(baseline, NM3(proj->K, 0, 0));
  return s;
}

// depth: host image.  The cloud must have been built from the same image, projector and sensor offset.
int run_compute_gaussians(nicp_context *ctx, nicp_cloud *cloud, const float *depth, const nicp_projector *proj,
                          float baseline, float alpha, const float sensorOffset[16]) {
  const int P = proj->rows * proj->cols;
  int rc = cloud_ensure_gaussians(ctx, cloud);
  if (rc) return rc;
  Bump b;
  const size_t need = pad256(sizeof(float) * P) + 2 * pad256(sizeof(int) * P) + pad256(sizeof(int) * scan_scratch_ints(P)) + 1024;
  if ((rc = map_scratch(ctx, need, &b))) return rc;
  float *d_depth = b.take<float>(P);
  int *d_flags = b.take<int>(P), *d_rank = b.take<int>(P), *d_scan = b.take<int>(scan_scratch_ints(P)), *d_total = b.take<int>(1);
  NICP_CUDA(cudaMemcpyAsync(d_depth, depth, sizeof(float) * P, cudaMemcpyHostToDevice, ctx->stream));
  k_valid_flags<<<(P + 255) / 256, 256, 0, ctx->stream>>>(d_depth, P, proj->min_distance, proj->max_distance, d_flags);
  NICP_CHECK_LAUNCH(ctx);
  if ((rc = exclusive_scan(ctx, d_flags, d_rank, P, d_scan, d_total))) return rc;
  const SensorModel sm = sensor_model(proj, baseline);
  k_gaussians<<<(P + 127) / 128, 128, 0, ctx->stream>>>(d_depth, d_rank, proj->rows, proj->cols, proj->min_distance,
                                                        proj->max_distance, sm.iK, sm.iKRt, sm.fB, alpha, cloud->capacity,
                                                        cloud->gauss, cloud->gflags);
  NICP_CHECK_LAUNCH(ctx);
  int total = 0;
  NICP_CUDA(cudaMemcpyAsync(&total, d_total, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  int n = 0;
  NICP_CUDA(cudaMemcpy(&n, cloud->d_n, sizeof(int), cudaMemcpyDeviceToHost));
  if (total != n) {
    set_error("nicp_cloud_compute_gaussians: the depth image has %d valid pixels but the cloud holds %d points", total, n);
    return NICP_ERR_INVALID;
  }
  if ((rc = launch_gauss_transform(ctx, cloud, nullptr, 0, cloud->d_n, n, sensorOffset))) return rc;
  cloud->has_gauss = true;
  return NICP_OK;
}

// ---------------------------------------------------------------------------------------------
// sensor-model gaussians of a MultiPointProjector rig (DESIGN.md, known deviations): the gaussian of a point of camera i
// is child i's PinholePointProjector model at its pixel (u, v) = (r, c - colOff_i) of the composite image, its mean is the
// rig point itself (pixel_point<true>) and its covariance is rotated into the rig frame by the rotation of offset_i
// ---------------------------------------------------------------------------------------------
// per camera: unProject matrix with the rig at identity (PrepCams::iKRt), K_i^-1, baseline_i * fx_i, alpha_i, the rotation
// of offset_i and whether it applies (0: offset_i is exactly the identity)
struct RigSensor {
  CamGeom g;
  Affine iKRt[kMaxCams];
  Mat3 iK[kMaxCams], R[kMaxCams];
  float fB[kMaxCams], alpha[kMaxCams];
  int rotate[kMaxCams];
};
static RigSensor rig_sensor(const CamSet &cams, const float *baseline, const float *alpha) {
  RigSensor s;
  memset(&s, 0, sizeof s);
  s.g = geom_of(cams);
  for (int i = 0; i < cams.n; i++) {
    float iKRt[16];
    compute_iKRt(cams.K[i], cams.offset[i], iKRt);
    s.iKRt[i] = affine_from(iKRt);
    mat3_inverse(cams.K[i], s.iK[i].m);
    s.fB[i] = fmul(baseline[i], NM3(cams.K[i], 0, 0));
    s.alpha[i] = alpha[i];
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) NM3(s.R[i].m, r, c) = NM4(cams.offset[i], r, c);
    s.rotate[i] = is_identity16(cams.offset[i]) ? 0 : 1;
  }
  return s;
}
// the camera whose column block holds composite column c (the blocks tile the columns; pixel_point<true>)
__device__ __forceinline__ int rig_block(const CamGeom &g, int c) {
  int cam = 0;
  for (int i = 0; i < g.n; i++)
    if (c >= g.colOff[i] && c < g.colOff[i] + g.height[i]) cam = i;
  return cam;
}
__device__ __forceinline__ bool rig_valid(const CamGeom &g, int cam, int r, float z) {
  return r < g.width[cam] && !(z < g.minD[cam] || z > g.maxD[cam]);
}
// the gaussian of the valid pixel (r, c) of camera cam, depth z, in the rig frame before the rig's sensor offset
__device__ __forceinline__ void rig_gaussian(const RigSensor &S, int cam, int r, int c, float z, float *g) {
  gauss_sensor_model((float)r, (float)(c - S.g.colOff[cam]), z, S.iK[cam], S.iKRt[cam], S.fB[cam], S.alpha[cam], g);
  if (S.rotate[cam]) gauss_rotate_cov(S.R[cam].m, g + 3);
}
// position of composite pixel (r, c) of camera cam in the rig's point order (camera by camera, raster order inside the
// camera's rows x height_i block): an exclusive scan of valid flags stored there is the compacted index of every valid pixel
__device__ __forceinline__ size_t rig_order(const CamGeom &g, int cam, int r, int c, int rows) {
  return (size_t)rows * g.colOff[cam] + (size_t)r * g.height[cam] + (c - g.colOff[cam]);
}
__global__ void k_rig_valid_flags(const float *__restrict__ depth, int rows, int cols, CamGeom g, int *__restrict__ flags) {
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= rows * cols) return;
  const int r = pix / cols, c = pix - r * cols;
  const int cam = rig_block(g, c);
  flags[rig_order(g, cam, r, c, rows)] = rig_valid(g, cam, r, depth[pix]) ? 1 : 0;
}
__global__ void k_rig_gaussians(const float *__restrict__ depth, const int *__restrict__ rank, int rows, int cols, RigSensor S,
                                int capacity, float *__restrict__ gauss, int *__restrict__ gflags) {
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= rows * cols) return;
  const float z = depth[pix];
  const int r = pix / cols, c = pix - r * cols;
  const int cam = rig_block(S.g, c);
  if (!rig_valid(S.g, cam, r, z)) return;
  const int slot = rank[rig_order(S.g, cam, r, c, rows)];
  if (slot >= capacity) return;
  float g[kGF];
  rig_gaussian(S, cam, r, c, z, g);
  gauss_store(gauss + (size_t)kGF * slot, g);
  gflags[slot] = NICP_GAUSS_MOMENTS;
}

// depth: host composite image (rows x cols) the cloud was built from with the same rig and sensor offset; baseline, alpha:
// one per camera
int run_multi_compute_gaussians(nicp_context *ctx, nicp_cloud *cloud, const float *depth, const CamSet &cams, int rows,
                                int cols, const float *baseline, const float *alpha, const float sensorOffset[16]) {
  const int P = rows * cols;
  int rc = cloud_ensure_gaussians(ctx, cloud);
  if (rc) return rc;
  Bump b;
  const size_t need = pad256(sizeof(float) * P) + 2 * pad256(sizeof(int) * P) + pad256(sizeof(int) * scan_scratch_ints(P)) + 1024;
  if ((rc = map_scratch(ctx, need, &b))) return rc;
  float *d_depth = b.take<float>(P);
  int *d_flags = b.take<int>(P), *d_rank = b.take<int>(P), *d_scan = b.take<int>(scan_scratch_ints(P)), *d_total = b.take<int>(1);
  NICP_CUDA(cudaMemcpyAsync(d_depth, depth, sizeof(float) * P, cudaMemcpyHostToDevice, ctx->stream));
  const RigSensor S = rig_sensor(cams, baseline, alpha);
  k_rig_valid_flags<<<(P + 255) / 256, 256, 0, ctx->stream>>>(d_depth, rows, cols, S.g, d_flags);
  NICP_CHECK_LAUNCH(ctx);
  if ((rc = exclusive_scan(ctx, d_flags, d_rank, P, d_scan, d_total))) return rc;
  k_rig_gaussians<<<(P + 127) / 128, 128, 0, ctx->stream>>>(d_depth, d_rank, rows, cols, S, cloud->capacity, cloud->gauss,
                                                            cloud->gflags);
  NICP_CHECK_LAUNCH(ctx);
  int total = 0;
  NICP_CUDA(cudaMemcpyAsync(&total, d_total, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  int n = 0;
  NICP_CUDA(cudaMemcpy(&n, cloud->d_n, sizeof(int), cudaMemcpyDeviceToHost));
  if (total != n) {
    set_error("nicp_multi_cloud_compute_gaussians: the depth image has %d valid pixels but the cloud holds %d points", total, n);
    return NICP_ERR_INVALID;
  }
  if ((rc = launch_gauss_transform(ctx, cloud, nullptr, 0, cloud->d_n, n, sensorOffset))) return rc;
  cloud->has_gauss = true;
  return NICP_OK;
}

// ---------------------------------------------------------------------------------------------
// local map from one launch set of the batched frame preparation (nicp_raw_depth_to_local_map)
// ---------------------------------------------------------------------------------------------
// The frame clouds of the set (frame f = blockIdx.y), the poses they are appended with and the sensor offset of their
// gaussians: a kernel parameter, like PrepBatch.
struct LocalMapSet {
  const float4 *points[kMaxPrepBatch], *normals[kMaxPrepBatch], *omega[kMaxPrepBatch];
  float *gauss[kMaxPrepBatch];
  int *gflags[kMaxPrepBatch];
  const int *count[kMaxPrepBatch];
  Affine pose[kMaxPrepBatch];
  int poseIdentity[kMaxPrepBatch];
  Affine offset;
  int offsetIdentity;
};

// nicp_cloud_compute_gaussians for every frame of the set, from the depth and integral images the set's preparation left
// in the batch scratch: the slot of a valid pixel is its raster rank from channel 0 of the integral image (the compacted
// index k_stats wrote the point to), then the sensor offset as a second rounded step (k_gauss_transform).
__global__ void k_local_map_gaussians(LocalMapSet S, const float *__restrict__ depth0, const float *__restrict__ integral0,
                                      size_t framePixels, int rows, int cols, float minD, float maxD, Mat3 iK, Affine iKRt,
                                      float fB, float alpha) {
  const int f = blockIdx.y;
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= rows * cols) return;
  const float z = depth0[(size_t)f * framePixels + pix];
  if (z < minD || z > maxD) return;
  const int r = pix / cols, c = pix - r * cols;
  const int slot = raster_rank(integral0 + (size_t)f * framePixels * kIntegralCh, r, c, cols);
  float g[kGF];
  gauss_sensor_model((float)c, (float)r, z, iK, iKRt, fB, alpha, g);
  if (!S.offsetIdentity) gauss_xform_moments(S.offset, g);
  gauss_store(S.gauss[f] + (size_t)kGF * slot, g);
  S.gflags[f][slot] = NICP_GAUSS_MOMENTS;
}
// the same for the rig frames of a set: the slot of a valid pixel is its rig rank (k_stats<true>)
__global__ void k_local_map_rig_gaussians(LocalMapSet S, const float *__restrict__ depth0, const float *__restrict__ integral0,
                                          size_t framePixels, int rows, int cols, RigSensor R) {
  const int f = blockIdx.y;
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= rows * cols) return;
  const float z = depth0[(size_t)f * framePixels + pix];
  const int r = pix / cols, c = pix - r * cols;
  const int cam = rig_block(R.g, c);
  if (!rig_valid(R.g, cam, r, z)) return;
  const int slot = rig_rank(integral0 + (size_t)f * framePixels * kIntegralCh, r, c, rows, cols, R.g.colOff[cam], R.g.height[cam]);
  float g[kGF];
  rig_gaussian(R, cam, r, c, z, g);
  if (!S.offsetIdentity) gauss_xform_moments(S.offset, g);
  gauss_store(S.gauss[f] + (size_t)kGF * slot, g);
  S.gflags[f][slot] = NICP_GAUSS_MOMENTS;
}

// Cloud::add (cloud.cpp:145-171) of one point with its gaussian: source point i moved by M (unless identity) and written at
// destination slot o.  The per-point body of k_local_map_append and k_scene_append.
__device__ __forceinline__ void append_point(const float4 *__restrict__ sp, const float4 *__restrict__ sn,
                                             const float4 *__restrict__ som, const float *__restrict__ sg,
                                             const int *__restrict__ sf, int i, const Affine &M, int identity,
                                             float4 *__restrict__ dp, float4 *__restrict__ dn, float4 *__restrict__ dom,
                                             float *__restrict__ dg, int *__restrict__ df, size_t o) {
  // the sources are read-only for the whole launch: read them through the non-coherent path (ld.global.nc), which the
  // restrict qualifiers of an inlined helper do not let the compiler infer on its own
  float4 p = __ldg(sp + i), nn = __ldg(sn + i);
  const float4 *so = som + 3 * (size_t)i;
  float4 o0 = __ldg(so), o1 = __ldg(so + 1), o2 = __ldg(so + 2);
  float g[kGF];
  const float4 *gs = reinterpret_cast<const float4 *>(sg + (size_t)kGF * i);
#pragma unroll
  for (int k = 0; k < kGF / 4; k++) {
    const float4 v = __ldg(gs + k);
    g[4 * k] = v.x; g[4 * k + 1] = v.y; g[4 * k + 2] = v.z; g[4 * k + 3] = v.w;
  }
  int gf = __ldg(sf + i);
  if (!identity) {
    xform_record(M, p, nn, o0, o1, o2);
    gauss_update_moments(g, gf);
    gauss_xform_moments(M, g);
    gf = NICP_GAUSS_MOMENTS;
  }
  dp[o] = p;
  dn[o] = nn;
  dom[3 * o] = o0;
  dom[3 * o + 1] = o1;
  dom[3 * o + 2] = o2;
  gauss_store(dg + kGF * o, g);
  df[o] = gf;
}

// Cloud::add (cloud.cpp:145-171) of every frame cloud of the set, in frame order, behind *run points: point record and
// gaussian of point i of frame f moved by pose f (k_cloud_append, k_gauss_append).  A set that does not fit below
// dstCapacity writes nothing; *run advances regardless (k_local_map_advance), so the final count is the size the map needs.
__global__ void __launch_bounds__(256) k_local_map_append(LocalMapSet S, int m, const long long *__restrict__ run,
                                                          int dstCapacity, float4 *__restrict__ dp, float4 *__restrict__ dn,
                                                          float4 *__restrict__ dom, float *__restrict__ dg,
                                                          int *__restrict__ df) {
  const int f = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = __ldg(S.count[f]);
  if (i >= n) return;
  long long before = 0, total = 0;
  for (int k = 0; k < m; k++) {
    const int nk = __ldg(S.count[k]);
    if (k < f) before += nk;
    total += nk;
  }
  const long long base = __ldg(run);
  if (base + total > dstCapacity) return;
  append_point(S.points[f], S.normals[f], S.omega[f], S.gauss[f], S.gflags[f], i, S.pose[f], S.poseIdentity[f], dp, dn, dom,
               dg, df, (size_t)(base + before + i));
}
__global__ void k_local_map_advance(LocalMapSet S, int m, long long *run) {
  long long total = 0;
  for (int k = 0; k < m; k++) total += *S.count[k];
  *run += total;
}
__global__ void k_local_map_begin(long long *run, const int *mapN) { *run = *mapN; }
__global__ void k_local_map_commit(int *mapN, const long long *run) { *mapN = (int)*run; }

int launch_local_map_begin(nicp_context *ctx, nicp_cloud *map, long long *d_run) {
  if (!map->has_gauss) {  // points the map already holds get default (all-zero) gaussians, as in launch_gauss_append
    int rc = cloud_ensure_gaussians(ctx, map);
    if (rc) return rc;
    NICP_CUDA(cudaMemsetAsync(map->gauss, 0, sizeof(float) * kGF * (size_t)map->capacity, ctx->stream));
    NICP_CUDA(cudaMemsetAsync(map->gflags, 0, sizeof(int) * (size_t)map->capacity, ctx->stream));
  }
  k_local_map_begin<<<1, 1, 0, ctx->stream>>>(d_run, map->d_n);
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

// the m frame clouds of the launch set that launch_raw_prep_batch has just queued (its depth and integral images are still
// in the batch scratch): gaussians, then one append launch behind *d_run.  baseline, alpha: one per camera of fs.
int launch_local_map_set(nicp_context *ctx, const FrameSet &fs, int m, nicp_cloud *const *frames, const float *poses,
                         const float *baseline, const float *alpha, const float sensorOffset[16], nicp_cloud *map,
                         long long *d_run) {
  const int P = fs.proj.rows * fs.proj.cols;
  int rc;
  if ((rc = launch_set_gaussians(ctx, fs, m, frames, baseline, alpha, sensorOffset))) return rc;
  LocalMapSet S;
  memset(&S, 0, sizeof S);
  for (int f = 0; f < m; f++) {
    S.points[f] = frames[f]->points;
    S.normals[f] = frames[f]->normals;
    S.omega[f] = frames[f]->omega;
    S.gauss[f] = frames[f]->gauss;
    S.gflags[f] = frames[f]->gflags;
    S.count[f] = frames[f]->d_n;
    float T[16];
    for (int k = 0; k < 16; k++) T[k] = poses[16 * f + k];
    fix_last_row(T);
    S.pose[f] = affine_from(T);
    S.poseIdentity[f] = is_identity16(T) ? 1 : 0;
  }
  k_local_map_append<<<dim3((P + 255) / 256, m), 256, 0, ctx->stream>>>(S, m, d_run, map->capacity, map->points, map->normals,
                                                                        map->omega, map->gauss, map->gflags);
  NICP_CHECK_LAUNCH(ctx);
  k_local_map_advance<<<1, 1, 0, ctx->stream>>>(S, m, d_run);
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

// the gaussians of the m frame clouds of the launch set that launch_raw_prep_batch has just queued, from its depth and
// integral images in the batch scratch.  baseline, alpha: one per camera of fs.
int launch_set_gaussians(nicp_context *ctx, const FrameSet &fs, int m, nicp_cloud *const *frames, const float *baseline,
                         const float *alpha, const float sensorOffset[16]) {
  const nicp_projector *proj = &fs.proj;
  const int P = proj->rows * proj->cols;
  LocalMapSet S;
  memset(&S, 0, sizeof S);
  for (int f = 0; f < m; f++) {
    int rc = cloud_ensure_gaussians(ctx, frames[f]);
    if (rc) return rc;
    S.gauss[f] = frames[f]->gauss;
    S.gflags[f] = frames[f]->gflags;
    frames[f]->has_gauss = true;
  }
  float M[16];
  for (int k = 0; k < 16; k++) M[k] = sensorOffset[k];
  fix_last_row(M);
  S.offset = affine_from(M);
  S.offsetIdentity = is_identity16(M) ? 1 : 0;
  if (fs.cams.multi) {
    k_local_map_rig_gaussians<<<dim3((P + 127) / 128, m), 128, 0, ctx->stream>>>(
        S, ctx->d_bDepth, ctx->d_bIntegral, ctx->batchPixels, proj->rows, proj->cols, rig_sensor(fs.cams, baseline, alpha));
  } else {
    const SensorModel sm = sensor_model(proj, baseline[0]);
    k_local_map_gaussians<<<dim3((P + 127) / 128, m), 128, 0, ctx->stream>>>(S, ctx->d_bDepth, ctx->d_bIntegral,
                                                                            ctx->batchPixels, proj->rows, proj->cols,
                                                                            proj->min_distance, proj->max_distance, sm.iK,
                                                                            sm.iKRt, sm.fB, alpha[0]);
  }
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

// Frames appended to their own maps in one launch (frame f = blockIdx.y of k_scene_append): source cloud, destination
// cloud and the pose the frame is appended with.  A kernel parameter (about 150 B per frame).
constexpr int kSceneAppendFrames = 64;
struct SceneAppendSet {
  const float4 *points[kSceneAppendFrames], *normals[kSceneAppendFrames], *omega[kSceneAppendFrames];
  const float *gauss[kSceneAppendFrames];
  const int *gflags[kSceneAppendFrames], *count[kSceneAppendFrames];
  float4 *dp[kSceneAppendFrames], *dn[kSceneAppendFrames], *dom[kSceneAppendFrames];
  float *dg[kSceneAppendFrames];
  int *df[kSceneAppendFrames], *dstN[kSceneAppendFrames];
  int dstCapacity[kSceneAppendFrames];
  Affine pose[kSceneAppendFrames];
  int poseIdentity[kSceneAppendFrames];
};

// Cloud::add (cloud.cpp:145-171) of m frames, each to its own map: point record and gaussian of point i of frame f moved
// by pose f (append_point) and written behind *dstN[f] points.  The caller has checked that every
// frame fits; a frame that would not fit writes nothing.  The counts advance in k_scene_append_advance.
__global__ void __launch_bounds__(256) k_scene_append(SceneAppendSet S) {
  const int f = blockIdx.y;
  const int n = *S.count[f];
  const long long base = *S.dstN[f];
  if (base + n > S.dstCapacity[f]) return;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    append_point(S.points[f], S.normals[f], S.omega[f], S.gauss[f], S.gflags[f], i, S.pose[f], S.poseIdentity[f], S.dp[f],
                 S.dn[f], S.dom[f], S.dg[f], S.df[f], (size_t)(base + i));
}
__global__ void k_scene_append_advance(SceneAppendSet S, int m) {
  const int f = threadIdx.x;
  if (f >= m) return;
  const int n = *S.count[f];
  if ((long long)*S.dstN[f] + n <= S.dstCapacity[f]) *S.dstN[f] += n;
}

// nicp_cloud_append(maps[k], frames[k], poses + 16 k) for n frames with gaussians and distinct maps that carry gaussians,
// one launch per kSceneAppendFrames frames.  framePoints / mapPoints: the host's counts, which the caller has checked to
// fit; they size the grid and the maps' host mirrors (the kernel reads the counts on the device).
int launch_scene_append(nicp_context *ctx, int n, nicp_cloud *const *frames, nicp_cloud *const *maps, const float *poses,
                        const int *framePoints, const int *mapPoints) {
  for (int base = 0; base < n; base += kSceneAppendFrames) {
    const int m = std::min(kSceneAppendFrames, n - base);
    SceneAppendSet S;
    memset(&S, 0, sizeof S);
    int maxPoints = 0;
    for (int f = 0; f < m; f++) {
      const int k = base + f;
      const nicp_cloud *src = frames[k];
      nicp_cloud *dst = maps[k];
      S.points[f] = src->points;
      S.normals[f] = src->normals;
      S.omega[f] = src->omega;
      S.gauss[f] = src->gauss;
      S.gflags[f] = src->gflags;
      S.count[f] = src->d_n;
      S.dp[f] = dst->points;
      S.dn[f] = dst->normals;
      S.dom[f] = dst->omega;
      S.dg[f] = dst->gauss;
      S.df[f] = dst->gflags;
      S.dstN[f] = dst->d_n;
      S.dstCapacity[f] = dst->capacity;
      float T[16];
      for (int i = 0; i < 16; i++) T[i] = poses[16 * (size_t)k + i];
      fix_last_row(T);
      S.pose[f] = affine_from(T);
      S.poseIdentity[f] = is_identity16(T) ? 1 : 0;
      maxPoints = std::max(maxPoints, framePoints[k]);
    }
    k_scene_append<<<dim3(std::max(1, (maxPoints + 255) / 256), m), 256, 0, ctx->stream>>>(S);
    NICP_CHECK_LAUNCH(ctx);
    k_scene_append_advance<<<1, kSceneAppendFrames, 0, ctx->stream>>>(S, m);
    NICP_CHECK_LAUNCH(ctx);
  }
  for (int k = 0; k < n; k++) {  // like launch_local_map_commit
    nicp_cloud *map = maps[k];
    map->points3_valid = false; map->pn_valid = false;
    map->has_stats = false;
    map->has_gauss = true;
    map->n_host = mapPoints[k] + framePoints[k];
    map->n_known = true;
  }
  return NICP_OK;
}

// the map takes the appended points: count from the device, flags and caches like nicp_cloud_append
int launch_local_map_commit(nicp_context *ctx, nicp_cloud *map, const long long *d_run, int newSize) {
  k_local_map_commit<<<1, 1, 0, ctx->stream>>>(map->d_n, d_run);
  NICP_CHECK_LAUNCH(ctx);
  map->points3_valid = false; map->pn_valid = false;
  map->has_stats = false;
  map->has_gauss = true;
  map->n_host = newSize;
  map->n_known = true;
  return NICP_OK;
}

// ---------------------------------------------------------------------------------------------
// generic row gathers (compaction / reordering of the per-point arrays)
// ---------------------------------------------------------------------------------------------
__global__ void k_gather_vec(const float4 *__restrict__ src, float4 *__restrict__ dst, const int *__restrict__ map,
                             const int *__restrict__ mPtr, int vecPerRow) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t j = t / vecPerRow;
  const int v = (int)(t - j * vecPerRow);
  if (j >= (size_t)*mPtr) return;
  dst[j * vecPerRow + v] = src[(size_t)map[j] * vecPerRow + v];
}
__global__ void k_gather_int(const int *__restrict__ src, int *__restrict__ dst, const int *__restrict__ map,
                             const int *__restrict__ mPtr) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= *mPtr) return;
  dst[j] = src[map[j]];
}
__global__ void k_gather_f3(const float *__restrict__ src, float *__restrict__ dst, const int *__restrict__ map,
                            const int *__restrict__ mPtr) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= *mPtr) return;
  const size_t s = 3 * (size_t)map[j];
  dst[3 * (size_t)j] = src[s];
  dst[3 * (size_t)j + 1] = src[s + 1];
  dst[3 * (size_t)j + 2] = src[s + 2];
}
__global__ void k_set_count(int *dst, const int *src) { *dst = *src; }

// reorders every per-point array of the cloud so that new[j] = old[map[j]], j < *d_m (n = upper bound of *d_m)
static int reorder_cloud(nicp_context *ctx, nicp_cloud *cloud, const int *d_map, const int *d_m, int n, void *tmp) {
  cloud->points3_valid = false; cloud->pn_valid = false;
  cudaStream_t st = ctx->stream;
  auto vec = [&](float4 *arr, int vecPerRow) -> int {
    const size_t threads = (size_t)n * vecPerRow;
    k_gather_vec<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(arr, static_cast<float4 *>(tmp), d_map, d_m, vecPerRow);
    NICP_CHECK_LAUNCH(ctx);
    NICP_CUDA(cudaMemcpyAsync(arr, tmp, sizeof(float4) * threads, cudaMemcpyDeviceToDevice, st));
    return NICP_OK;
  };
  int rc;
  if ((rc = vec(cloud->points, 1)) || (rc = vec(cloud->normals, 1)) || (rc = vec(cloud->omega, 3))) return rc;
  if (cloud->has_stats) {
    if ((rc = vec(reinterpret_cast<float4 *>(cloud->stats16), 4))) return rc;
    k_gather_f3<<<(n + 255) / 256, 256, 0, st>>>(cloud->eigvals, static_cast<float *>(tmp), d_map, d_m);
    NICP_CHECK_LAUNCH(ctx);
    NICP_CUDA(cudaMemcpyAsync(cloud->eigvals, tmp, sizeof(float) * 3 * n, cudaMemcpyDeviceToDevice, st));
    k_gather_int<<<(n + 255) / 256, 256, 0, st>>>(cloud->statsN, static_cast<int *>(tmp), d_map, d_m);
    NICP_CHECK_LAUNCH(ctx);
    NICP_CUDA(cudaMemcpyAsync(cloud->statsN, tmp, sizeof(int) * n, cudaMemcpyDeviceToDevice, st));
  }
  if (cloud->has_gauss) {
    if ((rc = vec(reinterpret_cast<float4 *>(cloud->gauss), kGF / 4))) return rc;
    k_gather_int<<<(n + 255) / 256, 256, 0, st>>>(cloud->gflags, static_cast<int *>(tmp), d_map, d_m);
    NICP_CHECK_LAUNCH(ctx);
    NICP_CUDA(cudaMemcpyAsync(cloud->gflags, tmp, sizeof(int) * n, cudaMemcpyDeviceToDevice, st));
  }
  k_set_count<<<1, 1, 0, st>>>(cloud->d_n, d_m);
  NICP_CHECK_LAUNCH(ctx);
  cloud->n_known = false;
  return NICP_OK;
}
static size_t reorder_tmp_bytes(const nicp_cloud *cloud, int n) {
  size_t row = 48;                                  // omega
  if (cloud->has_stats) row = 64;
  if (cloud->has_gauss) row = sizeof(float) * kGF;  // 96
  return pad256(row * (size_t)n);
}

// ---------------------------------------------------------------------------------------------
// Merger::merge (merger.cpp:15-119)
// ---------------------------------------------------------------------------------------------
// first loop, classification part (merger.cpp:44-79): collapsed[i] = i (the point is the z-buffer winner of its
// pixel), the winner's index (the point will be fused into it) or -1 (kept as it is)
__global__ void k_merge_classify(const float4 *__restrict__ points, const float4 *__restrict__ normals, int n, Affine KRt,
                                 int rows, int cols, float minD, float maxD, float distanceThreshold, float normalThreshold,
                                 float maxPointDepth, const unsigned long long *__restrict__ z, int *__restrict__ collapsed,
                                 int *__restrict__ count) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int res = -1;
  const float4 p = points[i];
  float ix, iy, depth;
  xform_point(KRt, p.x, p.y, p.z, ix, iy, depth);
  int r = -1, c = -1;
  if (!(depth < minD || depth > maxD)) {  // _project, pinholepointprojector.h:224-233
    const float s = frcp(depth);
    c = (int)roundf(fmul(ix, s));
    r = (int)roundf(fmul(iy, s));
  }
  if (!(depth < 0.0f || depth > maxPointDepth || r < 0 || r >= rows || c < 0 || c >= cols)) {
    const unsigned long long w = z[(size_t)r * cols + c];
    const int target = z_index(w, kEpochFresh);
    if (target >= 0) {
      if (target == i) {
        res = i;
      } else {
        const float targetZ = z_depth(w, kEpochFresh, FLT_MAX);
        const float4 cn = normals[i], tn = normals[target];
        if (fabsf(fsub(depth, targetZ)) < distanceThreshold &&
            dot3(cn.x, cn.y, cn.z, tn.x, tn.y, tn.z) > normalThreshold) {
          res = target;
          atomicAdd(&count[target], 1);
        }
      }
    }
  }
  collapsed[i] = res;
}
__global__ void k_merge_fill(const int *__restrict__ collapsed, int n, const int *__restrict__ offset, int *__restrict__ cursor,
                             int *__restrict__ list) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int t = collapsed[i];
  if (t < 0 || t == i) return;
  list[offset[t] + atomicAdd(&cursor[t], 1)] = i;
}
// Gaussian::addInformation in the reference's order (ascending contributor index), merger.cpp:73-76
__global__ void k_merge_accumulate(int n, const int *__restrict__ count, const int *__restrict__ offset, int *__restrict__ list,
                                   float *__restrict__ gauss, int *__restrict__ gflags) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int m = count[t];
  if (m <= 0) return;
  int *L = list + offset[t];
  for (int a = 1; a < m; a++) {  // insertion sort: the lists are a handful of entries long
    const int v = L[a];
    int b = a - 1;
    while (b >= 0 && L[b] > v) { L[b + 1] = L[b]; b--; }
    L[b + 1] = v;
  }
  float g[kGF];
  gauss_load(gauss + (size_t)kGF * t, g);
  int f = gflags[t];
  gauss_update_info(g, f);
  for (int a = 0; a < m; a++) {
    float cg[kGF];
    gauss_load(gauss + (size_t)kGF * L[a], cg);
    int cf = gflags[L[a]];
    gauss_update_info(cg, cf);
    for (int k = 0; k < 9; k++) g[15 + k] = fadd(g[15 + k], cg[15 + k]);
    for (int k = 0; k < 3; k++) g[12 + k] = fadd(g[12 + k], cg[12 + k]);
  }
  f &= ~NICP_GAUSS_MOMENTS;
  gauss_store(gauss + (size_t)kGF * t, g);
  gflags[t] = f;
}
// second loop (merger.cpp:90-107): winners take the mean of their gaussian; keep flag for the compaction
__global__ void k_merge_finalize(int n, const int *__restrict__ collapsed, float4 *__restrict__ points, float *__restrict__ gauss,
                                 int *__restrict__ gflags, int *__restrict__ keep) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int c = collapsed[i];
  if (c == i) {
    int f = gflags[i];
    if (!(f & NICP_GAUSS_MOMENTS)) {
      float g[kGF];
      gauss_load(gauss + (size_t)kGF * i, g);
      gauss_update_moments(g, f);
      gauss_store(gauss + (size_t)kGF * i, g);
      gflags[i] = f;
    }
    const float *g = gauss + (size_t)kGF * i;
    points[i] = make_float4(g[0], g[1], g[2], points[i].w);
  }
  keep[i] = (c < 0 || c == i) ? 1 : 0;
}
__global__ void k_compact_map(const int *__restrict__ keep, const int *__restrict__ pos, int n, int *__restrict__ map) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (keep[i]) map[pos[i]] = i;
}

int run_merge(nicp_context *ctx, nicp_cloud *cloud, const nicp_projector *proj, const float transform[16],
              const nicp_merge_params *mp, int n, int *collapsedHost, int *newSize) {
  cudaStream_t st = ctx->stream;
  const int P = proj->rows * proj->cols;
  const size_t scanInts = scan_scratch_ints(n);
  Bump b;
  const size_t need = pad256(sizeof(unsigned long long) * P) + 7 * pad256(sizeof(int) * n) + pad256(sizeof(int) * scanInts) +
                      reorder_tmp_bytes(cloud, n) + 2048;
  int rc;
  if ((rc = map_scratch(ctx, need, &b))) return rc;
  unsigned long long *d_z = b.take<unsigned long long>(P);
  int *d_collapsed = b.take<int>(n), *d_count = b.take<int>(n), *d_offset = b.take<int>(n), *d_cursor = b.take<int>(n);
  int *d_list = b.take<int>(n), *d_keep = b.take<int>(n), *d_pos = b.take<int>(n);
  int *d_scan = b.take<int>(scanInts), *d_total = b.take<int>(1);
  void *d_tmp = b.take<unsigned char>(reorder_tmp_bytes(cloud, n));
  if (!d_tmp) { set_error("nicp_merge: scratch accounting error"); return NICP_ERR_INVALID; }
  float KRt[16];
  compute_KRt(proj->K, transform, KRt);
  if ((rc = launch_project_single(ctx, cloud, KRt, proj->rows, proj->cols, proj->min_distance, proj->max_distance, d_z)))
    return rc;
  NICP_CUDA(cudaMemsetAsync(d_count, 0, sizeof(int) * n, st));
  NICP_CUDA(cudaMemsetAsync(d_cursor, 0, sizeof(int) * n, st));
  const int nb = (n + 255) / 256;
  k_merge_classify<<<nb, 256, 0, st>>>(cloud->points, cloud->normals, n, affine_from(KRt), proj->rows, proj->cols,
                                       proj->min_distance, proj->max_distance, mp->distance_threshold, mp->normal_threshold,
                                       mp->max_point_depth, d_z, d_collapsed, d_count);
  NICP_CHECK_LAUNCH(ctx);
  if ((rc = exclusive_scan(ctx, d_count, d_offset, n, d_scan, nullptr))) return rc;
  k_merge_fill<<<nb, 256, 0, st>>>(d_collapsed, n, d_offset, d_cursor, d_list);
  NICP_CHECK_LAUNCH(ctx);
  k_merge_accumulate<<<(n + 127) / 128, 128, 0, st>>>(n, d_count, d_offset, d_list, cloud->gauss, cloud->gflags);
  NICP_CHECK_LAUNCH(ctx);
  cloud->points3_valid = false; cloud->pn_valid = false;
  k_merge_finalize<<<nb, 256, 0, st>>>(n, d_collapsed, cloud->points, cloud->gauss, cloud->gflags, d_keep);
  NICP_CHECK_LAUNCH(ctx);
  if ((rc = exclusive_scan(ctx, d_keep, d_pos, n, d_scan, d_total))) return rc;
  k_compact_map<<<nb, 256, 0, st>>>(d_keep, d_pos, n, d_list);  // d_list is free again: it becomes the gather map
  NICP_CHECK_LAUNCH(ctx);
  if (collapsedHost) NICP_CUDA(cudaMemcpyAsync(collapsedHost, d_collapsed, sizeof(int) * n, cudaMemcpyDeviceToHost, st));
  if ((rc = reorder_cloud(ctx, cloud, d_list, d_total, n, d_tmp))) return rc;
  int total = 0;
  NICP_CUDA(cudaMemcpyAsync(&total, d_total, sizeof(int), cudaMemcpyDeviceToHost, st));
  NICP_CUDA(cudaStreamSynchronize(st));
  cloud->n_host = total;
  cloud->n_known = true;
  if (newSize) *newSize = total;
  return NICP_OK;
}

// ---------------------------------------------------------------------------------------------
// VoxelCalculator::compute (voxelcalculator.cpp:15-73)
// ---------------------------------------------------------------------------------------------
__global__ void k_voxel_coords(const float4 *__restrict__ points, int n, float inverseResolution, int3 *__restrict__ coords,
                               int *__restrict__ lohi /* min x,y,z then max x,y,z */) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int3 v = make_int3(0, 0, 0);
  const bool ok = i < n;
  if (ok) {
    const float4 p = points[i];
    v.x = __float2int_rz(fmul(p.x, inverseResolution));
    v.y = __float2int_rz(fmul(p.y, inverseResolution));
    v.z = __float2int_rz(fmul(p.z, inverseResolution));
    coords[i] = v;
  }
  int lo[3] = {ok ? v.x : INT_MAX, ok ? v.y : INT_MAX, ok ? v.z : INT_MAX};
  int hi[3] = {ok ? v.x : INT_MIN, ok ? v.y : INT_MIN, ok ? v.z : INT_MIN};
#pragma unroll
  for (int a = 0; a < 3; a++) {
    lo[a] = __reduce_min_sync(0xffffffffu, lo[a]);
    hi[a] = __reduce_max_sync(0xffffffffu, hi[a]);
  }
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int a = 0; a < 3; a++) {
      atomicMin(&lohi[a], lo[a]);
      atomicMax(&lohi[3 + a], hi[a]);
    }
  }
}
__global__ void k_voxel_pack(const int3 *__restrict__ coords, int n, int3 lo, int shiftX, int shiftY,
                             unsigned long long *__restrict__ keys, int *__restrict__ vals) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int3 v = coords[i];
  keys[i] = ((unsigned long long)(unsigned int)(v.x - lo.x) << shiftX) | ((unsigned long long)(unsigned int)(v.y - lo.y) << shiftY) |
            (unsigned long long)(unsigned int)(v.z - lo.z);
  vals[i] = i;
}
// stable LSD radix sort, 8 bits per pass.  A tile of kSortTile consecutive items belongs to one CTA in both
// kernels; the scatter walks its tile in order with one warp, ranking equal digits with match_any.
constexpr int kSortTile = 2048;
__global__ void __launch_bounds__(256) k_sort_hist(const unsigned long long *__restrict__ keys, int n, int shift, int numTiles,
                                                   int *__restrict__ hist /* [256][numTiles] */) {
  __shared__ int h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const int base = blockIdx.x * kSortTile;
  for (int k = threadIdx.x; k < kSortTile; k += 256)
    if (base + k < n) atomicAdd(&h[(int)((keys[base + k] >> shift) & 255ull)], 1);
  __syncthreads();
  hist[threadIdx.x * numTiles + blockIdx.x] = h[threadIdx.x];
}
__global__ void __launch_bounds__(32) k_sort_scatter(const unsigned long long *__restrict__ keysIn, const int *__restrict__ valsIn,
                                                     int n, int shift, int numTiles, const int *__restrict__ offsets,
                                                     unsigned long long *__restrict__ keysOut, int *__restrict__ valsOut) {
  __shared__ int cursor[256];
  const int lane = threadIdx.x;
  for (int d = lane; d < 256; d += 32) cursor[d] = offsets[d * numTiles + blockIdx.x];
  __syncwarp();
  const int base = blockIdx.x * kSortTile;
  for (int k = 0; k < kSortTile; k += 32) {
    const int i = base + k + lane;
    const bool ok = i < n;
    unsigned long long key = 0;
    int val = 0, digit = 256 + lane;  // idle lanes get digits of their own
    if (ok) {
      key = keysIn[i];
      val = valsIn[i];
      digit = (int)((key >> shift) & 255ull);
    }
    const unsigned int peers = __match_any_sync(0xffffffffu, digit);
    const int rank = __popc(peers & ((1u << lane) - 1u));
    int pos = 0;
    if (ok) pos = cursor[digit] + rank;
    __syncwarp();
    if (ok && rank == 0) cursor[digit] += __popc(peers);
    __syncwarp();
    if (ok) {
      keysOut[pos] = key;
      valsOut[pos] = val;
    }
    if (base + k + 32 >= n) break;
  }
}
__global__ void k_voxel_heads(const unsigned long long *__restrict__ keys, int n, int *__restrict__ head) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  head[j] = (j == 0 || keys[j] != keys[j - 1]) ? 1 : 0;
}
__global__ void k_voxel_reps(const int *__restrict__ head, const int *__restrict__ pos, const int *__restrict__ vals, int n,
                             int *__restrict__ rep) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  if (head[j]) rep[pos[j]] = vals[j];
}
static int bits_for(unsigned int range) {
  int b = 0;
  while (range) { b++; range >>= 1; }
  return b;
}

int run_voxelize(nicp_context *ctx, nicp_cloud *cloud, float resolution, int n, int *repHost, int *newSize) {
  cudaStream_t st = ctx->stream;
  const int numTiles = (n + kSortTile - 1) / kSortTile;
  const size_t histInts = 256 * (size_t)numTiles;
  const size_t scanInts = scan_scratch_ints((int)(histInts > (size_t)n ? histInts : (size_t)n));
  Bump b;
  const size_t need = pad256(sizeof(int3) * n) + 2 * pad256(sizeof(unsigned long long) * n) + 5 * pad256(sizeof(int) * n) +
                      2 * pad256(sizeof(int) * histInts) + pad256(sizeof(int) * scanInts) + reorder_tmp_bytes(cloud, n) + 4096;
  int rc;
  if ((rc = map_scratch(ctx, need, &b))) return rc;
  int3 *d_coords = b.take<int3>(n);
  unsigned long long *d_keys[2] = {b.take<unsigned long long>(n), b.take<unsigned long long>(n)};
  int *d_vals[2] = {b.take<int>(n), b.take<int>(n)};
  int *d_head = b.take<int>(n), *d_pos = b.take<int>(n), *d_rep = b.take<int>(n);
  int *d_hist = b.take<int>(histInts), *d_histScan = b.take<int>(histInts), *d_scan = b.take<int>(scanInts);
  int *d_lohi = b.take<int>(8), *d_total = b.take<int>(1);
  void *d_tmp = b.take<unsigned char>(reorder_tmp_bytes(cloud, n));
  if (!d_tmp) { set_error("nicp_voxelize: scratch accounting error"); return NICP_ERR_INVALID; }
  const int init[6] = {INT_MAX, INT_MAX, INT_MAX, INT_MIN, INT_MIN, INT_MIN};
  NICP_CUDA(cudaMemcpyAsync(d_lohi, init, sizeof init, cudaMemcpyHostToDevice, st));
  const int nb = (n + 255) / 256;
  k_voxel_coords<<<nb, 256, 0, st>>>(cloud->points, n, fdiv(1.0f, resolution), d_coords, d_lohi);
  NICP_CHECK_LAUNCH(ctx);
  int lohi[6];
  NICP_CUDA(cudaMemcpyAsync(lohi, d_lohi, sizeof lohi, cudaMemcpyDeviceToHost, st));
  NICP_CUDA(cudaStreamSynchronize(st));
  int bits[3];
  for (int a = 0; a < 3; a++) bits[a] = bits_for((unsigned int)((long long)lohi[3 + a] - (long long)lohi[a]));
  const int totalBits = bits[0] + bits[1] + bits[2];
  if (totalBits > 64) {
    set_error("nicp_voxelize: the voxel grid needs %d key bits (more than 64); use a coarser resolution", totalBits);
    return NICP_ERR_INVALID;
  }
  k_voxel_pack<<<nb, 256, 0, st>>>(d_coords, n, make_int3(lohi[0], lohi[1], lohi[2]), bits[1] + bits[2], bits[2], d_keys[0],
                                   d_vals[0]);
  NICP_CHECK_LAUNCH(ctx);
  int cur = 0;
  for (int shift = 0; shift < totalBits; shift += 8) {
    k_sort_hist<<<numTiles, 256, 0, st>>>(d_keys[cur], n, shift, numTiles, d_hist);
    NICP_CHECK_LAUNCH(ctx);
    if ((rc = exclusive_scan(ctx, d_hist, d_histScan, (int)histInts, d_scan, nullptr))) return rc;
    k_sort_scatter<<<numTiles, 32, 0, st>>>(d_keys[cur], d_vals[cur], n, shift, numTiles, d_histScan, d_keys[cur ^ 1],
                                           d_vals[cur ^ 1]);
    NICP_CHECK_LAUNCH(ctx);
    cur ^= 1;
  }
  k_voxel_heads<<<nb, 256, 0, st>>>(d_keys[cur], n, d_head);
  NICP_CHECK_LAUNCH(ctx);
  if ((rc = exclusive_scan(ctx, d_head, d_pos, n, d_scan, d_total))) return rc;
  k_voxel_reps<<<nb, 256, 0, st>>>(d_head, d_pos, d_vals[cur], n, d_rep);
  NICP_CHECK_LAUNCH(ctx);
  int total = 0;
  NICP_CUDA(cudaMemcpyAsync(&total, d_total, sizeof(int), cudaMemcpyDeviceToHost, st));
  NICP_CUDA(cudaStreamSynchronize(st));
  if (repHost) NICP_CUDA(cudaMemcpyAsync(repHost, d_rep, sizeof(int) * total, cudaMemcpyDeviceToHost, st));
  if ((rc = reorder_cloud(ctx, cloud, d_rep, d_total, n, d_tmp))) return rc;
  NICP_CUDA(cudaStreamSynchronize(st));
  cloud->n_host = total;
  cloud->n_known = true;
  if (newSize) *newSize = total;
  return NICP_OK;
}

}  // namespace nicp

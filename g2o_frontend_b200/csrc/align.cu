// align.cu -- the NICP alignment loop on the device.
//
// Replaces, for a batch of independent (reference, current) cloud pairs processed in lock step:
//   PinholePointProjector::project      pinholepointprojector.cpp:33-66   -> k_project
//   CorrespondenceFinder::compute       correspondencefinder.cpp:20-118  \  k_corr_lin_group<0> / k_corr_lin_tiled<0> (fused,
//   Linearizer::update                  linearizer.cpp:17-115            /  corr_lin.cuh); <1>: from the stored correspondences
//   Aligner::align loop body            aligner.cpp:66-118                -> k_reduce_solve
//   PwnMatcherBase::matchClouds stats   pwn_tracker2/pwn_matcher_base.cpp:167-196 -> folded into k_corr_lin_*<1>
//
// z-buffer: one 64-bit word per pixel, (epoch | float_bits(depth * 2^-110)) << 32 | pointIndex, filled
// with atomicMin (z_encode in nicp_internal.cuh).  depth > 0 so unsigned order == float order: the
// nearest point wins and, on equal depth, the lowest point index wins -- exactly the outcome of the
// reference's sequential scatter with its strict `otherDistance > d` test.  Fresh = all ones
// (index decodes to -1); the epoch tag lets later iterations reuse a buffer without clearing it.
//
// Reduction: every thread accumulates 30 float sums over its pixels (21 unique H entries, 6 b,
// chi2, inliers, correspondences), a transposing warp butterfly leaves component j in lane j
// (31 shuffles instead of 160) and one partial row per (pair, tile) goes to global memory.
// k_reduce_solve adds the rows in fixed order, so H, b and the pose are bit-reproducible run to
// run (no float atomics anywhere).
#include "nicp_internal.cuh"
#include "nicp_stats_tail.cuh"
#include "corr_lin.cuh"

#include <algorithm>

namespace nicp {

// KRt of every camera for the projector pose `pose` (PinholePointProjector::_updateMatrices after
// MultiPointProjector::setTransform(pose): child pose = pose * offset_i, multipointprojector.cpp:207-215)
__device__ void store_cam_KRt(const CamSet *cams, const float *pose, PairState *st) {
  for (int i = 0; i < cams->n; i++) {
    float Tc[16], KRt[16];
    iso_mul(pose, cams->offset[i], Tc);
    compute_KRt(cams->K[i], Tc, KRt);
    for (int k = 0; k < 16; k++) st->KRt[i][k] = KRt[k];
  }
}

// ---------------------------------------------------------------------------------------------
__global__ void k_init_pairs(PairDesc *desc, int n, AlignConsts ac) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  PairState *st = desc[i].state;
  float T[16], tmp[16];
  for (int k = 0; k < 16; k++) T[k] = desc[i].guess[k];
  fix_last_row(T);
  for (int k = 0; k < 16; k++) st->T[k] = T[k];
  iso_inverse(T, tmp);
  for (int k = 0; k < 16; k++) st->invT[k] = tmp[k];
  iso_mul(T, ac.refOffset, tmp);
  store_cam_KRt(ac.cams, tmp, st);
  for (int k = 0; k < 36; k++) { st->H[k] = 0.f; st->statH[k] = 0.f; }
  for (int k = 0; k < 6; k++) { st->b[k] = 0.f; st->statb[k] = 0.f; }
  st->error = 0.f;
  st->inliers = 0;
  st->ncorr = 0;
  st->img_nonzeros = 0;
  st->img_inliers = 0;
  st->img_sum = 0.f;
  st->sumMidx = 0.f;
  st->sumMacc = 0.f;
  st->ticket = 0;
}

// ---------------------------------------------------------------------------------------------
// _project (pinholepointprojector.h:224-233) + the z-test of project (pinholepointprojector.cpp:52-64)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void project_point(const Affine &KRt, float4 p, int i, int rows, int cols, float minD,
                                              float maxD, unsigned long long *__restrict__ z, int epoch) {
  // straight-line code with one predicated reduction at the end (the kernel is issue bound; early returns cost
  // divergence bookkeeping).  A zero / negative / NaN depth fails the range tests below like in the reference.
  float ix, iy, d;
  xform_point(KRt, p.x, p.y, p.z, ix, iy, d);
  // the packed z-buffer word orders positive depths below 32 km (z_encode); anything else cannot be a valid range image
  bool ok = !(d < minD || d > maxD) && d > 0.0f && d < 32768.0f;
  const float s = frcp(d);
  const float fx = roundf(fmul(ix, s)), fy = roundf(fmul(iy, s));
  ok = ok && fx >= 0.0f && fx < (float)cols && fy >= 0.0f && fy < (float)rows;
  if (ok) z_min(&z[(size_t)(int)fy * cols + (int)fx], z_encode(d, i, epoch));
}

CamGeom geom_of(const CamSet &c) {
  CamGeom g;
  g.n = c.n;
  g.multi = c.multi;
  for (int i = 0; i < kMaxCams; i++) {
    g.width[i] = c.width[i]; g.height[i] = c.height[i]; g.colOff[i] = c.colOff[i];
    g.minD[i] = c.minD[i]; g.maxD[i] = c.maxD[i];
  }
  return g;
}

// MultiPointProjector::project per point (multipointprojector.cpp:157-205) under the base-class z-buffer
// (pointprojector.cpp:17-40): the first camera whose pinhole projection lands inside its
// [0,width) x [0,height) wins; composite pixel = (row u, col v + colOff).
template <typename MatSrc>
__device__ __forceinline__ void project_point_multi(const CamGeom &g, const MatSrc &mats, float4 p, int i, int rows,
                                                    int cols, unsigned long long *__restrict__ z, int epoch) {
  for (int c = 0; c < g.n; c++) {
    const Affine KRt = mats(c);
    float ix, iy, d;
    xform_point(KRt, p.x, p.y, p.z, ix, iy, d);
    if (d < g.minD[c] || d > g.maxD[c]) continue;
    float s = frcp(d);
    float fx = roundf(fmul(ix, s)), fy = roundf(fmul(iy, s));
    if (!(d > 0.0f && d < 32768.0f) || !(fx >= 0.0f && fx < (float)g.width[c] && fy >= 0.0f && fy < (float)g.height[c])) continue;
    int X = (int)fx, Y = (int)fy + g.colOff[c];
    if (X < rows && Y < cols) z_min(&z[(size_t)X * cols + Y], z_encode(d, i, epoch));
    return;
  }
}
struct MatsFromState {
  const PairState *st;
  __device__ __forceinline__ Affine operator()(int c) const { return affine_from(st->KRt[c]); }
};
struct MatsFromParam {
  const CamMats *m;
  __device__ __forceinline__ Affine operator()(int c) const { return m->M[c]; }
};

// which: 0/1 = reference cloud into refZ[which] with the pair's KRt; 2 = current cloud into curZ
// with the (shared) current-sensor KRt, only for the pair that owns that buffer.
// order (which 0/1, optional): blockIdx.y -> descriptor, pairs that project the same reference cloud adjacent, so that
// their CTAs run together and all but the first read the cloud's point stream out of L2.
__global__ void __launch_bounds__(256) k_project(const PairDesc *__restrict__ desc, int which, Affine curKRt, int rows,
                                                 int cols, float minD, float maxD, const int *__restrict__ ownsCur,
                                                 int epoch, const int *__restrict__ order) {
  const PairDesc &D = desc[order ? order[blockIdx.y] : blockIdx.y];
  const float4 *pts;
  unsigned long long *z;
  int n;
  Affine KRt;
  if (which == 2) {
    if (!ownsCur[blockIdx.y]) return;
    pts = D.curPoints;
    n = *D.curN;
    z = D.curZ;
    KRt = curKRt;
  } else {
    pts = D.refPoints;
    n = *D.refN;
    z = D.refZ[which];
    KRt = affine_from(D.state->KRt[0]);
  }
  if (which != 2 && D.refPoints3) {
    // 12-byte point stream (the kernel is DRAM bound and the w = 1 lane of the float4 points is a quarter of its read
    // traffic).  A warp takes 128 consecutive points = 96 float4, loaded fully coalesced (3 per lane), parked in shared
    // memory and read back as x,y,z of points lane, lane+32, lane+64, lane+96 (word stride 3: conflict free).
    __shared__ float4 stage[8][2][96];
    const float4 *__restrict__ q = reinterpret_cast<const float4 *>(D.refPoints3);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int chunks = (n + 127) >> 7;
    const int wstride = gridDim.x * (blockDim.x >> 5);
    for (int c = blockIdx.x * (blockDim.x >> 5) + warp; c < chunks; c += 2 * wstride) {
      const int c2 = c + wstride;
      const bool two = c2 < chunks;
      float4 a[3], b[3];
#pragma unroll
      for (int m = 0; m < 3; m++) a[m] = q[(size_t)c * 96 + lane + 32 * m];
      if (two) {
#pragma unroll
        for (int m = 0; m < 3; m++) b[m] = q[(size_t)c2 * 96 + lane + 32 * m];
      }
#pragma unroll
      for (int m = 0; m < 3; m++) stage[warp][0][lane + 32 * m] = a[m];
      if (two) {
#pragma unroll
        for (int m = 0; m < 3; m++) stage[warp][1][lane + 32 * m] = b[m];
      }
      __syncwarp();
      const float *f0 = reinterpret_cast<const float *>(stage[warp][0]);
      const float *f1 = reinterpret_cast<const float *>(stage[warp][1]);
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const int l = lane + 32 * j, i = c * 128 + l;
        if (i < n) project_point(KRt, make_float4(f0[3 * l], f0[3 * l + 1], f0[3 * l + 2], 1.0f), i, rows, cols, minD, maxD, z, epoch);
      }
      if (two) {
#pragma unroll
        for (int j = 0; j < 4; j++) {
          const int l = lane + 32 * j, i = c2 * 128 + l;
          if (i < n) project_point(KRt, make_float4(f1[3 * l], f1[3 * l + 1], f1[3 * l + 2], 1.0f), i, rows, cols, minD, maxD, z, epoch);
        }
      }
      __syncwarp();
    }
    return;
  }
  // four independent point loads in flight per thread (the loop was load -> compute -> atomic, one at a time)
  const int stride = gridDim.x * blockDim.x;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < n; i += 4 * stride) {
    const float4 p0 = pts[i], p1 = pts[i + stride], p2 = pts[i + 2 * stride], p3 = pts[i + 3 * stride];
    project_point(KRt, p0, i, rows, cols, minD, maxD, z, epoch);
    project_point(KRt, p1, i + stride, rows, cols, minD, maxD, z, epoch);
    project_point(KRt, p2, i + 2 * stride, rows, cols, minD, maxD, z, epoch);
    project_point(KRt, p3, i + 3 * stride, rows, cols, minD, maxD, z, epoch);
  }
  for (; i < n; i += stride) project_point(KRt, pts[i], i, rows, cols, minD, maxD, z, epoch);
}

// the same for a MultiPointProjector camera set
__global__ void __launch_bounds__(256) k_project_multi(const PairDesc *__restrict__ desc, int which, CamGeom g,
                                                       const CamMats *__restrict__ curMats, int rows, int cols,
                                                       const int *__restrict__ ownsCur, int epoch) {
  const PairDesc &D = desc[blockIdx.y];
  if (which == 2) {
    if (!ownsCur[blockIdx.y]) return;
    const int n = *D.curN;
    MatsFromParam mats{curMats};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
      project_point_multi(g, mats, D.curPoints[i], i, rows, cols, D.curZ, epoch);
  } else {
    const int n = *D.refN;
    MatsFromState mats{D.state};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
      project_point_multi(g, mats, D.refPoints[i], i, rows, cols, D.refZ[which], epoch);
  }
}

__global__ void __launch_bounds__(256) k_project_single(const float4 *__restrict__ pts, const int *__restrict__ nPtr,
                                                        Affine KRt, int rows, int cols, float minD, float maxD,
                                                        unsigned long long *__restrict__ z) {
  int n = *nPtr;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    project_point(KRt, pts[i], i, rows, cols, minD, maxD, z, kEpochFresh);
}

__global__ void __launch_bounds__(256) k_project_single_multi(const float4 *__restrict__ pts, const int *__restrict__ nPtr,
                                                              CamGeom g, const CamMats *__restrict__ matsPtr, int rows,
                                                              int cols, unsigned long long *__restrict__ z) {
  int n = *nPtr;
  MatsFromParam mats{matsPtr};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    project_point_multi(g, mats, pts[i], i, rows, cols, z, kEpochFresh);
}

__global__ void k_decode_z(const unsigned long long *__restrict__ z, int n, int *__restrict__ index,
                           float *__restrict__ depth, float emptyDepth, int epoch) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned long long v = z[i];
  if (index) index[i] = z_index(v, epoch);
  if (depth) depth[i] = z_depth(v, epoch, emptyDepth);
}

__global__ void k_decode_cur(const PairDesc *__restrict__ desc, int P, const int *__restrict__ ownsCur, int epoch) {
  if (!ownsCur[blockIdx.y]) return;
  const PairDesc &D = desc[blockIdx.y];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < P; i += gridDim.x * blockDim.x)
    D.curIndex[i] = z_index(D.curZ[i], epoch);
}

// x,y,z of every point packed at 12 bytes (the buffer holds capacity rounded up to 128 points, so a warp of
// k_project can always load a whole chunk)
__global__ void k_pack3(const float4 *__restrict__ pts, const int *__restrict__ nPtr, int capacity, float *__restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = min(*nPtr, capacity);
  if (i >= n) return;
  const float4 p = pts[i];
  out[3 * (size_t)i] = p.x;
  out[3 * (size_t)i + 1] = p.y;
  out[3 * (size_t)i + 2] = p.z;
}
int ensure_points3(nicp_context *ctx, nicp_cloud *cloud) {
#ifndef NICP_VERIFY_BUILD
  if (cloud->points3 && cloud->points3_valid) return NICP_OK;
#endif  // the verification build never trusts the cache: it repacks for every alignment
  if (!cloud->points3) {
    NICP_CUDA(cudaSetDevice(ctx->device));
    const size_t floats = 3 * (((size_t)cloud->capacity + 127) & ~(size_t)127);
    cudaError_t e = cudaMalloc(&cloud->points3, floats * sizeof(float));
    if (e != cudaSuccess) {
      set_error("cudaMalloc of the packed point stream (%zu bytes) failed: %s", floats * sizeof(float), cudaGetErrorString(e));
      return NICP_ERR_ALLOC;
    }
    NICP_CUDA(cudaMemsetAsync(cloud->points3, 0, floats * sizeof(float), ctx->stream));
  }
  k_pack3<<<(cloud->capacity + 255) / 256, 256, 0, ctx->stream>>>(cloud->points, cloud->d_n, cloud->capacity, cloud->points3);
  NICP_CHECK_LAUNCH(ctx);
  cloud->points3_valid = true;
  return NICP_OK;
}

// point + normal interleaved, one 32-byte sector per point: (px, nx, py, ny) (pz, nz, 1, curvature)
__global__ void k_pack_pn(const float4 *__restrict__ pts, const float4 *__restrict__ nrm, const int *__restrict__ nPtr, int capacity,
                          float4 *__restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = min(*nPtr, capacity);
  if (i >= n) return;
  const float4 p = pts[i], q = nrm[i];
  out[2 * (size_t)i] = make_float4(p.x, q.x, p.y, q.y);
  out[2 * (size_t)i + 1] = make_float4(p.z, q.z, 1.0f, q.w);
}
int ensure_pn(nicp_context *ctx, nicp_cloud *cloud) {
#ifndef NICP_VERIFY_BUILD
  if (cloud->pn && cloud->pn_valid) return NICP_OK;
#endif  // the verification build never trusts the cache
  if (!cloud->pn) {
    NICP_CUDA(cudaSetDevice(ctx->device));
    cudaError_t e = cudaMalloc(&cloud->pn, 2 * (size_t)cloud->capacity * sizeof(float4));
    if (e != cudaSuccess) {
      set_error("cudaMalloc of the interleaved point/normal cache (%zu bytes) failed: %s", 2 * (size_t)cloud->capacity * sizeof(float4),
                cudaGetErrorString(e));
      return NICP_ERR_ALLOC;
    }
  }
  k_pack_pn<<<(cloud->capacity + 255) / 256, 256, 0, ctx->stream>>>(cloud->points, cloud->normals, cloud->d_n, cloud->capacity, cloud->pn);
  NICP_CHECK_LAUNCH(ctx);
  cloud->pn_valid = true;
  return NICP_OK;
}

int launch_project_single(nicp_context *ctx, const nicp_cloud *cloud, const float KRt[16], int rows, int cols,
                          float minD, float maxD, unsigned long long *d_z) {
  NICP_CUDA(cudaMemsetAsync(d_z, 0xFF, (size_t)rows * cols * sizeof(unsigned long long), ctx->stream));
  int blocks = (cloud->capacity + 255) / 256;
  if (blocks < 1) blocks = 1;
  k_project_single<<<blocks, 256, 0, ctx->stream>>>(cloud->points, cloud->d_n, affine_from(KRt), rows, cols, minD, maxD,
                                                    d_z);
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

// host: per-camera KRt for the projector pose T
void cam_mats_KRt(const CamSet &cams, const float T[16], CamMats &out) {
  for (int i = 0; i < cams.n; i++) {
    float Tc[16], KRt[16];
    iso_mul(T, cams.offset[i], Tc);
    compute_KRt(cams.K[i], Tc, KRt);
    out.M[i] = affine_from(KRt);
  }
}

static int upload_cam_mats(nicp_context *ctx, const CamMats &m, CamMats **d_out) {
  CamMats *d = &ctx->d_cams->curMats;
  NICP_CUDA(cudaMemcpyAsync(d, &m, sizeof(CamMats), cudaMemcpyHostToDevice, ctx->stream));
  *d_out = d;
  return NICP_OK;
}

int launch_project_cams(nicp_context *ctx, const nicp_cloud *cloud, const CamSet &cams, const float T[16], int rows,
                        int cols, unsigned long long *d_z) {
  NICP_CUDA(cudaMemsetAsync(d_z, 0xFF, (size_t)rows * cols * sizeof(unsigned long long), ctx->stream));
  CamMats m, *d_m = nullptr;
  cam_mats_KRt(cams, T, m);
  int rc = upload_cam_mats(ctx, m, &d_m);
  if (rc) return rc;
  int blocks = (cloud->capacity + 255) / 256;
  if (blocks < 1) blocks = 1;
  k_project_single_multi<<<blocks, 256, 0, ctx->stream>>>(cloud->points, cloud->d_n, geom_of(cams), d_m, rows, cols, d_z);
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

int launch_decode_z(nicp_context *ctx, const unsigned long long *d_z, int n, int *d_index, float *d_depth, float emptyDepth,
                    int epoch) {
  k_decode_z<<<(n + 255) / 256, 256, 0, ctx->stream>>>(d_z, n, d_index, d_depth, emptyDepth, epoch);
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

// nicp_project of the maps of a launch set (map f = blockIdx.y), each with its own KRt, into z-buffers zStride words apart;
// then their depth images (FLT_MAX where empty) into depth slots depthStride floats apart.  The z pass is k_project_single's
// (project_point: nearest wins, lowest index wins ties), so each depth image is nicp_project's bit for bit.
__global__ void __launch_bounds__(256) k_render_maps_z(MapRenderSet R, int rows, int cols, float minD, float maxD,
                                                       unsigned long long *__restrict__ z0, size_t zStride) {
  const int f = blockIdx.y;
  const int n = *R.count[f];
  const float4 *__restrict__ pts = R.points[f];
  unsigned long long *z = z0 + (size_t)f * zStride;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    project_point(R.KRt[f], pts[i], i, rows, cols, minD, maxD, z, kEpochFresh);
}
__global__ void k_render_maps_depth(const unsigned long long *__restrict__ z0, size_t zStride, int P, float *__restrict__ depth0,
                                    size_t depthStride) {
  const int f = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  depth0[(size_t)f * depthStride + i] = z_depth(z0[(size_t)f * zStride + i], kEpochFresh, FLT_MAX);
}

int launch_render_maps(nicp_context *ctx, const MapRenderSet &R, int m, int maxPoints, const nicp_projector *proj,
                       unsigned long long *d_z, size_t zStride, float *d_depth, size_t depthStride) {
  const int P = proj->rows * proj->cols;
  for (int f = 0; f < m; f++)
    NICP_CUDA(cudaMemsetAsync(d_z + (size_t)f * zStride, 0xFF, (size_t)P * sizeof(unsigned long long), ctx->stream));
  // grid-stride over the points: the counts are read on the device, maxPoints (the host's mirror) only sizes the grid
  const int blocks = std::max(1, std::min((maxPoints + 255) / 256, ctx->smCount * 8));
  k_render_maps_z<<<dim3(blocks, m), 256, 0, ctx->stream>>>(R, proj->rows, proj->cols, proj->min_distance,
                                                            proj->max_distance, d_z, zStride);
  NICP_CHECK_LAUNCH(ctx);
  k_render_maps_depth<<<dim3((P + 255) / 256, m), 256, 0, ctx->stream>>>(d_z, zStride, P, d_depth, depthStride);
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

// ---------------------------------------------------------------------------------------------
// SE3Prior / SE3RelativePrior / SE3AbsolutePrior (se3_prior.cpp:8-71) and their use in the
// Gauss-Newton step (aligner.cpp:97-108), evaluated by the solving thread.  Numeric Jacobians with
// eps = 1e-3 exactly as the reference; the 6x6 inverse of Jz (Eigen's general inverse) is a
// Gauss-Jordan elimination with partial pivoting in float64 (tolerance-level parity, like the oracle).
// ---------------------------------------------------------------------------------------------
struct DevPrior {
  int kind;
  float mean[16];
  float refInv[16];
  float info[36];
};

__device__ __noinline__ void prior_error(const DevPrior &pr, const float *mean, const float *invT, float *e) {
  float t[16];
  if (pr.kind == 0) {
    iso_mul(invT, mean, t);
  } else {
    float u[16];
    iso_mul(invT, pr.refInv, u);
    iso_mul(u, mean, t);
  }
  t2v(t, e);
}
__device__ __noinline__ void mat6_mul(const float *A, const float *B, float *C) {
  float t[36];
  for (int c = 0; c < 6; c++)
    for (int r = 0; r < 6; r++) {
      float s = 0.0f;
      for (int k = 0; k < 6; k++) s = fadd(s, fmul(NM6(A, r, k), NM6(B, k, c)));
      NM6(t, r, c) = s;
    }
  for (int i = 0; i < 36; i++) C[i] = t[i];
}
__device__ __noinline__ void mat6_transpose(const float *A, float *At) {
  float t[36];
  for (int r = 0; r < 6; r++)
    for (int c = 0; c < 6; c++) NM6(t, r, c) = NM6(A, c, r);
  for (int i = 0; i < 36; i++) At[i] = t[i];
}
__device__ __noinline__ void mat6_inverse(const float *A, float *Ai) {
  double a[6][12];
  for (int r = 0; r < 6; r++)
    for (int c = 0; c < 6; c++) {
      a[r][c] = NM6(A, r, c);
      a[r][c + 6] = (r == c) ? 1.0 : 0.0;
    }
  for (int k = 0; k < 6; k++) {
    int piv = k;
    for (int r = k + 1; r < 6; r++)
      if (fabs(a[r][k]) > fabs(a[piv][k])) piv = r;
    if (piv != k)
      for (int c = 0; c < 12; c++) { double t = a[k][c]; a[k][c] = a[piv][c]; a[piv][c] = t; }
    double d = a[k][k];
    for (int c = 0; c < 12; c++) a[k][c] = __ddiv_rn(a[k][c], d);
    for (int r = 0; r < 6; r++)
      if (r != k) {
        double f = a[r][k];
        if (f != 0.0)
          for (int c = 0; c < 12; c++) a[r][c] = __dsub_rn(a[r][c], __dmul_rn(f, a[k][c]));
      }
  }
  for (int r = 0; r < 6; r++)
    for (int c = 0; c < 6; c++) NM6(Ai, r, c) = (float)a[r][c + 6];
}
__device__ __noinline__ void add_priors(const DevPrior *priors, int numPriors, const float *invT, float *H, float *b) {
  const float epsilon = 1e-3f, iEps = fdiv(0.5f, epsilon);
  for (int j = 0; j < numPriors; j++) {
    const DevPrior &pr = priors[j];
    float e[6], J[36], Jz[36];
    prior_error(pr, pr.mean, invT, e);
    for (int i = 0; i < 6; i++) {
      float up[6] = {0, 0, 0, 0, 0, 0}, dn[6] = {0, 0, 0, 0, 0, 0}, Tu[16], Td[16], A[16], eu[6], ed[6];
      up[i] = epsilon;
      dn[i] = -epsilon;
      v2t(up, Tu);
      v2t(dn, Td);
      // SE3Prior::jacobian: perturb the estimate on the left
      iso_mul(Tu, invT, A);
      prior_error(pr, pr.mean, A, eu);
      iso_mul(Td, invT, A);
      prior_error(pr, pr.mean, A, ed);
      for (int r = 0; r < 6; r++) NM6(J, r, i) = fmul(iEps, fsub(eu[r], ed[r]));
      // SE3Prior::jacobianZ: perturb the prior mean on the right
      iso_mul(pr.mean, Tu, A);
      prior_error(pr, A, invT, eu);
      iso_mul(pr.mean, Td, A);
      prior_error(pr, A, invT, ed);
      for (int r = 0; r < 6; r++) NM6(Jz, r, i) = fmul(iEps, fsub(eu[r], ed[r]));
    }
    float iJz[36], iJzT[36], info[36], Jt[36], A[36], Hp[36];
    mat6_inverse(Jz, iJz);
    mat6_transpose(iJz, iJzT);
    mat6_mul(iJzT, pr.info, A);
    mat6_mul(A, iJz, info);
    mat6_transpose(J, Jt);
    mat6_mul(Jt, info, A);
    mat6_mul(A, J, Hp);
    for (int i = 0; i < 36; i++) H[i] = fadd(H[i], Hp[i]);
    for (int r = 0; r < 6; r++) {
      float s = 0.0f;
      for (int k = 0; k < 6; k++) s = fadd(s, fmul(NM6(A, r, k), e[k]));
      b[r] = fadd(b[r], s);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Sum the per-CTA partial rows in fixed order, assemble H/b (linearizer.cpp:109-114), then:
//  mode 0: one Gauss-Newton step of Aligner::align (aligner.cpp:84-118): H += I + 1000 I,
//          dx = LDLT(H)^-1 (-b), invT = v2t(dx) invT; if lastInner: T = invT^-1, T = v2t(t2v(T)),
//          and the matrices of the next iteration (invT = T^-1, KRt for the next projection).
//  mode 1: _computeStatistics' linearisation: store H/b + image statistics, write the result record.
//  mode 2: stage-level call: store H/b/error/inliers/ncorr only.
// ---------------------------------------------------------------------------------------------
// (kRowGroups, first-level CTAs per pair of k_reduce_solve, lives in nicp_internal.cuh: it sizes partials2)

// the dense part, executed by one thread: tot = the 32 sums of the pair
// PRIORS selects the instantiation that carries the SE(3)-prior code (numeric Jacobians, 6x6 float64 inverse): it is
// ~4x the size of the plain one, and the solving thread's run time is dominated by instruction fetch.
template <bool PRIORS>
__device__ __forceinline__ void solve_step(const PairDesc &D, const float *tot, int mode, int lastInner, int firstInner, int iter,
                                           const AlignConsts &ac) {
  PairState *st = D.state;
  float H[36], b[6];
  // Htt / Hrr upper triangles mirrored, Htr full
  const int ut[3][3] = {{0, 1, 2}, {1, 3, 4}, {2, 4, 5}};
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) {
      NM6(H, r, c) = tot[A_HTT + ut[r][c]];
      NM6(H, r + 3, c + 3) = tot[A_HRR + ut[r][c]];
      NM6(H, r, c + 3) = tot[A_HTR + r * 3 + c];
      NM6(H, c + 3, r) = tot[A_HTR + r * 3 + c];
    }
  for (int r = 0; r < 3; r++) { b[r] = tot[A_BT + r]; b[r + 3] = tot[A_BR + r]; }

  if (mode == 1) {
    for (int k = 0; k < 36; k++) st->statH[k] = H[k];
    for (int k = 0; k < 6; k++) st->statb[k] = b[k];
    st->img_sum = tot[29];
    st->img_nonzeros = (int)tot[30];
    st->img_inliers = (int)tot[31];
    nicp_align_result *res = D.result;
    if (res) {
      for (int k = 0; k < 16; k++) res->T[k] = st->T[k];
      res->error = st->error;
      res->inliers = st->inliers;
      res->num_correspondences = st->ncorr;
      res->image_non_zeros = st->img_nonzeros;
      res->image_inliers = st->img_inliers;
      res->image_outliers = st->img_nonzeros - st->img_inliers;
      res->image_reprojection_distance = fdiv(st->img_sum, (float)st->img_nonzeros);
      res->status = NICP_OK;
      res->reserved[0] = st->sumMidx;
      res->reserved[1] = st->sumMacc;
    }
    return;
  }

  for (int k = 0; k < 36; k++) st->H[k] = H[k];
  for (int k = 0; k < 6; k++) st->b[k] = b[k];
  st->error = tot[A_ERR];
  st->inliers = (int)tot[A_INL];
  if (firstInner) {
    st->ncorr = (int)tot[A_NCORR];
    st->sumMidx += tot[A_MIDX];
    st->sumMacc += tot[A_NCORR];
  }
  if (mode == 2) return;

  if (D.trace && firstInner) {
    float *tr = D.trace + 61 * iter;
    for (int k = 0; k < 16; k++) tr[k] = st->T[k];
    for (int k = 0; k < 36; k++) tr[16 + k] = H[k];
    for (int k = 0; k < 6; k++) tr[52 + k] = b[k];
    tr[58] = st->error;
    tr[59] = (float)st->inliers;
    tr[60] = (float)st->ncorr;
  }

  // aligner.cpp:92-94: H = H_lin + I; H += 1000 I
  for (int d = 0; d < 6; d++) NM6(H, d, d) = fadd(fadd(NM6(H, d, d), 1.0f), 1000.0f);
  float nb[6], dx[6], dT[16], invT[16];
  for (int k = 0; k < 16; k++) invT[k] = st->invT[k];
  if (PRIORS) {
    if (D.numPriors > 0) add_priors(reinterpret_cast<const DevPrior *>(D.priors), D.numPriors, invT, H, b);
  }
  for (int k = 0; k < 6; k++) nb[k] = -b[k];
  ldlt_solve6(H, nb, dx);
  v2t(dx, dT);
  iso_mul(dT, invT, invT);
  if (!lastInner) {
    fix_last_row(invT);
    for (int k = 0; k < 16; k++) st->invT[k] = invT[k];
    return;
  }
  // aligner.cpp:115-117
  float T[16], v[6], tmp[16];
  iso_inverse(invT, T);
  t2v(T, v);
  v2t(v, T);
  fix_last_row(T);
  for (int k = 0; k < 16; k++) st->T[k] = T[k];
  iso_inverse(T, invT);
  fix_last_row(invT);
  for (int k = 0; k < 16; k++) st->invT[k] = invT[k];
  iso_mul(T, ac.refOffset, tmp);
  store_cam_KRt(ac.cams, tmp, st);
}

// Deterministic final pass + solve in ONE launch: kRowGroups CTAs per pair; CTA g adds the partial rows of its contiguous
// group (warp w takes rows w, w+8, ... in order, 8 loads in flight; the 8 warps are added in order) and writes one row of
// partials2.  The CTA that finishes last (ticket in PairState) adds the kRowGroups rows in order and runs the dense
// step, so H, b and the pose do not depend on which CTA that is.
template <bool PRIORS>
__global__ void __launch_bounds__(256) k_reduce_solve(const PairDesc *__restrict__ desc, int numBlocks, int mode, int lastInner,
                                                      int firstInner, int iter, AlignConsts ac) {
  const PairDesc &D = desc[blockIdx.y];
  __shared__ float red[8][kAccum];
  __shared__ float tot[kAccum];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int per = (numBlocks + kRowGroups - 1) / kRowGroups;
  const int begin = blockIdx.x * per, end = min(begin + per, numBlocks);
  float s = 0.0f;
  const float *__restrict__ rows = D.partials + lane;
  // warp w adds rows w, w + 8, ... of the CTA's group in order; 16 loads in flight (a 640x480 pair has 200 rows per CTA:
  // two rounds per warp), rows past the end are not added.  (The grouping is part of the result's bits: 32 groups were
  // measured 13 us faster per alignment and moved two free-running comparisons with the oracle outside their tolerance.)
  for (int bi = begin + warp; bi < end; bi += 16 * 8) {
    float v[16];
#pragma unroll
    for (int u = 0; u < 16; u++) v[u] = bi + u * 8 < end ? __ldcg(rows + (size_t)(bi + u * 8) * kAccum) : 0.0f;
#pragma unroll
    for (int u = 0; u < 16; u++)
      if (bi + u * 8 < end) s += v[u];
  }
  red[warp][lane] = s;
  __syncthreads();
  if (warp != 0) return;
  float t = red[0][lane];
#pragma unroll
  for (int w = 1; w < 8; w++) t += red[w][lane];
  D.partials2[blockIdx.x * kAccum + lane] = t;
  __threadfence();
  __syncwarp();
  int last = 0;
  if (lane == 0) last = (atomicAdd(&D.state->ticket, 1) == kRowGroups - 1) ? 1 : 0;
  last = __shfl_sync(0xffffffffu, last, 0);
  if (!last) return;
  __threadfence();
  float sum = 0.0f;
#pragma unroll
  for (int g = 0; g < kRowGroups; g++) sum += __ldcg(&D.partials2[g * kAccum + lane]);
  tot[lane] = sum;
  __syncwarp();
  if (lane != 0) return;
  D.state->ticket = 0;
  solve_step<PRIORS>(D, tot, mode, lastInner, firstInner, iter, ac);
}

// Aligner::_computeStatistics' dense tail for a batch: one thread per pair (sigma points, 6x6 pseudo-inverse and inverse,
// eigen-ratios; nicp_stats_tail.cuh -- the function a single alignment runs on the host, bit for bit).  Works on the
// result records and the gathered H of a chunk (both indexed by the caller's pair index), not on the slot state: it runs
// on the tail stream while the next chunk already reuses the slots.
__global__ void __launch_bounds__(32) k_statistics(nicp_align_result *__restrict__ results, const float *__restrict__ statHb, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  nicp_align_result *res = results + i;
  float H[36], T[16], omega[36], tr, rr;
  for (int k = 0; k < 36; k++) H[k] = statHb[(size_t)i * 42 + k];
  for (int k = 0; k < 16; k++) T[k] = res->T[k];
  compute_statistics_tail(H, T, omega, &tr, &rr);
  for (int k = 0; k < 36; k++) res->omega[k] = omega[k];
  res->translational_eigen_ratio = tr;
  res->rotational_eigen_ratio = rr;
}

// H / b of the _computeStatistics linearisation, to the slot of the pair's RESULT record (descriptors are ordered by
// current cloud inside a chunk, results by the caller's pair index)
__global__ void k_gather_stat(const PairDesc *__restrict__ desc, int n, const nicp_align_result *__restrict__ results,
                              float *__restrict__ statHb) {
  int i = blockIdx.x;
  const PairState *st = desc[i].state;
  const size_t slot = (size_t)(desc[i].result - results);
  for (int k = threadIdx.x; k < 42; k += blockDim.x) statHb[slot * 42 + k] = k < 36 ? st->statH[k] : st->statb[k - 36];
}

// ---------------------------------------------------------------------------------------------
// host drivers
// ---------------------------------------------------------------------------------------------
int partial_rows_for(const nicp_context *ctx, size_t pixels) {
  int a = (int)((pixels + kTilePixels - 1) / kTilePixels);
  return a > ctx->blocksPerPair ? a : ctx->blocksPerPair;
}

// per-pair kernel: grid = tiles x pairs, swapped to pair-fastest when the tile count fits gridDim.y
template <int MODE>
static void launch_tiled(nicp_context *ctx, dim3 grid, int parity, int epoch, int writeCorr, const AlignConsts &ac, int P,
                         int imgStats, float imgThr, int curEpoch) {
  constexpr size_t smem = 3 * kTilePixels * sizeof(float4);
  const bool swap = grid.x <= 65535;
  const dim3 g = swap ? dim3(grid.y, grid.x) : grid;
  k_corr_lin_tiled<MODE><<<g, kTileLanes, smem, ctx->stream>>>(ctx->d_desc, parity, epoch, writeCorr, ac, P, imgStats, imgThr,
                                                               swap ? 1 : 0, curEpoch);
}
// the pair groups live behind the flags and the projection order in the descriptor staging area, 16-byte aligned
static size_t groups_offset(const nicp_context *ctx) {
  size_t off = sizeof(PairDesc) * (size_t)ctx->slots + 2 * sizeof(int) * (size_t)ctx->slots;
  return (off + 15) & ~(size_t)15;
}
const PairGroup *device_groups(const nicp_context *ctx) {
  return reinterpret_cast<const PairGroup *>(reinterpret_cast<const unsigned char *>(ctx->d_desc) + groups_offset(ctx));
}
PairGroup *host_groups(nicp_context *ctx) {
  return reinterpret_cast<PairGroup *>(reinterpret_cast<unsigned char *>(ctx->h_desc) + groups_offset(ctx));
}
// grouped kernel: grid = groups x tiles, group-fastest when the group count fits gridDim.x
template <int MODE>
static void launch_group(nicp_context *ctx, int nGroups, int tiles, int parity, int epoch, int writeCorr, const AlignConsts &ac,
                         int P, int imgStats, float imgThr, int curEpoch) {
  const PairGroup *d_groups = device_groups(ctx);
  const bool groupFast = tiles <= 65535;
  const dim3 g = groupFast ? dim3(nGroups, tiles) : dim3(tiles, nGroups);
  SlotBases B;
  B.refZ = ctx->d_refZ + (size_t)parity * ctx->slots * ctx->slotPixels;
  B.curZ = ctx->d_curZ;
  B.curIndex = ctx->d_curIndex;
  B.corrImage = ctx->d_corrImage;
  B.partials = ctx->d_partials;
  B.state = ctx->d_state;
  B.slotPixels = (long long)ctx->slotPixels;
  B.partialStride = (long long)ctx->partialRows * kAccum;
  if (ac.robust)
    k_corr_lin_group<MODE, true><<<g, kTileLanes, 0, ctx->stream>>>(ctx->d_desc, d_groups, B, epoch, writeCorr, ac, P, imgStats,
                                                                    imgThr, groupFast ? 1 : 0, curEpoch);
  else
    k_corr_lin_group<MODE, false><<<g, kTileLanes, 0, ctx->stream>>>(ctx->d_desc, d_groups, B, epoch, writeCorr, ac, P, imgStats,
                                                                     imgThr, groupFast ? 1 : 0, curEpoch);
}
// MODE 0 / 1 launch of the fused kernel over nb tiles per pair.  Pairs that share their current cloud with at least a few
// others go through the grouped kernel; lone pairs (a single alignment, a batch of unrelated pairs) through the per-pair
// kernel, whose prologue is shorter.  The rows they produce are bit-identical (same term, same lane / pixel mapping, same
// butterfly).
static void launch_corr_lin(nicp_context *ctx, int mode, int nPairs, int nGroups, int nb, int parity, int epoch, int writeCorr,
                            const AlignConsts &ac, int P, int imgStats, float imgThr, int curEpoch = kEpochFresh) {
  const bool grouped = takes_grouped(ctx, nPairs, nGroups);
  const dim3 grid(nb, nPairs);
  if (mode == 0) {
    if (grouped) launch_group<0>(ctx, nGroups, nb, parity, epoch, writeCorr, ac, P, imgStats, imgThr, curEpoch);
    else launch_tiled<0>(ctx, grid, parity, epoch, writeCorr, ac, P, imgStats, imgThr, curEpoch);
  } else {
    if (grouped) launch_group<1>(ctx, nGroups, nb, parity, epoch, writeCorr, ac, P, imgStats, imgThr, curEpoch);
    else launch_tiled<1>(ctx, grid, parity, epoch, writeCorr, ac, P, imgStats, imgThr, curEpoch);
  }
}

static cudaEvent_t next_event(std::vector<cudaEvent_t> *pool, size_t &used) {
  if (used == pool->size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    pool->push_back(e);
  }
  return (*pool)[used++];
}
#define NICP_TIME_BEGIN(pool, used) \
  if (ctx->timing) cudaEventRecord(next_event(ctx->pool, ctx->used), st)
#define NICP_TIME_END(pool, used) \
  if (ctx->timing) cudaEventRecord(next_event(ctx->pool, ctx->used), st)

// runs Aligner::align for the nPairs descriptors staged in ctx->h_desc (one lock-step chunk).
// ownsCur: per pair, 1 if the pair's curZ/curIndex buffers must be produced by it.
int run_align_chunk(nicp_context *ctx, int nPairs, const AlignConsts &ac, const CamSet &cams, const float curOffset[16],
                    int outerIters, int innerIters, float imgThreshold, int nGroups, const int *h_ownsCur,
                    bool fresh, int resultOffset) {
  cudaStream_t st = ctx->stream;
  const int P = ac.rows * ac.cols;
  const int nb = std::max(1, (P + kTilePixels - 1) / kTilePixels);
  bool anyPriors = false;  // the solve kernel carrying the SE(3)-prior code is only launched when a pair of the chunk needs it
  for (int i = 0; i < nPairs; i++) anyPriors = anyPriors || ctx->h_desc[i].numPriors > 0;
  // descriptors + ownership flags (flags live right after the descriptors in the staging buffer)
  int *h_flags = reinterpret_cast<int *>(ctx->h_desc + ctx->slots);
  int *d_flags = reinterpret_cast<int *>(ctx->d_desc + ctx->slots);
  for (int i = 0; i < nPairs; i++) h_flags[i] = h_ownsCur ? h_ownsCur[i] : 1;
  // projection order: descriptors sorted by reference cloud (stable).  A chunk's descriptors are ordered by CURRENT cloud
  // for the grouped kernel; k_project is DRAM bound and reads the reference's 12-byte point stream, so pairs with the same
  // reference should be neighbours in ITS grid.
  int *h_order = h_flags + ctx->slots, *d_order = nullptr;
  {
    bool sharedRef = false;
    for (int i = 0; i < nPairs; i++) h_order[i] = i;
    std::stable_sort(h_order, h_order + nPairs,
                     [&](int a, int b) { return (uintptr_t)ctx->h_desc[a].refPoints < (uintptr_t)ctx->h_desc[b].refPoints; });
    for (int i = 1; i < nPairs && !sharedRef; i++)
      sharedRef = ctx->h_desc[h_order[i]].refPoints == ctx->h_desc[h_order[i - 1]].refPoints;
    if (sharedRef) d_order = d_flags + ctx->slots;
  }
  NICP_CUDA(cudaMemcpyAsync(ctx->d_desc, ctx->h_desc, sizeof(PairDesc) * nPairs, cudaMemcpyHostToDevice, st));
  // flags and the pair groups (staged by the caller behind the flags) in one copy
  NICP_CUDA(cudaMemcpyAsync(d_flags, h_flags, (groups_offset(ctx) - sizeof(PairDesc) * (size_t)ctx->slots) + sizeof(PairGroup) * nGroups,
                            cudaMemcpyHostToDevice, st));
  // z-buffer words carry an epoch tag instead of being cleared per iteration (z_encode in nicp_internal.cuh).
  // (slot buffers are contiguous: refZ is laid out [2][slots][slotPixels], curZ [slots][slotPixels])
  //  fresh (single-pair nicp_align, the CUDA-graph path): this call clears its own slots and counts its iterations
  //    from 0; the buffers as a whole are left inconsistent (zIter / zCurGen = -1).
  //  batch: all slots share one running iteration count zIter across chunks and calls, so the reference z-buffers are
  //    cleared only when the 4-bit epoch wraps (every 32 iterations) and the current z-buffers every 16 chunks, always
  //    over all slots.
  unsigned long long *const refZbuf[2] = {ctx->d_refZ, ctx->d_refZ + (size_t)ctx->slots * ctx->slotPixels};
  const size_t zBytes = sizeof(unsigned long long) * ctx->slotPixels * nPairs;
  const size_t zBytesAll = sizeof(unsigned long long) * ctx->slotPixels * ctx->slots;
  long long iterBase = 0;
  int curEpoch = kEpochFresh;
  if (fresh) {
    NICP_CUDA(cudaMemsetAsync(refZbuf[0], 0xFF, zBytes, st));
    NICP_CUDA(cudaMemsetAsync(refZbuf[1], 0xFF, zBytes, st));
    NICP_CUDA(cudaMemsetAsync(ctx->d_curZ, 0xFF, zBytes, st));
    ctx->zIter = -1;
    ctx->zCurGen = -1;
  } else {
    if (ctx->zIter < 0) {
      NICP_CUDA(cudaMemsetAsync(refZbuf[0], 0xFF, zBytesAll, st));
      NICP_CUDA(cudaMemsetAsync(refZbuf[1], 0xFF, zBytesAll, st));
      ctx->zIter = 0;
    }
    if (ctx->zCurGen < 0 || (ctx->zCurGen & 15) == 0) {
      NICP_CUDA(cudaMemsetAsync(ctx->d_curZ, 0xFF, zBytesAll, st));
      if (ctx->zCurGen < 0) ctx->zCurGen = 0;
    }
    iterBase = ctx->zIter;
    curEpoch = kEpochFresh - (ctx->zCurGen & 15);
    ctx->zIter += outerIters > 0 ? outerIters : 0;
    ctx->zCurGen++;
  }
  k_init_pairs<<<(nPairs + 63) / 64, 64, 0, st>>>(ctx->d_desc, nPairs, ac);
  NICP_CHECK_LAUNCH(ctx);
  // grid-stride, 8 points per thread at full density (two rounds of four loads in flight).  The kernel is DRAM bound
  // (16-byte points + read-modify-write of the z-buffer sectors): 64/128/256 threads x 4/8/16 points all land on 82-86 us
  // A lone pair (or a handful) is latency bound instead: 150 CTAs would leave most SMs with one CTA, so the grid is sized
  // for two points per thread there.
  constexpr int projThreads = 256;
  const int projPerThread = nPairs >= 8 ? 8 : 2;
  const int projBlocks = (P + projThreads * projPerThread - 1) / (projThreads * projPerThread);
  dim3 pg(projBlocks, nPairs);
  // aligner.cpp:60-63: the current cloud is projected once with projector->setTransform(_currentSensorOffset)
  CamMats curMats, *d_curMats = nullptr;
  cam_mats_KRt(cams, curOffset, curMats);
  const CamGeom geom = geom_of(cams);
  if (cams.multi) {
    int rcm = upload_cam_mats(ctx, curMats, &d_curMats);
    if (rcm) return rcm;
    k_project_multi<<<pg, 256, 0, st>>>(ctx->d_desc, 2, geom, d_curMats, ac.rows, ac.cols, d_flags, curEpoch);
  } else {
    k_project<<<pg, projThreads, 0, st>>>(ctx->d_desc, 2, curMats.M[0], ac.rows, ac.cols, ac.minD, ac.maxD, d_flags, curEpoch, nullptr);
  }
  NICP_CHECK_LAUNCH(ctx);
  k_decode_cur<<<dim3((P + 1023) / 1024, nPairs), 256, 0, st>>>(ctx->d_desc, P, d_flags, curEpoch);
  NICP_CHECK_LAUNCH(ctx);
  const Affine dummy = curMats.M[0];
  int parity = (int)(iterBase & 1), epoch = epoch_of_iteration((int)(iterBase & 1023));
  for (int it = 0; it < outerIters; it++) {
    const long long G = iterBase + it;
    parity = (int)(G & 1);
    epoch = epoch_of_iteration((int)(G & 1023));
    // the 4-bit epoch wraps every 32 iterations: start that buffer fresh again
    if (G >= 2 && epoch == kEpochFresh)
      NICP_CUDA(cudaMemsetAsync(refZbuf[parity], 0xFF, fresh ? zBytes : zBytesAll, st));
    const int writeCorr = (it == outerIters - 1 || innerIters > 1) ? 1 : 0;
    NICP_TIME_BEGIN(evProj, evProjUsed);
    if (cams.multi)
      k_project_multi<<<pg, 256, 0, st>>>(ctx->d_desc, parity, geom, d_curMats, ac.rows, ac.cols, d_flags, epoch);
    else
      k_project<<<pg, projThreads, 0, st>>>(ctx->d_desc, parity, dummy, ac.rows, ac.cols, ac.minD, ac.maxD, d_flags, epoch, d_order);
    NICP_TIME_END(evProj, evProjUsed);
    NICP_CHECK_LAUNCH(ctx);
    for (int k = 0; k < innerIters; k++) {
      if (k == 0) {
        NICP_TIME_BEGIN(evCorr, evCorrUsed);
        launch_corr_lin(ctx, 0, nPairs, nGroups, nb, parity, epoch, writeCorr, ac, P, 0, 0.0f);
        NICP_TIME_END(evCorr, evCorrUsed);
      } else {
        launch_corr_lin(ctx, 1, nPairs, nGroups, nb, parity, epoch, 0, ac, P, 0, 0.0f, curEpoch);
      }
      NICP_CHECK_LAUNCH(ctx);
      if (anyPriors)
        k_reduce_solve<true><<<dim3(kRowGroups, nPairs), 256, 0, st>>>(ctx->d_desc, nb, 0, k == innerIters - 1, k == 0, it, ac);
      else
        k_reduce_solve<false><<<dim3(kRowGroups, nPairs), 256, 0, st>>>(ctx->d_desc, nb, 0, k == innerIters - 1, k == 0, it, ac);
      NICP_CHECK_LAUNCH(ctx);
    }
  }
  if (outerIters <= 0 || innerIters <= 0) {
    // no loop linearisation happened: the correspondence image must still be defined (all -1)
    for (int i = 0; i < nPairs; i++)
      NICP_CUDA(cudaMemsetAsync(ctx->h_desc[i].corrImage, 0xFF, sizeof(int) * P, st));
  }
  // _computeStatistics linearisation at the final T over the last correspondences + image statistics
  launch_corr_lin(ctx, 1, nPairs, nGroups, nb, parity, epoch, 0, ac, P, 1, imgThreshold, curEpoch);
  NICP_CHECK_LAUNCH(ctx);
  k_reduce_solve<false><<<dim3(kRowGroups, nPairs), 256, 0, st>>>(ctx->d_desc, nb, 1, 0, 0, 0, ac);
  NICP_CHECK_LAUNCH(ctx);
  (void)resultOffset;
  k_gather_stat<<<nPairs, 64, 0, st>>>(ctx->d_desc, nPairs, ctx->d_results, ctx->d_statHb);
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

// a batch: the records [base, base + n) leave the device complete (a single alignment finishes them on the host)
int launch_statistics(nicp_context *ctx, cudaStream_t s, int base, int n) {
  k_statistics<<<(n + 31) / 32, 32, 0, s>>>(ctx->d_results + base, ctx->d_statHb + (size_t)base * 42, n);
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

// stage-level: slot's refZ[0]/curIndex (or corrImage when fromCorrImage) already staged, state->invT set.
int run_correspond_linearize(nicp_context *ctx, const AlignConsts &ac, bool fromCorrImage, int numPixels) {
  cudaStream_t st = ctx->stream;
  const int nb = (numPixels + kTilePixels - 1) / kTilePixels;
  launch_corr_lin(ctx, fromCorrImage ? 1 : 0, 1, 1, nb, 0, kEpochFresh, 1, ac, numPixels, 0, 0.0f);
  NICP_CHECK_LAUNCH(ctx);
  k_reduce_solve<false><<<dim3(kRowGroups, 1), 256, 0, st>>>(ctx->d_desc, nb, 2, 0, 1, 0, ac);
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

}  // namespace nicp

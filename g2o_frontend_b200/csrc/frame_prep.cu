// frame_prep.cu -- depth image -> point/normal/curvature/information-matrix cloud.
//
// Replaces DepthImageConverterIntegralImage::compute (depthimageconverterintegralimage.cpp:15-55)
// and the pieces it calls:
//   PinholePointProjector::unProject / projectIntervals   pinholepointprojector.cpp:68-147
//   PointIntegralImage::compute / getRegion                 pointintegralimage.cpp:7-66
//   StatsCalculatorIntegralImage::compute                   statscalculatorintegralimage.cpp:14-82
//   Point/NormalInformationMatrixCalculator::compute        informationmatrixcalculator.cpp:9-58
//   Cloud::transformInPlace                                 cloud.cpp:173-186
//   DepthImage_convert_16UC1_to_32FC1 / DepthImage_scale    pwn_static.cpp:5-68
//
// Three kernels per frame:
//   k_integral_rows   one CTA per image row: unproject in registers, stage the 10 accumulator
//                     channels of the row in shared memory, scan them SEQUENTIALLY along image-x
//                     (the reference's float32 summation order is part of the result -- SURVEY.md
//                     section 7 hard part 1), write back coalesced (planar [10][rows][cols]).
//   k_integral_cols   one thread per (channel, column): sequential scan along image-y, coalesced
//                     across the warp, loads software-prefetched 16 rows ahead.
//   k_stats           one thread per pixel: compacted index straight from channel 0 of the
//                     integral image (no separate compaction pass), 4-corner region, covariance,
//                     closed-form 3x3 eigen-decomposition, normal / curvature / Omega_P / Omega_N,
//                     sensor-offset transform fused into the writes.
#include "nicp_internal.cuh"

namespace nicp {

// ---------------------------------------------------------------------------------------------
// DepthImage_convert_16UC1_to_32FC1 (pwn_static.cpp:54-68) + DepthImage_scale (:5-36)
// ---------------------------------------------------------------------------------------------
// Frames of one launch set (kernel parameter, no device-side descriptor array): frame f = blockIdx.y (depth convert, row
// pass), blockIdx.z (column pass, statistics).  A single frame is a batch of one.
struct PrepBatch {
  int n;
  const uint16_t *raw[kMaxPrepBatch];
  float *depth[kMaxPrepBatch];
  float *integral[kMaxPrepBatch];     // planar [10][rows][cols]
  float4 *points[kMaxPrepBatch], *normals[kMaxPrepBatch], *omega[kMaxPrepBatch];
  float *stats16[kMaxPrepBatch], *eigvals[kMaxPrepBatch];
  int *statsN[kMaxPrepBatch];
  int *count[kMaxPrepBatch];
};

// DepthImage_convert_16UC1_to_32FC1 of one raw value
__device__ __forceinline__ float depth_u16_to_m(uint16_t v, float scale) { return v ? fmul(scale, (float)v) : 0.0f; }

// DepthImage_scale(step > 1) of the converted rows x cols raw image at scaled pixel (r, c)
__device__ __forceinline__ float depth_scale_pixel(const uint16_t *__restrict__ raw, int rows, int cols, int r, int c, float scale,
                                                   int step, float maxCov) {
  float acc = 0.f, acc2 = 0.f;
  int np = 0;
  int sr = r * step, sc = c * step;
  for (int a = 0; a < step; a++)
    for (int b = 0; b < step; b++) {
      if (sr + a < rows && sc + b < cols) {
        float f = depth_u16_to_m(raw[(size_t)(sr + a) * cols + sc + b], scale);
        acc = fadd(acc, f);
        acc2 = fadd(acc2, fmul(f, f));
        np += f > 0;
      }
    }
  float res = 0.0f;
  if (np) {
    float mu = fdiv(acc, (float)np);
    float sigma = fsub(fdiv(acc2, (float)np), fmul(mu, mu));
    if (!(sigma > maxCov)) res = mu;
  }
  return res;
}

__global__ void k_depth_convert(PrepBatch B, int rows, int cols, float scale, int step, float maxCov) {
  const uint16_t *__restrict__ raw = B.raw[blockIdx.y];
  float *__restrict__ out = B.depth[blockIdx.y];
  int drows = rows / step, dcols = cols / step;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= drows * dcols) return;
  int r = i / dcols, c = i - r * dcols;
  if (step <= 1) {
    out[i] = depth_u16_to_m(raw[i], scale);
    return;
  }
  out[i] = depth_scale_pixel(raw, rows, cols, r, c, scale, step, maxCov);
}

// Raw frames of a MultiPointProjector rig -> composite depth images in the layout of CamSet (the one the Aligner projects
// into): camera i's raw image is H_i x W_i in sensor orientation (row = v, column = u) and scales to height_i x width_i;
// composite[u][colOff_i + v] = scaled pixel (v, u), and rows [width_i, rows) of camera i's column block are 0.
// grid = (ceil(max height / 32), ceil(rows / 32), frames x cameras), 32 x 8 threads: a 32 x 32 tile is converted along u
// (coalesced raw reads at step 1; at step > 1 a lane reads its own step x step box) into shared memory and written out
// transposed along v (coalesced composite writes).
struct RigFrames {
  const uint16_t *raw[kMaxPrepBatch * kMaxCams];  // frame f, camera i at f * nCams + i
  float *depth[kMaxPrepBatch];
  int nCams;
  int rawRows[kMaxCams], rawCols[kMaxCams], width[kMaxCams], height[kMaxCams], colOff[kMaxCams];
};

__global__ void __launch_bounds__(256) k_rig_depth_convert(RigFrames R, int rows, int cols, float scale, int step, float maxCov) {
  __shared__ float tile[32][33];  // [v][u], +1: the transposed reads hit 32 different banks
  const int f = blockIdx.z / R.nCams, cam = blockIdx.z - f * R.nCams;
  const int width = R.width[cam], height = R.height[cam];
  const int v0 = blockIdx.x * 32, u0 = blockIdx.y * 32;
  if (v0 >= height) return;  // the grid covers the tallest camera
  const uint16_t *__restrict__ raw = R.raw[blockIdx.z];
  const int rawRows = R.rawRows[cam], rawCols = R.rawCols[cam];
  for (int k = threadIdx.y; k < 32; k += 8) {
    const int v = v0 + k, u = u0 + threadIdx.x;
    float d = 0.0f;
    if (v < height && u < width)
      d = step <= 1 ? depth_u16_to_m(raw[(size_t)v * rawCols + u], scale) : depth_scale_pixel(raw, rawRows, rawCols, v, u, scale, step, maxCov);
    tile[k][threadIdx.x] = d;
  }
  __syncthreads();
  float *__restrict__ out = R.depth[f] + R.colOff[cam];
  for (int k = threadIdx.y; k < 32; k += 8) {
    const int u = u0 + k, v = v0 + threadIdx.x;
    if (u < rows && v < height) out[(size_t)u * cols + v] = tile[threadIdx.x][k];
  }
}

int launch_depth_convert(nicp_context *ctx, const uint16_t *d_raw, int rows, int cols, float scale, int step,
                         float maxCov, float *d_out) {
  if (step < 1) step = 1;
  int n = (rows / step) * (cols / step);
  PrepBatch B;
  memset(&B, 0, sizeof B);
  B.n = 1;
  B.raw[0] = d_raw;
  B.depth[0] = d_out;
  k_depth_convert<<<(n + 255) / 256, 256, 0, ctx->stream>>>(B, rows, cols, scale, step, maxCov);
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

// ---------------------------------------------------------------------------------------------
// pixel -> sensor-frame point.  Pinhole: _unProject(p, x = c, y = r, d) (pinholepointprojector.cpp:68-91).
// MultiPointProjector: the inverse of the composite layout the Aligner projects into (row = pixel u,
// col = pixel v + colOff of the camera): camera of the column block, _unProject(p, x = r, y = c - colOff, d).
// Returns false for an invalid depth (or a pixel outside every camera); iv = max-interval numerators.
// ---------------------------------------------------------------------------------------------
template <bool MULTI>
__device__ __forceinline__ bool pixel_point(const Affine &iKRt, float minD, float maxD, float ivx0, float ivy0,
                                            const PrepCams *__restrict__ pc, int r, int c, float d, float &x, float &y,
                                            float &z, float &ivx, float &ivy, int &camOut) {
  camOut = 0;
  if (!MULTI) {
    if (d < minD || d > maxD) return false;
    xform_point(iKRt, fmul((float)c, d), fmul((float)r, d), d, x, y, z);
    ivx = ivx0;
    ivy = ivy0;
    return true;
  } else {
    int cam = -1;
    for (int i = 0; i < pc->g.n; i++)
      if (c >= pc->g.colOff[i] && c < pc->g.colOff[i] + pc->g.height[i]) cam = i;
    if (cam < 0 || r >= pc->g.width[cam]) return false;
    if (d < pc->g.minD[cam] || d > pc->g.maxD[cam]) return false;
    const int v = c - pc->g.colOff[cam];
    camOut = cam;
    xform_point(pc->iKRt[cam], fmul((float)r, d), fmul((float)v, d), d, x, y, z);
    ivx = pc->ivx[cam];
    ivy = pc->ivy[cam];
    return true;
  }
}

// ---------------------------------------------------------------------------------------------
// PointIntegralImage::compute, pass 1 (scatter + prefix along image-x)
// ---------------------------------------------------------------------------------------------
template <bool MULTI>
__global__ void __launch_bounds__(256) k_integral_rows(PrepBatch B, int rows, int cols, Affine iKRt,
                                                       float minD, float maxD, const PrepCams *__restrict__ pc) {
  extern __shared__ float sm[];  // [10][stride]
  const float *__restrict__ depth = B.depth[blockIdx.y];
  float *__restrict__ I = B.integral[blockIdx.y];
  const int stride = cols + 1;   // +1: the 10 scanning lanes hit 10 different banks
  const int r = blockIdx.x;
  const float *drow = depth + (size_t)r * cols;
  for (int c = threadIdx.x; c < cols; c += blockDim.x) {
    float d = drow[c];
    float ch[kIntegralCh];
    float x, y, z, ivx, ivy;
    int cam;
    if (!pixel_point<MULTI>(iKRt, minD, maxD, 0.f, 0.f, pc, r, c, d, x, y, z, ivx, ivy, cam)) {
#pragma unroll
      for (int k = 0; k < kIntegralCh; k++) ch[k] = 0.0f;
    } else {
      ch[0] = 1.0f; ch[1] = x; ch[2] = y; ch[3] = z;
      ch[4] = fmul(x, x); ch[5] = fmul(x, y); ch[6] = fmul(x, z);
      ch[7] = fmul(y, y); ch[8] = fmul(y, z); ch[9] = fmul(z, z);
    }
#pragma unroll
    for (int k = 0; k < kIntegralCh; k++) sm[k * stride + c] = ch[k];
  }
  __syncthreads();
  if (threadIdx.x < kIntegralCh) {
    float *p = sm + threadIdx.x * stride;
    float v = p[0];
    int c = 1;
    for (; c + 8 <= cols; c += 8) {
      float t[8];
#pragma unroll
      for (int u = 0; u < 8; u++) t[u] = p[c + u];
#pragma unroll
      for (int u = 0; u < 8; u++) { v = fadd(t[u], v); p[c + u] = v; }
    }
    for (; c < cols; c++) { v = fadd(p[c], v); p[c] = v; }
  }
  __syncthreads();
  const size_t plane = (size_t)rows * cols;
  for (int k = 0; k < kIntegralCh; k++) {
    float *orow = I + k * plane + (size_t)r * cols;
    for (int c = threadIdx.x; c < cols; c += blockDim.x) orow[c] = sm[k * stride + c];
  }
}

// ---------------------------------------------------------------------------------------------
// PointIntegralImage::compute, pass 2 (prefix along image-y)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(64) k_integral_cols(PrepBatch B, int rows, int cols) {
  int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= cols) return;
  float *p = B.integral[blockIdx.z] + (size_t)blockIdx.y * rows * cols + x;
  float v = p[0];
  int y = 1;
  constexpr int U = 16;
  for (; y + U <= rows; y += U) {
    float t[U];
#pragma unroll
    for (int u = 0; u < U; u++) t[u] = p[(size_t)(y + u) * cols];
#pragma unroll
    for (int u = 0; u < U; u++) { v = fadd(t[u], v); p[(size_t)(y + u) * cols] = v; }
  }
  for (; y < rows; y++) { v = fadd(p[(size_t)y * cols], v); p[(size_t)y * cols] = v; }
}

// ---------------------------------------------------------------------------------------------
// Eigen::SelfAdjointEigenSolver<Matrix3f>::computeDirect (Eigen 3.2.x, SURVEY.md Appendix A4),
// called at statscalculatorintegralimage.cpp:56-57.  C symmetric (6 unique), evals ascending,
// U column-major.  atan2/cos/sin are evaluated in float64 and rounded to float32.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void cross3(const float *a, const float *b, float *o) {
  o[0] = fsub(fmul(a[1], b[2]), fmul(a[2], b[1]));
  o[1] = fsub(fmul(a[2], b[0]), fmul(a[0], b[2]));
  o[2] = fsub(fmul(a[0], b[1]), fmul(a[1], b[0]));
}
__device__ __forceinline__ float sqnorm3(const float *a) {
  return fadd(fadd(fmul(a[0], a[0]), fmul(a[1], a[1])), fmul(a[2], a[2]));
}
__device__ __forceinline__ void unit_orthogonal(const float *s, float *o) {
  const float prec = 1e-5f;
  if (!(fabsf(s[0]) <= fmul(fabsf(s[2]), prec)) || !(fabsf(s[1]) <= fmul(fabsf(s[2]), prec))) {
    float invnm = fdiv(1.0f, fsqrt(fadd(fmul(s[0], s[0]), fmul(s[1], s[1]))));
    o[0] = fmul(-s[1], invnm); o[1] = fmul(s[0], invnm); o[2] = 0.0f;
  } else {
    float invnm = fdiv(1.0f, fsqrt(fadd(fmul(s[1], s[1]), fmul(s[2], s[2]))));
    o[0] = 0.0f; o[1] = fmul(-s[2], invnm); o[2] = fmul(s[1], invnm);
  }
}
__device__ __forceinline__ void set_col(float *U, int col, const float *v) {
  // static-index friendly
  if (col == 0) { U[0] = v[0]; U[1] = v[1]; U[2] = v[2]; }
  else if (col == 1) { U[3] = v[0]; U[4] = v[1]; U[5] = v[2]; }
  else { U[6] = v[0]; U[7] = v[1]; U[8] = v[2]; }
}
__device__ void eigen3(float c00, float c10, float c20, float c11, float c21, float c22, float *evals, float *U) {
  const float eps = FLT_EPSILON;
  float scale = fmaxf(fmaxf(fmaxf(fabsf(c00), fabsf(c10)), fmaxf(fabsf(c20), fabsf(c11))), fmaxf(fabsf(c21), fabsf(c22)));
  float m00 = fdiv(c00, scale), m10 = fdiv(c10, scale), m20 = fdiv(c20, scale);
  float m11 = fdiv(c11, scale), m21 = fdiv(c21, scale), m22 = fdiv(c22, scale);
  const float s_inv3 = 1.0f / 3.0f;
  const float s_sqrt3 = 1.7320508075688772f;  // sqrtf(3.0f)
  float c0 = fsub(fsub(fsub(fadd(fmul(fmul(m00, m11), m22), fmul(fmul(fmul(2.0f, m10), m20), m21)),
                            fmul(fmul(m00, m21), m21)),
                       fmul(fmul(m11, m20), m20)),
                  fmul(fmul(m22, m10), m10));
  float c1 = fsub(fadd(fsub(fadd(fsub(fmul(m00, m11), fmul(m10, m10)), fmul(m00, m22)), fmul(m20, m20)), fmul(m11, m22)),
                  fmul(m21, m21));
  float c2 = fadd(fadd(m00, m11), m22);
  float c2_over_3 = fmul(c2, s_inv3);
  float a_over_3 = fmul(fsub(c1, fmul(c2, c2_over_3)), s_inv3);
  if (a_over_3 > 0.0f) a_over_3 = 0.0f;
  float half_b = fmul(0.5f, fadd(c0, fmul(c2_over_3, fsub(fmul(fmul(2.0f, c2_over_3), c2_over_3), c1))));
  float q = fadd(fmul(half_b, half_b), fmul(fmul(a_over_3, a_over_3), a_over_3));
  if (q > 0.0f) q = 0.0f;
  float rho = fsqrt(-a_over_3);
  float theta = fmul((float)atan2((double)fsqrt(-q), (double)half_b), s_inv3);
  float cos_theta = (float)cos((double)theta);
  float sin_theta = (float)sin((double)theta);
  float r0 = fadd(c2_over_3, fmul(fmul(2.0f, rho), cos_theta));
  float r1 = fsub(c2_over_3, fmul(rho, fadd(cos_theta, fmul(s_sqrt3, sin_theta))));
  float r2 = fsub(c2_over_3, fmul(rho, fsub(cos_theta, fmul(s_sqrt3, sin_theta))));
  float tsw;
  if (r0 >= r1) { tsw = r0; r0 = r1; r1 = tsw; }
  if (r1 >= r2) {
    tsw = r1; r1 = r2; r2 = tsw;
    if (r0 >= r1) { tsw = r0; r0 = r1; r1 = tsw; }
  }
  evals[0] = fmul(r0, scale); evals[1] = fmul(r1, scale); evals[2] = fmul(r2, scale);
  const float safeNorm2 = eps * eps;
  U[0] = 1.f; U[1] = 0.f; U[2] = 0.f; U[3] = 0.f; U[4] = 1.f; U[5] = 0.f; U[6] = 0.f; U[7] = 0.f; U[8] = 1.f;
  if (fsub(r2, r0) <= eps) return;
  float d0 = fsub(r2, r1), d1 = fsub(r1, r0);
  int k = d0 > d1 ? 2 : 0;
  float evk = d0 > d1 ? r2 : r0;
  d0 = d0 > d1 ? d1 : d0;
  float row0[3] = {fsub(m00, evk), m10, m20};
  float row1[3] = {m10, fsub(m11, evk), m21};
  float row2[3] = {m20, m21, fsub(m22, evk)};
  float cr[3], n, uk[3], u1[3], ul[3];
  cross3(row0, row1, cr);
  n = sqnorm3(cr);
  if (!(n > safeNorm2)) {
    cross3(row0, row2, cr);
    n = sqnorm3(cr);
    if (!(n > safeNorm2)) {
      cross3(row1, row2, cr);
      n = sqnorm3(cr);
      if (!(n > safeNorm2)) return;  // NumericalIssue: identity eigenvectors (oracle's definition)
    }
  }
  { float sn = fsqrt(n); uk[0] = fdiv(cr[0], sn); uk[1] = fdiv(cr[1], sn); uk[2] = fdiv(cr[2], sn); }
  if (d0 <= eps) {
    unit_orthogonal(uk, u1);
  } else {
    float r0v[3] = {fsub(m00, r1), m10, m20};
    float r1v[3] = {m10, fsub(m11, r1), m21};
    float r2v[3] = {m20, m21, fsub(m22, r1)};
    float nr0 = fsqrt(sqnorm3(r0v));
    float r0n[3] = {fdiv(r0v[0], nr0), fdiv(r0v[1], nr0), fdiv(r0v[2], nr0)};
    bool have = true;
    cross3(uk, r0n, cr);
    n = sqnorm3(cr);
    if (!(n > safeNorm2)) {
      cross3(uk, r1v, cr);
      n = sqnorm3(cr);
      if (!(n > safeNorm2)) {
        cross3(uk, r2v, cr);
        n = sqnorm3(cr);
        if (!(n > safeNorm2)) { unit_orthogonal(uk, u1); have = false; }
      }
    }
    if (have) { float sn = fsqrt(n); u1[0] = fdiv(cr[0], sn); u1[1] = fdiv(cr[1], sn); u1[2] = fdiv(cr[2], sn); }
    float t1[3], t2[3];
    cross3(u1, uk, t1);
    cross3(uk, t1, t2);
    float sn = fsqrt(sqnorm3(t2));
    u1[0] = fdiv(t2[0], sn); u1[1] = fdiv(t2[1], sn); u1[2] = fdiv(t2[2], sn);
  }
  {
    float t[3];
    cross3(uk, u1, t);
    float sn = fsqrt(sqnorm3(t));
    ul[0] = fdiv(t[0], sn); ul[1] = fdiv(t[1], sn); ul[2] = fdiv(t[2], sn);
  }
  set_col(U, k, uk);
  set_col(U, 1, u1);
  set_col(U, k == 2 ? 0 : 2, ul);
}

struct StatsConsts {
  Affine iKRt;      // unProject matrix with the projector at identity
  float minD, maxD;
  float ivx, ivy;   // K * (worldRadius, worldRadius, 0), rows 0 and 1 (projectIntervals)
  int minR, maxR, minPoints;
  float curvThr, omegaCurvThr;
  float flatP[3], flatN[3], nonflatN[3];
  int applyOffset;
  float M[16];      // sensor offset (last row fixed)
};

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// R * Om * R^T for the 3x3 blocks (InformationMatrixVector::transformInPlace, informationmatrix.h:111-121)
__device__ __forceinline__ void rotate_sym(const float *M, const float *Om /*3x3 col-major*/, float *out) {
  float t[9];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++)
      NM3(t, r, c) = dot3(NM4(M, r, 0), NM4(M, r, 1), NM4(M, r, 2), NM3(Om, 0, c), NM3(Om, 1, c), NM3(Om, 2, c));
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++)
      NM3(out, r, c) = dot3(NM3(t, r, 0), NM3(t, r, 1), NM3(t, r, 2), NM4(M, c, 0), NM4(M, c, 1), NM4(M, c, 2));
}

// StatsCalculatorIntegralImage::compute for one pixel (statscalculatorintegralimage.cpp:41-78): region sums of the window
// of radius clamp(k), mean / covariance (pointaccumulator.h:65-86), computeDirect, curvature, normal orientation.
// Returns false when the window holds fewer than minPoints points (outputs untouched).
__device__ __forceinline__ bool stats_core(const float *__restrict__ I, size_t plane, int rows, int cols, int r, int c, int k,
                                           const StatsConsts &sc, float px, float py, float pz, float &nx, float &ny, float &nz,
                                           float &curv, float *U, float *ev, float *mu, int &npts) {
  k = clampi(k, sc.minR, sc.maxR);
  // getRegion(c-k, c+k, r-k, r+k) (pointintegralimage.cpp:53-66)
  int x0 = clampi(c - k - 1, 0, cols - 1), x1 = clampi(c + k - 1, 0, cols - 1);
  int y0 = clampi(r - k - 1, 0, rows - 1), y1 = clampi(r + k - 1, 0, rows - 1);
  size_t o11 = (size_t)y1 * cols + x1, o00 = (size_t)y0 * cols + x0;
  size_t o10 = (size_t)y1 * cols + x0, o01 = (size_t)y0 * cols + x1;
  float acc[kIntegralCh];
#pragma unroll
  for (int ch = 0; ch < kIntegralCh; ch++) {
    const float *P = I + ch * plane;
    acc[ch] = fsub(fsub(fadd(P[o11], P[o00]), P[o10]), P[o01]);
  }
  if ((int)acc[0] < sc.minPoints) return false;
  npts = (int)acc[0];
  float dd = fdiv(1.0f, acc[0]);
  mu[0] = fmul(acc[1], dd); mu[1] = fmul(acc[2], dd); mu[2] = fmul(acc[3], dd);
  float c00 = fsub(fmul(acc[4], dd), fmul(mu[0], mu[0]));
  float c10 = fsub(fmul(acc[5], dd), fmul(mu[0], mu[1]));
  float c20 = fsub(fmul(acc[6], dd), fmul(mu[0], mu[2]));
  float c11 = fsub(fmul(acc[7], dd), fmul(mu[1], mu[1]));
  float c21 = fsub(fmul(acc[8], dd), fmul(mu[1], mu[2]));
  float c22 = fsub(fmul(acc[9], dd), fmul(mu[2], mu[2]));
  eigen3(c00, c10, c20, c11, c21, c22, ev, U);
  if (ev[0] < 0.0f) ev[0] = 0.0f;
  // Stats::curvature (stats.h:98-103): float sum, double divide
  curv = (float)((double)ev[0] / ((double)fadd(fadd(ev[0], ev[1]), ev[2]) + 1e-9));
  nx = U[0]; ny = U[1]; nz = U[2];
  if (curv < sc.curvThr) {
    if (dot4(nx, ny, nz, 0.0f, px, py, pz, 1.0f) > 0) { nx = -nx; ny = -ny; nz = -nz; }
  } else {
    nx = ny = nz = 0.0f;
  }
  return true;
}

// Point / NormalInformationMatrixCalculator::compute for one point (informationmatrixcalculator.cpp:17-35, 46-57):
// OP / ON stay zero for a zero normal
__device__ __forceinline__ void information_core(float nx, float ny, float nz, float curv, const float *U, const float *ev,
                                                 const StatsConsts &sc, float *OP, float *ON) {
  float sq = fadd(fadd(fmul(nx, nx), fmul(ny, ny)), fmul(nz, nz));
  if (sq > 0) {
    bool flat = curv < sc.omegaCurvThr;
    float dg[3];
    if (flat) { dg[0] = sc.flatP[0]; dg[1] = sc.flatP[1]; dg[2] = sc.flatP[2]; }
    else { dg[0] = fdiv(1.0f, ev[0]); dg[1] = fdiv(1.0f, ev[1]); dg[2] = fdiv(1.0f, ev[2]); }
    float UD[9];
    for (int rr = 0; rr < 3; rr++)
      for (int cc = 0; cc < 3; cc++) NM3(UD, rr, cc) = fmul(NM3(U, rr, cc), dg[cc]);
    for (int rr = 0; rr < 3; rr++)
      for (int cc = 0; cc < 3; cc++)
        NM3(OP, rr, cc) = dot3(NM3(UD, rr, 0), NM3(UD, rr, 1), NM3(UD, rr, 2), NM3(U, cc, 0), NM3(U, cc, 1), NM3(U, cc, 2));
    const float *dn = flat ? sc.flatN : sc.nonflatN;
    ON[0] = dn[0]; ON[4] = dn[1]; ON[8] = dn[2];
  }
}

template <bool MULTI>
__global__ void __launch_bounds__(256, 4) k_stats(PrepBatch B, int rows, int cols, StatsConsts sc,
                                               const PrepCams *__restrict__ pc, int *__restrict__ index,
                                               int *__restrict__ interval) {
  // index / interval images (single-frame calls that asked for them) may be null: a batch does not materialise them
  const int f = blockIdx.z;
  const float *__restrict__ depth = B.depth[f];
  const float *__restrict__ I = B.integral[f];
  float4 *__restrict__ points = B.points[f];
  float4 *__restrict__ normals = B.normals[f];
  float4 *__restrict__ omega = B.omega[f];
  float *__restrict__ stats16 = B.stats16[f];
  float *__restrict__ eigvalsOut = B.eigvals[f];
  int *__restrict__ statsN = B.statsN[f];
  int *__restrict__ countOut = B.count[f];
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = blockIdx.y * blockDim.y + threadIdx.y;
  if (c >= cols || r >= rows) return;
  const size_t plane = (size_t)rows * cols;
  const size_t pix = (size_t)r * cols + c;
  if (r == rows - 1 && c == cols - 1) *countOut = (int)I[pix];
  const float d = depth[pix];
  float px, py, pz, ivx, ivy;
  int cam;
  if (!pixel_point<MULTI>(sc.iKRt, sc.minD, sc.maxD, sc.ivx, sc.ivy, pc, r, c, d, px, py, pz, ivx, ivy, cam)) {
    if (index) index[pix] = -1;
    if (interval) interval[pix] = -1;
    return;
  }
  // compacted index from channel 0 of the integral image (exact integer counts in float32)
  int idx;
  if (!MULTI) {
    // raster order: valid pixels in the rows above + valid pixels of this row up to c
    float above = r > 0 ? I[(size_t)(r - 1) * cols + cols - 1] : 0.0f;
    float upto = I[pix] - (r > 0 ? I[pix - cols] : 0.0f);
    idx = (int)above + (int)upto - 1;
  } else {
    // MultiPointProjector::unProject concatenates the children's clouds (multipointprojector.cpp:59-90):
    // points of the earlier column blocks, then raster order inside this camera's block
    const int off = pc->g.colOff[cam], last = off + pc->g.height[cam] - 1;
    const float *Ir = I + (size_t)r * cols;
    const float *Ip = r > 0 ? Ir - cols : nullptr;
    float before = off > 0 ? I[(size_t)(rows - 1) * cols + off - 1] : 0.0f;
    float aboveBlock = Ip ? Ip[last] - (off > 0 ? Ip[off - 1] : 0.0f) : 0.0f;
    float rowUpTo = (Ir[c] - (Ip ? Ip[c] : 0.0f)) - (off > 0 ? (Ir[off - 1] - (Ip ? Ip[off - 1] : 0.0f)) : 0.0f);
    idx = (int)before + (int)aboveBlock + (int)rowUpTo - 1;
  }
  if (index) index[pix] = idx;

  // _projectInterval (pinholepointprojector.h:264-274)
  float invd = fdiv(1.0f, d);
  float ia = fmul(ivx, invd), ib = fmul(ivy, invd);
  int k = (ia > ib) ? (int)ia : (int)ib;
  if (interval) interval[pix] = k;

  float nx = 0.f, ny = 0.f, nz = 0.f, curv = 0.f;
  float OP[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  float ON[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  float U[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  float ev[3] = {0, 0, 0};
  float mu[3] = {0, 0, 0};
  int npts = 0;
  bool computed = false;

  if (k >= 0) {
    computed = stats_core(I, plane, rows, cols, r, c, k, sc, px, py, pz, nx, ny, nz, curv, U, ev, mu, npts);
    if (computed) information_core(nx, ny, nz, curv, U, ev, sc, OP, ON);
  }

  float S[16];
  if (stats16) {
    for (int i = 0; i < 16; i++) S[i] = 0.0f;
    for (int rr = 0; rr < 3; rr++)
      for (int cc = 0; cc < 3; cc++) NM4(S, rr, cc) = NM3(U, rr, cc);
    if (computed) { NM4(S, 0, 3) = mu[0]; NM4(S, 1, 3) = mu[1]; NM4(S, 2, 3) = mu[2]; }
    NM4(S, 3, 3) = 1.0f;
  }

  if (sc.applyOffset) {
    // Cloud::transformInPlace (cloud.cpp:173-186)
    Affine M = affine_from(sc.M);
    float tx, ty, tz;
    xform_point(M, px, py, pz, tx, ty, tz);
    px = tx; py = ty; pz = tz;
    xform_normal(M, nx, ny, nz, tx, ty, tz);
    nx = tx; ny = ty; nz = tz;
    float t9[9];
    rotate_sym(sc.M, OP, t9);
    for (int i = 0; i < 9; i++) OP[i] = t9[i];
    rotate_sym(sc.M, ON, t9);
    for (int i = 0; i < 9; i++) ON[i] = t9[i];
    if (stats16) {
      float o[16];
      for (int cc = 0; cc < 4; cc++)
        for (int rr = 0; rr < 4; rr++)
          NM4(o, rr, cc) = dot4(NM4(sc.M, rr, 0), NM4(sc.M, rr, 1), NM4(sc.M, rr, 2), NM4(sc.M, rr, 3), NM4(S, 0, cc),
                                NM4(S, 1, cc), NM4(S, 2, cc), NM4(S, 3, cc));
      for (int i = 0; i < 16; i++) S[i] = o[i];
    }
  }

  points[idx] = make_float4(px, py, pz, 1.0f);
  normals[idx] = make_float4(nx, ny, nz, curv);
  {
    const float P6[6] = {NM3(OP, 0, 0), NM3(OP, 0, 1), NM3(OP, 0, 2), NM3(OP, 1, 1), NM3(OP, 1, 2), NM3(OP, 2, 2)};
    const float N6[6] = {NM3(ON, 0, 0), NM3(ON, 0, 1), NM3(ON, 0, 2), NM3(ON, 1, 1), NM3(ON, 1, 2), NM3(ON, 2, 2)};
    const Omega3 w = omega_pack(P6, N6);
    omega[3 * (size_t)idx + 0] = w.o0;
    omega[3 * (size_t)idx + 1] = w.o1;
    omega[3 * (size_t)idx + 2] = w.o2;
  }
  if (stats16) {
    float4 *so = reinterpret_cast<float4 *>(stats16 + 16 * (size_t)idx);
    so[0] = make_float4(S[0], S[1], S[2], S[3]);
    so[1] = make_float4(S[4], S[5], S[6], S[7]);
    so[2] = make_float4(S[8], S[9], S[10], S[11]);
    so[3] = make_float4(S[12], S[13], S[14], S[15]);
    eigvalsOut[3 * (size_t)idx + 0] = ev[0];
    eigvalsOut[3 * (size_t)idx + 1] = ev[1];
    eigvalsOut[3 * (size_t)idx + 2] = ev[2];
    statsN[idx] = npts;
  }
}

static bool is_identity16(const float *m) {
  for (int r = 0; r < 4; r++)
    for (int c = 0; c < 4; c++)
      if (NM4(m, r, c) != (r == c ? 1.0f : 0.0f)) return false;
  return true;
}

// Shared-memory staged version of pass 2: a CTA owns a strip of 32 columns of one channel, pulls the whole
// strip (rows x 32 floats) into shared memory with coalesced loads from all its threads, lets 32 threads walk
// their column sequentially (the reference's order) at shared-memory latency, and writes the strip back
// coalesced.  ~8x faster than the register-prefetch version, which is kept for images too tall for 227 KB.
__global__ void __launch_bounds__(256) k_integral_cols_smem(PrepBatch B, int rows, int cols) {
  extern __shared__ float strip[];  // [rows][32]
  const int x0 = blockIdx.x * 32;
  float *plane = B.integral[blockIdx.z] + (size_t)blockIdx.y * rows * cols;
  const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;
  const bool inside = x0 + lx < cols;
#pragma unroll 8
  for (int y = ly; y < rows; y += 8) strip[y * 32 + lx] = inside ? plane[(size_t)y * cols + x0 + lx] : 0.0f;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = strip[lx];
    int y = 1;
    for (; y + 8 <= rows; y += 8) {
      float t[8];
#pragma unroll
      for (int u = 0; u < 8; u++) t[u] = strip[(y + u) * 32 + lx];
#pragma unroll
      for (int u = 0; u < 8; u++) { v = fadd(t[u], v); strip[(y + u) * 32 + lx] = v; }
    }
    for (; y < rows; y++) { v = fadd(strip[y * 32 + lx], v); strip[y * 32 + lx] = v; }
  }
  __syncthreads();
  if (inside) {
#pragma unroll 8
    for (int y = ly; y < rows; y += 8) plane[(size_t)y * cols + x0 + lx] = strip[y * 32 + lx];
  }
}

// Streaming version of pass 2 for batches: one thread per (column, channel, frame) walks its column in the reference's
// order with the next 16 rows already in flight while the current 16 are added (32 independent loads per thread); a warp
// covers 32 adjacent columns, so every load / store is one full 128-byte line and nothing is staged in shared memory.
// With F frames there are F * 6400 such threads: enough bytes in flight to run at memory speed, which a single frame
// (6400 threads) is not -- that case keeps the shared-memory strips above.
__global__ void __launch_bounds__(128) k_integral_cols_stream(PrepBatch B, int rows, int cols) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= cols) return;
  float *p = B.integral[blockIdx.z] + (size_t)blockIdx.y * rows * cols + x;
  constexpr int U = 16;
  float cur[U], nxt[U];
  float v = 0.0f;
  int y = 0;
  if (rows >= U) {
#pragma unroll
    for (int u = 0; u < U; u++) cur[u] = p[(size_t)u * cols];
  }
  for (; y + U <= rows; y += U) {
    const bool more = y + 2 * U <= rows;
    if (more) {
#pragma unroll
      for (int u = 0; u < U; u++) nxt[u] = p[(size_t)(y + U + u) * cols];
    }
    if (y == 0) {
      v = cur[0];  // row 0 is its own prefix (no 0 + x: -0.0f must stay -0.0f like in the reference)
#pragma unroll
      for (int u = 1; u < U; u++) { v = fadd(cur[u], v); p[(size_t)(y + u) * cols] = v; }
    } else {
#pragma unroll
      for (int u = 0; u < U; u++) { v = fadd(cur[u], v); p[(size_t)(y + u) * cols] = v; }
    }
    if (more) {
#pragma unroll
      for (int u = 0; u < U; u++) cur[u] = nxt[u];
    }
  }
  if (y == 0) { v = p[0]; y = 1; }
  for (; y < rows; y++) { v = fadd(p[(size_t)y * cols], v); p[(size_t)y * cols] = v; }
}

// one launch set (row pass, column pass, statistics) for the B.n frames of `B`: depth images already on the device
static int launch_prep_set(nicp_context *ctx, const PrepBatch &B, const nicp_projector *proj, const nicp_stats_params *sp,
                           const float sensorOffset[16], int *d_index, int *d_interval, const CamSet *cams) {
  const int rows = proj->rows, cols = proj->cols, F = B.n;
  const bool multi = cams && cams->multi;
  const PrepCams *d_pc = nullptr;
  if (multi) {
    // DepthImageConverterIntegralImage::compute sets the projector to identity, so child i sits at offset_i
    PrepCams pc;
    pc.g = geom_of(*cams);
    for (int i = 0; i < cams->n; i++) {
      float iKRt[16];
      compute_iKRt(cams->K[i], cams->offset[i], iKRt);
      pc.iKRt[i] = affine_from(iKRt);
      const float *Kc = cams->K[i];
      pc.ivx[i] = dot3(NM3(Kc, 0, 0), NM3(Kc, 0, 1), NM3(Kc, 0, 2), sp->world_radius, sp->world_radius, 0.0f);
      pc.ivy[i] = dot3(NM3(Kc, 1, 0), NM3(Kc, 1, 1), NM3(Kc, 1, 2), sp->world_radius, sp->world_radius, 0.0f);
    }
    NICP_CUDA(cudaMemcpyAsync(&ctx->d_cams->prep, &pc, sizeof pc, cudaMemcpyHostToDevice, ctx->stream));
    d_pc = &ctx->d_cams->prep;
  }
  float I4[16], iKRt[16];
  mat4_identity(I4);
  compute_iKRt(proj->K, I4, iKRt);
  Affine a = affine_from(iKRt);
  size_t smem = (size_t)kIntegralCh * (cols + 1) * sizeof(float);
  if (smem > 48 * 1024 && smem > ctx->rowsSmemCfg) {
    NICP_CUDA(cudaFuncSetAttribute(k_integral_rows<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    NICP_CUDA(cudaFuncSetAttribute(k_integral_rows<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ctx->rowsSmemCfg = smem;
  }
  if (multi)
    k_integral_rows<true><<<dim3(rows, F), 256, smem, ctx->stream>>>(B, rows, cols, a, proj->min_distance, proj->max_distance, d_pc);
  else
    k_integral_rows<false><<<dim3(rows, F), 256, smem, ctx->stream>>>(B, rows, cols, a, proj->min_distance, proj->max_distance, d_pc);
  NICP_CHECK_LAUNCH(ctx);
  const size_t stripBytes = (size_t)rows * 32 * sizeof(float);
  // batches of 4 or more frames stream the columns (enough threads to cover the memory latency); fewer frames stage strips
  // in shared memory
  if (F >= 4) {
    k_integral_cols_stream<<<dim3((cols + 127) / 128, kIntegralCh, F), 128, 0, ctx->stream>>>(B, rows, cols);
  } else if (stripBytes <= 200 * 1024) {
    // per context = per device: the attribute is a per-device property of the kernel
    if (stripBytes > 48 * 1024 && stripBytes > ctx->colsSmemCfg) {
      NICP_CUDA(cudaFuncSetAttribute(k_integral_cols_smem, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)stripBytes));
      ctx->colsSmemCfg = stripBytes;
    }
    k_integral_cols_smem<<<dim3((cols + 31) / 32, kIntegralCh, F), 256, stripBytes, ctx->stream>>>(B, rows, cols);
  } else {
    k_integral_cols<<<dim3((cols + 63) / 64, kIntegralCh, F), 64, 0, ctx->stream>>>(B, rows, cols);
  }
  NICP_CHECK_LAUNCH(ctx);

  StatsConsts sc;
  sc.iKRt = a;
  sc.minD = proj->min_distance;
  sc.maxD = proj->max_distance;
  const float *K = proj->K;
  sc.ivx = dot3(NM3(K, 0, 0), NM3(K, 0, 1), NM3(K, 0, 2), sp->world_radius, sp->world_radius, 0.0f);
  sc.ivy = dot3(NM3(K, 1, 0), NM3(K, 1, 1), NM3(K, 1, 2), sp->world_radius, sp->world_radius, 0.0f);
  sc.minR = sp->min_image_radius;
  sc.maxR = sp->max_image_radius;
  sc.minPoints = sp->min_points;
  sc.curvThr = sp->curvature_threshold;
  sc.omegaCurvThr = sp->omega_curvature_threshold;
  for (int i = 0; i < 3; i++) {
    sc.flatP[i] = sp->flat_omega_p[i];
    sc.flatN[i] = sp->flat_omega_n[i];
    sc.nonflatN[i] = sp->nonflat_omega_n[i];
  }
  for (int i = 0; i < 16; i++) sc.M[i] = sensorOffset[i];
  fix_last_row(sc.M);
  sc.applyOffset = is_identity16(sc.M) ? 0 : 1;
  dim3 bs(32, 8);
  dim3 gs((cols + 31) / 32, (rows + 7) / 8, F);
  if (multi)
    k_stats<true><<<gs, bs, 0, ctx->stream>>>(B, rows, cols, sc, d_pc, d_index, d_interval);
  else
    k_stats<false><<<gs, bs, 0, ctx->stream>>>(B, rows, cols, sc, d_pc, d_index, d_interval);
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

static void prep_batch_add(PrepBatch &B, float *d_depth, float *d_integral, nicp_cloud *cloud, bool keepStats) {
  const int f = B.n++;
  B.depth[f] = d_depth;
  B.integral[f] = d_integral;
  B.points[f] = cloud->points;
  B.normals[f] = cloud->normals;
  B.omega[f] = cloud->omega;
  const bool ks = keepStats && cloud->stats16;
  B.stats16[f] = ks ? cloud->stats16 : nullptr;
  B.eigvals[f] = ks ? cloud->eigvals : nullptr;
  B.statsN[f] = ks ? cloud->statsN : nullptr;
  B.count[f] = cloud->d_n;
  cloud->points3_valid = false; cloud->pn_valid = false;
  cloud->n_known = false;
  cloud->has_stats = ks;
}

int launch_frame_prep(nicp_context *ctx, const float *d_depth, const nicp_projector *proj, const nicp_stats_params *sp,
                      const float sensorOffset[16], int keepStats, nicp_cloud *cloud, int *d_index, const CamSet *cams) {
  PrepBatch B;
  memset(&B, 0, sizeof B);
  prep_batch_add(B, const_cast<float *>(d_depth), ctx->d_integral, cloud, keepStats != 0);
  int rc = launch_prep_set(ctx, B, proj, sp, sensorOffset, d_index, ctx->d_interval, cams);
  if (rc) return rc;
  ctx->lastRows = proj->rows;
  ctx->lastCols = proj->cols;
  return NICP_OK;
}

// n raw 16-bit frames already on the device (d_raw[f]) -> n clouds: depth conversion + the launch set above, in
// sub-batches of at most kMaxPrepBatch frames whose scratch (depth + integral image, 44 B/pixel/frame) stays L2 resident
int launch_raw_prep_batch(nicp_context *ctx, int n, const uint16_t *const *d_raw, int rawRows, int rawCols, float scale, int step,
                          float maxCov, const nicp_projector *proj, const nicp_stats_params *sp, const float sensorOffset[16],
                          int keepStats, nicp_cloud *const *clouds) {
  const size_t px = (size_t)proj->rows * proj->cols;
  if (n > ctx->batchSlots || px > ctx->batchPixels) {
    set_error("internal: batch prep scratch too small");
    return NICP_ERR_INVALID;
  }
  PrepBatch B;
  memset(&B, 0, sizeof B);
  for (int f = 0; f < n; f++) {
    prep_batch_add(B, ctx->d_bDepth + (size_t)f * ctx->batchPixels, ctx->d_bIntegral + (size_t)f * ctx->batchPixels * kIntegralCh,
                   clouds[f], keepStats != 0);
    B.raw[f] = d_raw[f];
  }
  const int outPx = (rawRows / step) * (rawCols / step);
  k_depth_convert<<<dim3((outPx + 255) / 256, n), 256, 0, ctx->stream>>>(B, rawRows, rawCols, scale, step, maxCov);
  NICP_CHECK_LAUNCH(ctx);
  return launch_prep_set(ctx, B, proj, sp, sensorOffset, nullptr, nullptr, nullptr);
}

// the same for n rig frames: d_raw[f * cams.n + i] = camera i of frame f on the device (rawRows[i] x rawCols[i]), proj = the
// composite image (rows = max width, cols = sum of heights); one conversion launch for every camera of every frame
int launch_rig_raw_prep_batch(nicp_context *ctx, int n, const uint16_t *const *d_raw, const int *rawRows, const int *rawCols,
                              float scale, int step, float maxCov, const nicp_projector *proj, const CamSet &cams,
                              const nicp_stats_params *sp, const float sensorOffset[16], int keepStats, nicp_cloud *const *clouds) {
  const size_t px = (size_t)proj->rows * proj->cols;
  if (n > ctx->batchSlots || px > ctx->batchPixels) {
    set_error("internal: batch prep scratch too small");
    return NICP_ERR_INVALID;
  }
  PrepBatch B;
  memset(&B, 0, sizeof B);
  RigFrames R;
  memset(&R, 0, sizeof R);
  R.nCams = cams.n;
  int maxHeight = 0;
  for (int i = 0; i < cams.n; i++) {
    R.rawRows[i] = rawRows[i];
    R.rawCols[i] = rawCols[i];
    R.width[i] = cams.width[i];
    R.height[i] = cams.height[i];
    R.colOff[i] = cams.colOff[i];
    if (cams.height[i] > maxHeight) maxHeight = cams.height[i];
  }
  for (int f = 0; f < n; f++) {
    prep_batch_add(B, ctx->d_bDepth + (size_t)f * ctx->batchPixels, ctx->d_bIntegral + (size_t)f * ctx->batchPixels * kIntegralCh,
                   clouds[f], keepStats != 0);
    R.depth[f] = B.depth[f];
    for (int i = 0; i < cams.n; i++) R.raw[f * cams.n + i] = d_raw[f * cams.n + i];
  }
  k_rig_depth_convert<<<dim3((maxHeight + 31) / 32, (proj->rows + 31) / 32, n * cams.n), dim3(32, 8), 0, ctx->stream>>>(
      R, proj->rows, proj->cols, scale, step, maxCov);
  NICP_CHECK_LAUNCH(ctx);
  return launch_prep_set(ctx, B, proj, sp, sensorOffset, nullptr, nullptr, &cams);
}

// ---------------------------------------------------------------------------------------------
// Stage-level StatsCalculatorIntegralImage::compute(normals, stats, points, indexImage) with its _intervalImage
// (statscalculatorintegralimage.cpp:14-82) and Point / NormalInformationMatrixCalculator::compute
// (informationmatrixcalculator.cpp:9-58): the virtuals of the boundary that take an arbitrary point vector + index
// image (any projector pose, merged clouds, ...), not a depth image.
// ---------------------------------------------------------------------------------------------
// PointIntegralImage::compute pass 1 from (index image, points): same row staging / sequential scan as k_integral_rows
__global__ void __launch_bounds__(256) k_integral_rows_indexed(const int *__restrict__ index, const float4 *__restrict__ points,
                                                               int rows, int cols, float *__restrict__ I) {
  extern __shared__ float sm[];  // [10][stride]
  const int stride = cols + 1;
  const int r = blockIdx.x;
  for (int c = threadIdx.x; c < cols; c += blockDim.x) {
    const int idx = index[(size_t)r * cols + c];
    float ch[kIntegralCh];
    if (idx < 0) {
#pragma unroll
      for (int k = 0; k < kIntegralCh; k++) ch[k] = 0.0f;
    } else {
      const float4 p = points[idx];
      ch[0] = 1.0f; ch[1] = p.x; ch[2] = p.y; ch[3] = p.z;
      ch[4] = fmul(p.x, p.x); ch[5] = fmul(p.x, p.y); ch[6] = fmul(p.x, p.z);
      ch[7] = fmul(p.y, p.y); ch[8] = fmul(p.y, p.z); ch[9] = fmul(p.z, p.z);
    }
#pragma unroll
    for (int k = 0; k < kIntegralCh; k++) sm[k * stride + c] = ch[k];
  }
  __syncthreads();
  if (threadIdx.x < kIntegralCh) {
    float *p = sm + threadIdx.x * stride;
    float v = p[0];
    for (int c = 1; c < cols; c++) { v = fadd(p[c], v); p[c] = v; }
  }
  __syncthreads();
  const size_t plane = (size_t)rows * cols;
  for (int k = 0; k < kIntegralCh; k++) {
    float *orow = I + k * plane + (size_t)r * cols;
    for (int c = threadIdx.x; c < cols; c += blockDim.x) orow[c] = sm[k * stride + c];
  }
}

// Stats() / Normal::Zero() defaults of every point (statscalculatorintegralimage.cpp:22-28)
__global__ void k_stats_defaults(int n, float4 *__restrict__ normals, float *__restrict__ stats16, float *__restrict__ eigvals,
                                 int *__restrict__ statsN, float *__restrict__ curvature) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  normals[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 *so = reinterpret_cast<float4 *>(stats16 + 16 * (size_t)i);
  so[0] = make_float4(1.f, 0.f, 0.f, 0.f);
  so[1] = make_float4(0.f, 1.f, 0.f, 0.f);
  so[2] = make_float4(0.f, 0.f, 1.f, 0.f);
  so[3] = make_float4(0.f, 0.f, 0.f, 1.f);
  eigvals[3 * (size_t)i] = eigvals[3 * (size_t)i + 1] = eigvals[3 * (size_t)i + 2] = 0.0f;
  statsN[i] = 0;
  curvature[i] = 0.0f;
}

__global__ void __launch_bounds__(256) k_stats_stage(const float *__restrict__ I, const int *__restrict__ index,
                                                     const int *__restrict__ interval, const float4 *__restrict__ points,
                                                     int rows, int cols, int n, StatsConsts sc, float4 *__restrict__ normals,
                                                     float *__restrict__ stats16, float *__restrict__ eigvals,
                                                     int *__restrict__ statsN, float *__restrict__ curvature) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = blockIdx.y * blockDim.y + threadIdx.y;
  if (c >= cols || r >= rows) return;
  const size_t pix = (size_t)r * cols + c;
  const int idx = index[pix], k = interval[pix];
  if (idx < 0 || idx >= n || k < 0) return;
  const float4 p = points[idx];
  float nx = 0.f, ny = 0.f, nz = 0.f, curv = 0.f, U[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, ev[3] = {0, 0, 0}, mu[3] = {0, 0, 0};
  int npts = 0;
  if (!stats_core(I, (size_t)rows * cols, rows, cols, r, c, k, sc, p.x, p.y, p.z, nx, ny, nz, curv, U, ev, mu, npts)) return;
  normals[idx] = make_float4(nx, ny, nz, 0.0f);
  float4 *so = reinterpret_cast<float4 *>(stats16 + 16 * (size_t)idx);
  so[0] = make_float4(U[0], U[1], U[2], 0.0f);
  so[1] = make_float4(U[3], U[4], U[5], 0.0f);
  so[2] = make_float4(U[6], U[7], U[8], 0.0f);
  so[3] = make_float4(mu[0], mu[1], mu[2], 1.0f);
  eigvals[3 * (size_t)idx] = ev[0];
  eigvals[3 * (size_t)idx + 1] = ev[1];
  eigvals[3 * (size_t)idx + 2] = ev[2];
  statsN[idx] = npts;
  curvature[idx] = curv;
}

__global__ void k_information_stage(int n, const float4 *__restrict__ normals, const float *__restrict__ stats16,
                                    const float *__restrict__ eigvals, const float *__restrict__ curvature, StatsConsts sc,
                                    float *__restrict__ omegaP6, float *__restrict__ omegaN6) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 nn = normals[i];
  const float *S = stats16 + 16 * (size_t)i;
  const float U[9] = {S[0], S[1], S[2], S[4], S[5], S[6], S[8], S[9], S[10]};
  const float ev[3] = {eigvals[3 * (size_t)i], eigvals[3 * (size_t)i + 1], eigvals[3 * (size_t)i + 2]};
  float OP[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, ON[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  information_core(nn.x, nn.y, nn.z, curvature[i], U, ev, sc, OP, ON);
  if (omegaP6) {
    float *o = omegaP6 + 6 * (size_t)i;
    o[0] = NM3(OP, 0, 0); o[1] = NM3(OP, 0, 1); o[2] = NM3(OP, 0, 2); o[3] = NM3(OP, 1, 1); o[4] = NM3(OP, 1, 2); o[5] = NM3(OP, 2, 2);
  }
  if (omegaN6) {
    float *o = omegaN6 + 6 * (size_t)i;
    o[0] = NM3(ON, 0, 0); o[1] = NM3(ON, 0, 1); o[2] = NM3(ON, 0, 2); o[3] = NM3(ON, 1, 1); o[4] = NM3(ON, 1, 2); o[5] = NM3(ON, 2, 2);
  }
}

static StatsConsts stage_consts(const nicp_stats_params *sp) {
  StatsConsts sc;
  memset(&sc, 0, sizeof sc);
  sc.minR = sp->min_image_radius;
  sc.maxR = sp->max_image_radius;
  sc.minPoints = sp->min_points;
  sc.curvThr = sp->curvature_threshold;
  sc.omegaCurvThr = sp->omega_curvature_threshold;
  for (int i = 0; i < 3; i++) {
    sc.flatP[i] = sp->flat_omega_p[i];
    sc.flatN[i] = sp->flat_omega_n[i];
    sc.nonflatN[i] = sp->nonflat_omega_n[i];
  }
  return sc;
}

// device buffers in, device buffers out; d_integral = [10][rows][cols] scratch
int launch_stats_stage(nicp_context *ctx, const float4 *d_points, int n, const int *d_index, const int *d_interval, int rows,
                       int cols, const nicp_stats_params *sp, float *d_integral, float4 *d_normals, float *d_stats16,
                       float *d_eigvals, int *d_statsN, float *d_curvature) {
  const size_t smem = (size_t)kIntegralCh * (cols + 1) * sizeof(float);
  if (smem > 200 * 1024) {
    set_error("image too wide for the row pass (%d columns)", cols);
    return NICP_ERR_INVALID;
  }
  if (smem > 48 * 1024) NICP_CUDA(cudaFuncSetAttribute(k_integral_rows_indexed, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_integral_rows_indexed<<<rows, 256, smem, ctx->stream>>>(d_index, d_points, rows, cols, d_integral);
  NICP_CHECK_LAUNCH(ctx);
  PrepBatch B;
  memset(&B, 0, sizeof B);
  B.n = 1;
  B.integral[0] = d_integral;
  k_integral_cols<<<dim3((cols + 63) / 64, kIntegralCh, 1), 64, 0, ctx->stream>>>(B, rows, cols);
  NICP_CHECK_LAUNCH(ctx);
  if (n > 0) {
    k_stats_defaults<<<(n + 255) / 256, 256, 0, ctx->stream>>>(n, d_normals, d_stats16, d_eigvals, d_statsN, d_curvature);
    NICP_CHECK_LAUNCH(ctx);
  }
  const StatsConsts sc = stage_consts(sp);
  k_stats_stage<<<dim3((cols + 31) / 32, (rows + 7) / 8), dim3(32, 8), 0, ctx->stream>>>(d_integral, d_index, d_interval, d_points, rows,
                                                                                         cols, n, sc, d_normals, d_stats16, d_eigvals,
                                                                                         d_statsN, d_curvature);
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

int launch_information_stage(nicp_context *ctx, int n, const float4 *d_normals, const float *d_stats16, const float *d_eigvals,
                             const float *d_curvature, const nicp_stats_params *sp, float *d_omegaP6, float *d_omegaN6) {
  if (n <= 0) return NICP_OK;
  k_information_stage<<<(n + 255) / 256, 256, 0, ctx->stream>>>(n, d_normals, d_stats16, d_eigvals, d_curvature, stage_consts(sp),
                                                                d_omegaP6, d_omegaN6);
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

// ---------------------------------------------------------------------------------------------
// PinholePointProjector::unProject stand-alone (arbitrary projector pose): row counts, then
// one CTA per row writes its points at (valid pixels in earlier rows) + (rank inside the row).
// ---------------------------------------------------------------------------------------------
__global__ void k_row_counts(const float *__restrict__ depth, int rows, int cols, float minD, float maxD,
                             int *__restrict__ rowCount) {
  __shared__ int s;
  if (threadIdx.x == 0) s = 0;
  __syncthreads();
  int r = blockIdx.x, cnt = 0;
  for (int c = threadIdx.x; c < cols; c += blockDim.x) {
    float d = depth[(size_t)r * cols + c];
    cnt += !(d < minD || d > maxD);
  }
  for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(&s, cnt);
  __syncthreads();
  if (threadIdx.x == 0) rowCount[r] = s;
}

__global__ void __launch_bounds__(256) k_unproject_rows(const float *__restrict__ depth, int rows, int cols, Affine iKRt,
                                                        float minD, float maxD, const int *__restrict__ rowCount,
                                                        float4 *__restrict__ points, int *__restrict__ index,
                                                        int *__restrict__ countOut) {
  __shared__ int sbase;
  __shared__ int warpTot[8];
  const int r = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) sbase = 0;
  __syncthreads();
  int part = 0;
  for (int i = threadIdx.x; i < r; i += blockDim.x) part += rowCount[i];
  for (int o = 16; o; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
  if (lane == 0 && part) atomicAdd(&sbase, part);
  __syncthreads();
  int base = sbase;
  if (r == rows - 1 && threadIdx.x == 0) *countOut = base + rowCount[r];
  for (int c0 = 0; c0 < cols; c0 += blockDim.x) {
    int c = c0 + threadIdx.x;
    float d = c < cols ? depth[(size_t)r * cols + c] : -1.0f;
    bool valid = c < cols && !(d < minD || d > maxD);
    unsigned m = __ballot_sync(0xffffffffu, valid);
    if (lane == 0) warpTot[warp] = __popc(m);
    __syncthreads();
    int off = base + __popc(m & ((1u << lane) - 1));
    int tot = 0;
    for (int w = 0; w < 8; w++) {
      if (w < warp) off += warpTot[w];
      tot += warpTot[w];
    }
    if (c < cols) {
      if (valid) {
        float x, y, z;
        xform_point(iKRt, fmul((float)c, d), fmul((float)r, d), d, x, y, z);
        points[off] = make_float4(x, y, z, 1.0f);
        if (index) index[(size_t)r * cols + c] = off;
      } else if (index) {
        index[(size_t)r * cols + c] = -1;
      }
    }
    base += tot;
    __syncthreads();
  }
}

int launch_unproject(nicp_context *ctx, const float *d_depth, int rows, int cols, const float iKRt[16], float minD,
                     float maxD, nicp_cloud *cloud, int *d_index) {
  cloud->points3_valid = false; cloud->pn_valid = false;
  int *rowCount = ctx->d_interval;  // scratch (rows ints)
  k_row_counts<<<rows, 256, 0, ctx->stream>>>(d_depth, rows, cols, minD, maxD, rowCount);
  NICP_CHECK_LAUNCH(ctx);
  k_unproject_rows<<<rows, 256, 0, ctx->stream>>>(d_depth, rows, cols, affine_from(iKRt), minD, maxD, rowCount,
                                                  cloud->points, d_index, cloud->d_n);
  NICP_CHECK_LAUNCH(ctx);
  cloud->n_known = false;
  cloud->has_stats = false;
  return NICP_OK;
}

__global__ void k_intervals(const float *__restrict__ depth, int n, float minD, float maxD, float ivx, float ivy,
                            int *__restrict__ interval) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float d = depth[i];
  if (d < minD || d > maxD) { interval[i] = -1; return; }
  float invd = fdiv(1.0f, d);
  float a = fmul(ivx, invd), b = fmul(ivy, invd);
  interval[i] = (a > b) ? (int)a : (int)b;
}

int launch_intervals(nicp_context *ctx, const float *d_depth, const nicp_projector *proj, float worldRadius,
                     int *d_interval) {
  const float *K = proj->K;
  float ivx = dot3(NM3(K, 0, 0), NM3(K, 0, 1), NM3(K, 0, 2), worldRadius, worldRadius, 0.0f);
  float ivy = dot3(NM3(K, 1, 0), NM3(K, 1, 1), NM3(K, 1, 2), worldRadius, worldRadius, 0.0f);
  int n = proj->rows * proj->cols;
  k_intervals<<<(n + 255) / 256, 256, 0, ctx->stream>>>(d_depth, n, proj->min_distance, proj->max_distance, ivx, ivy,
                                                        d_interval);
  NICP_CHECK_LAUNCH(ctx);
  return NICP_OK;
}

// Cloud::transformInPlace on an existing device cloud
__global__ void k_cloud_transform(int capacity, const int *__restrict__ nPtr, Affine M, float4 *__restrict__ points,
                                  float4 *__restrict__ normals, float4 *__restrict__ omega, float *__restrict__ stats16) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= *nPtr || i >= capacity) return;
  float M16[16];
  mat4_identity(M16);
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 4; c++) NM4(M16, r, c) = M.r[r][c];
  float4 p = points[i], nn = normals[i];
  float x, y, z;
  xform_point(M, p.x, p.y, p.z, x, y, z);
  points[i] = make_float4(x, y, z, 1.0f);
  xform_normal(M, nn.x, nn.y, nn.z, x, y, z);
  normals[i] = make_float4(x, y, z, nn.w);
  float4 o0 = omega[3 * (size_t)i], o1 = omega[3 * (size_t)i + 1], o2 = omega[3 * (size_t)i + 2];
  float P6[6], N6[6];
  omega_unpack(o0, o1, o2, P6, N6);
  float OP[9] = {P6[0], P6[1], P6[2], P6[1], P6[3], P6[4], P6[2], P6[4], P6[5]};
  float ON[9] = {N6[0], N6[1], N6[2], N6[1], N6[3], N6[4], N6[2], N6[4], N6[5]};
  float tp[9], tn[9];
  rotate_sym(M16, OP, tp);
  rotate_sym(M16, ON, tn);
  {
    const float Q6[6] = {NM3(tp, 0, 0), NM3(tp, 0, 1), NM3(tp, 0, 2), NM3(tp, 1, 1), NM3(tp, 1, 2), NM3(tp, 2, 2)};
    const float R6[6] = {NM3(tn, 0, 0), NM3(tn, 0, 1), NM3(tn, 0, 2), NM3(tn, 1, 1), NM3(tn, 1, 2), NM3(tn, 2, 2)};
    const Omega3 w = omega_pack(Q6, R6);
    omega[3 * (size_t)i + 0] = w.o0;
    omega[3 * (size_t)i + 1] = w.o1;
    omega[3 * (size_t)i + 2] = w.o2;
  }
  if (stats16) {
    float *S = stats16 + 16 * (size_t)i;
    float o[16];
    for (int cc = 0; cc < 4; cc++)
      for (int rr = 0; rr < 4; rr++)
        NM4(o, rr, cc) = dot4(NM4(M16, rr, 0), NM4(M16, rr, 1), NM4(M16, rr, 2), NM4(M16, rr, 3), NM4(S, 0, cc),
                              NM4(S, 1, cc), NM4(S, 2, cc), NM4(S, 3, cc));
    for (int k = 0; k < 16; k++) S[k] = o[k];
  }
}

// Cloud::add (cloud.cpp:145-171): dst[nDst + i] = T * src[i]
__global__ void k_cloud_append(int srcCapacity, const int *__restrict__ srcN, const int *__restrict__ dstN, int dstCapacity,
                               Affine M, int identity, const float4 *__restrict__ sp, const float4 *__restrict__ sn,
                               const float4 *__restrict__ so, float4 *__restrict__ dp, float4 *__restrict__ dn,
                               float4 *__restrict__ dom) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= *srcN || i >= srcCapacity) return;
  const size_t o = (size_t)*dstN + i;
  if (o >= (size_t)dstCapacity) return;
  float4 p = sp[i], nn = sn[i];
  float4 o0 = so[3 * (size_t)i], o1 = so[3 * (size_t)i + 1], o2 = so[3 * (size_t)i + 2];
  if (!identity) {
    float M16[16];
    mat4_identity(M16);
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 4; c++) NM4(M16, r, c) = M.r[r][c];
    float x, y, z;
    xform_point(M, p.x, p.y, p.z, x, y, z);
    p = make_float4(x, y, z, 1.0f);
    xform_normal(M, nn.x, nn.y, nn.z, x, y, z);
    nn = make_float4(x, y, z, nn.w);
    float P6[6], N6[6];
    omega_unpack(o0, o1, o2, P6, N6);
    float OP[9] = {P6[0], P6[1], P6[2], P6[1], P6[3], P6[4], P6[2], P6[4], P6[5]};
    float ON[9] = {N6[0], N6[1], N6[2], N6[1], N6[3], N6[4], N6[2], N6[4], N6[5]};
    float tp[9], tn[9];
    rotate_sym(M16, OP, tp);
    rotate_sym(M16, ON, tn);
    const float Q6[6] = {NM3(tp, 0, 0), NM3(tp, 0, 1), NM3(tp, 0, 2), NM3(tp, 1, 1), NM3(tp, 1, 2), NM3(tp, 2, 2)};
    const float R6[6] = {NM3(tn, 0, 0), NM3(tn, 0, 1), NM3(tn, 0, 2), NM3(tn, 1, 1), NM3(tn, 1, 2), NM3(tn, 2, 2)};
    const Omega3 w = omega_pack(Q6, R6);
    o0 = w.o0;
    o1 = w.o1;
    o2 = w.o2;
  }
  dp[o] = p;
  dn[o] = nn;
  dom[3 * o] = o0;
  dom[3 * o + 1] = o1;
  dom[3 * o + 2] = o2;
}
__global__ void k_add_count(int *dstN, const int *srcN, int dstCapacity) {
  int n = *dstN + *srcN;
  *dstN = n > dstCapacity ? dstCapacity : n;
}

int launch_cloud_append(nicp_context *ctx, nicp_cloud *dst, const nicp_cloud *src, const float T[16]) {
  dst->points3_valid = false; dst->pn_valid = false;
  float m[16];
  for (int i = 0; i < 16; i++) m[i] = T[i];
  fix_last_row(m);
  k_cloud_append<<<(src->capacity + 255) / 256, 256, 0, ctx->stream>>>(src->capacity, src->d_n, dst->d_n, dst->capacity,
                                                                      affine_from(m), is_identity16(m) ? 1 : 0, src->points,
                                                                      src->normals, src->omega, dst->points, dst->normals,
                                                                      dst->omega);
  NICP_CHECK_LAUNCH(ctx);
  int rcg = launch_gauss_append(ctx, dst, src, T);
  if (rcg) return rcg;
  k_add_count<<<1, 1, 0, ctx->stream>>>(dst->d_n, src->d_n, dst->capacity);
  NICP_CHECK_LAUNCH(ctx);
  dst->n_known = false;
  dst->has_stats = false;
  return NICP_OK;
}

int launch_cloud_transform(nicp_context *ctx, nicp_cloud *cloud, const float T[16]) {
  float m[16];
  for (int i = 0; i < 16; i++) m[i] = T[i];
  fix_last_row(m);
  if (is_identity16(m)) return NICP_OK;
  cloud->points3_valid = false; cloud->pn_valid = false;
  k_cloud_transform<<<(cloud->capacity + 255) / 256, 256, 0, ctx->stream>>>(
      cloud->capacity, cloud->d_n, affine_from(m), cloud->points, cloud->normals, cloud->omega,
      cloud->has_stats ? cloud->stats16 : nullptr);
  NICP_CHECK_LAUNCH(ctx);
  if (cloud->has_gauss) return launch_gauss_transform(ctx, cloud, nullptr, 0, cloud->d_n, cloud->capacity, T);
  return NICP_OK;
}

}  // namespace nicp

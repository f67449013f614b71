/*
 * pwn_oracle.c -- CPU restatement of the pwn_core NICP hot path (see pwn_oracle.h header:
 * TEST INFRASTRUCTURE ONLY; pinned against the reference's own sources except for
 * Eigen's numerical kernels, see pwn_oracle.h).
 *
 * Build (verification flavour, canonical float32 evaluation order, no FMA contraction):
 *     gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC pwn_oracle.c -lm
 * Build (performance flavour, the reference's own flags, /root/reference/CMakeLists.txt:135,145,171):
 *     gcc -O3 -march=native -fopenmp -shared -fPIC pwn_oracle.c -lm
 *
 * Every function cites the reference file:line (relative to
 * /root/reference/g2o_frontend/pwn_core/) it follows.
 */
#include "pwn_oracle.h"
#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define M4(m, r, c) ((m)[(c) * 4 + (r)])
#define M3(m, r, c) ((m)[(c) * 3 + (r)])
#define M6(m, r, c) ((m)[(c) * 6 + (r)])

/* ------------------------------------------------------------------------------------------
 * canonical small-matrix arithmetic (SURVEY.md Appendix A1: Eigen's order is implicit, the
 * oracle fixes ((a0*b0 + a1*b1) + a2*b2) + a3*b3)
 * ---------------------------------------------------------------------------------------- */
static inline float dot3(float a0, float a1, float a2, float b0, float b1, float b2) {
  return (a0 * b0 + a1 * b1) + a2 * b2;
}
static inline float dot4(float a0, float a1, float a2, float a3, float b0, float b1, float b2, float b3) {
  return ((a0 * b0 + a1 * b1) + a2 * b2) + a3 * b3;
}
/* rows 0..2 of (4x4 matrix) * (x,y,z,w) */
static inline void xform3(const float *m, float x, float y, float z, float w, float out[3]) {
  for (int i = 0; i < 3; i++) out[i] = dot4(M4(m, i, 0), M4(m, i, 1), M4(m, i, 2), M4(m, i, 3), x, y, z, w);
}
static void mat4_mul(const float *A, const float *B, float *C) {
  float t[16];
  for (int c = 0; c < 4; c++)
    for (int r = 0; r < 4; r++)
      M4(t, r, c) = dot4(M4(A, r, 0), M4(A, r, 1), M4(A, r, 2), M4(A, r, 3), M4(B, 0, c), M4(B, 1, c), M4(B, 2, c), M4(B, 3, c));
  memcpy(C, t, sizeof t);
}
static void mat4_identity(float *m) {
  memset(m, 0, 16 * sizeof(float));
  m[0] = m[5] = m[10] = m[15] = 1.0f;
}
static void fix_last_row(float *T) { M4(T, 3, 0) = 0.f; M4(T, 3, 1) = 0.f; M4(T, 3, 2) = 0.f; M4(T, 3, 3) = 1.f; }

/* ------------------------------------------------------------------------------------------
 * pwn_static.cpp
 * ---------------------------------------------------------------------------------------- */
/* DepthImage_convert_16UC1_to_32FC1, pwn_static.cpp:54-68 */
void orc_depth_u16_to_f32(const uint16_t *src, int n, float scale, float *dst) {
  for (int i = 0; i < n; i++) dst[i] = src[i] ? scale * (float)src[i] : 0.0f;
}
/* DepthImage_convert_32FC1_to_16UC1, pwn_static.cpp:38-52 */
void orc_depth_f32_to_u16(const float *src, int n, float scale, uint16_t *dst) {
  for (int i = 0; i < n; i++) dst[i] = (src[i] < FLT_MAX) ? (uint16_t)(scale * src[i]) : 0;
}
/* DepthImage_scale, pwn_static.cpp:5-36 */
void orc_depth_scale(const float *src, int rows, int cols, int step, float maxDepthCov, float *dst) {
  int drows = rows / step, dcols = cols / step;
  for (int r = 0; r < drows; r++)
    for (int c = 0; c < dcols; c++) {
      float acc = 0, acc2 = 0;
      int np = 0;
      int sr = r * step, sc = c * step;
      dst[r * dcols + c] = 0.0f;
      for (int i = 0; i < step; i++)
        for (int j = 0; j < step; j++)
          if (sr + i < rows && sc + j < cols) {
            float f = src[(sr + i) * cols + sc + j];
            acc += f;
            acc2 += f * f;
            np += f > 0;
          }
      if (np) {
        float mu = acc / np;
        float sigma = acc2 / np - mu * mu;
        if (sigma > maxDepthCov) continue;
        dst[r * dcols + c] = mu;
      }
    }
}

/* ------------------------------------------------------------------------------------------
 * bm_se3.h
 * ---------------------------------------------------------------------------------------- */
/* quat2mat bm_se3.h:9-21, v2t :36-43 */
void orc_v2t(const float v[6], float T[16]) {
  float qx = v[3], qy = v[4], qz = v[5];
  float qw = sqrtf(1.f - ((qx * qx + qy * qy) + qz * qz));
  mat4_identity(T);
  M4(T, 0, 0) = qw * qw + qx * qx - qy * qy - qz * qz;
  M4(T, 0, 1) = 2 * (qx * qy - qw * qz);
  M4(T, 0, 2) = 2 * (qx * qz + qw * qy);
  M4(T, 1, 0) = 2 * (qx * qy + qz * qw);
  M4(T, 1, 1) = qw * qw - qx * qx + qy * qy - qz * qz;
  M4(T, 1, 2) = 2 * (qy * qz - qx * qw);
  M4(T, 2, 0) = 2 * (qx * qz - qy * qw);
  M4(T, 2, 1) = 2 * (qy * qz + qx * qw);
  M4(T, 2, 2) = qw * qw - qx * qx - qy * qy + qz * qz;
  M4(T, 0, 3) = v[0];
  M4(T, 1, 3) = v[1];
  M4(T, 2, 3) = v[2];
}
/* mat2quat bm_se3.h:24-34 (Eigen::Quaternion(R), normalize, sign), t2v :45-52 */
void orc_t2v(const float T[16], float v[6]) {
  float q[4]; /* x y z w */
  float t = (M4(T, 0, 0) + M4(T, 1, 1)) + M4(T, 2, 2);
  if (t > 0.f) {
    t = sqrtf(t + 1.0f);
    q[3] = 0.5f * t;
    t = 0.5f / t;
    q[0] = (M4(T, 2, 1) - M4(T, 1, 2)) * t;
    q[1] = (M4(T, 0, 2) - M4(T, 2, 0)) * t;
    q[2] = (M4(T, 1, 0) - M4(T, 0, 1)) * t;
  } else {
    int i = 0;
    if (M4(T, 1, 1) > M4(T, 0, 0)) i = 1;
    if (M4(T, 2, 2) > M4(T, i, i)) i = 2;
    int j = (i + 1) % 3, k = (j + 1) % 3;
    t = sqrtf(M4(T, i, i) - M4(T, j, j) - M4(T, k, k) + 1.0f);
    q[i] = 0.5f * t;
    t = 0.5f / t;
    q[3] = (M4(T, k, j) - M4(T, j, k)) * t;
    q[j] = (M4(T, j, i) + M4(T, i, j)) * t;
    q[k] = (M4(T, k, i) + M4(T, i, k)) * t;
  }
  float nrm = sqrtf(((q[0] * q[0] + q[1] * q[1]) + q[2] * q[2]) + q[3] * q[3]);
  for (int i = 0; i < 4; i++) q[i] = q[i] / nrm;
  v[0] = M4(T, 0, 3);
  v[1] = M4(T, 1, 3);
  v[2] = M4(T, 2, 3);
  if (q[3] < 0) { v[3] = -q[0]; v[4] = -q[1]; v[5] = -q[2]; }
  else          { v[3] =  q[0]; v[4] =  q[1]; v[5] =  q[2]; }
}
/* Eigen Isometry3f::inverse(): R' = R^T, t' = -(R^T t) */
void orc_iso_inverse(const float T[16], float Ti[16]) {
  float o[16];
  mat4_identity(o);
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) M4(o, r, c) = M4(T, c, r);
  for (int r = 0; r < 3; r++)
    M4(o, r, 3) = -dot3(M4(o, r, 0), M4(o, r, 1), M4(o, r, 2), M4(T, 0, 3), M4(T, 1, 3), M4(T, 2, 3));
  memcpy(Ti, o, sizeof o);
}
/* Isometry * Isometry: R = Ra Rb, t = Ra tb + ta (the full 4x4 product; zeros add exactly) */
void orc_iso_mul(const float A[16], const float B[16], float C[16]) {
  float o[16];
  mat4_identity(o);
  for (int r = 0; r < 3; r++) {
    for (int c = 0; c < 3; c++)
      M4(o, r, c) = dot3(M4(A, r, 0), M4(A, r, 1), M4(A, r, 2), M4(B, 0, c), M4(B, 1, c), M4(B, 2, c));
    M4(o, r, 3) = dot3(M4(A, r, 0), M4(A, r, 1), M4(A, r, 2), M4(B, 0, 3), M4(B, 1, 3), M4(B, 2, 3)) + M4(A, r, 3);
  }
  memcpy(C, o, sizeof o);
}

/* ------------------------------------------------------------------------------------------
 * PinholePointProjector
 * ---------------------------------------------------------------------------------------- */
/* Eigen 3x3 inverse (cofactors / determinant, Eigen/src/LU/Inverse.h compute_inverse<.,.,3>) */
static void mat3_inverse(const float *m, float *inv) {
#define COF(i, j) (M3(m, ((i) + 1) % 3, ((j) + 1) % 3) * M3(m, ((i) + 2) % 3, ((j) + 2) % 3) - \
                   M3(m, ((i) + 1) % 3, ((j) + 2) % 3) * M3(m, ((i) + 2) % 3, ((j) + 1) % 3))
  float c00 = COF(0, 0), c10 = COF(1, 0), c20 = COF(2, 0);
  float det = (c00 * M3(m, 0, 0) + c10 * M3(m, 1, 0)) + c20 * M3(m, 2, 0);
  float invdet = 1.0f / det;
  M3(inv, 0, 0) = c00 * invdet;
  M3(inv, 0, 1) = c10 * invdet;
  M3(inv, 0, 2) = c20 * invdet;
  M3(inv, 1, 0) = COF(0, 1) * invdet;
  M3(inv, 1, 1) = COF(1, 1) * invdet;
  M3(inv, 1, 2) = COF(2, 1) * invdet;
  M3(inv, 2, 0) = COF(0, 2) * invdet;
  M3(inv, 2, 1) = COF(1, 2) * invdet;
  M3(inv, 2, 2) = COF(2, 2) * invdet;
#undef COF
}
/* PinholePointProjector::_updateMatrices, pinholepointprojector.cpp:17-31 */
void orc_update_matrices(const float K[9], const float T[16], float KRt[16], float iKRt[16]) {
  float t[16], iK[9];
  orc_iso_inverse(T, t);
  mat3_inverse(K, iK);
  mat4_identity(KRt);
  mat4_identity(iKRt);
  for (int r = 0; r < 3; r++) {
    for (int c = 0; c < 3; c++) {
      M4(KRt, r, c) = dot3(M3(K, r, 0), M3(K, r, 1), M3(K, r, 2), M4(t, 0, c), M4(t, 1, c), M4(t, 2, c));
      M4(iKRt, r, c) = dot3(M4(T, r, 0), M4(T, r, 1), M4(T, r, 2), M3(iK, 0, c), M3(iK, 1, c), M3(iK, 2, c));
    }
    M4(KRt, r, 3) = dot3(M3(K, r, 0), M3(K, r, 1), M3(K, r, 2), M4(t, 0, 3), M4(t, 1, 3), M4(t, 2, 3));
    M4(iKRt, r, 3) = M4(T, r, 3);
  }
}
/* unProject pinholepointprojector.cpp:68-91, _unProject pinholepointprojector.h:246-251 */
int orc_unproject(const float *depth, int rows, int cols, const float iKRt[16], float minD, float maxD,
                  float *points, int *index) {
  int count = 0;
  for (int r = 0; r < rows; r++)
    for (int c = 0; c < cols; c++) {
      float d = depth[r * cols + c];
      if (d < minD || d > maxD) { index[r * cols + c] = -1; continue; }
      float *p = points + 4 * count;
      xform3(iKRt, c * d, r * d, d, 1.0f, p);
      p[3] = 1.0f;
      index[r * cols + c] = count++;
    }
  return count;
}
/* projectIntervals pinholepointprojector.cpp:135-147, _projectInterval .h:264-274 */
void orc_project_intervals(const float *depth, int rows, int cols, const float K[9], float minD, float maxD,
                           float worldRadius, int *interval) {
  /* p = K * (worldRadius, worldRadius, 0) */
  float p0 = dot3(M3(K, 0, 0), M3(K, 0, 1), M3(K, 0, 2), worldRadius, worldRadius, 0.0f);
  float p1 = dot3(M3(K, 1, 0), M3(K, 1, 1), M3(K, 1, 2), worldRadius, worldRadius, 0.0f);
  for (int i = 0; i < rows * cols; i++) {
    float d = depth[i];
    if (d < minD || d > maxD) { interval[i] = -1; continue; }
    float s = 1.0f / d;
    float a = p0 * s, b = p1 * s;
    interval[i] = (a > b) ? (int)a : (int)b;
  }
}
/* project pinholepointprojector.cpp:33-66, _project pinholepointprojector.h:224-233 */
void orc_project(const float *points, int n, int rows, int cols, const float KRt[16], float minD, float maxD,
                 int *index, float *depth) {
  for (int i = 0; i < rows * cols; i++) { depth[i] = FLT_MAX; index[i] = -1; }
  for (int i = 0; i < n; i++) {
    const float *p = points + 4 * i;
    float ip[3];
    xform3(KRt, p[0], p[1], p[2], p[3], ip);
    float d = ip[2];
    if (d < minD || d > maxD) continue;
    float s = 1.0f / d;
    float fx = roundf(ip[0] * s), fy = roundf(ip[1] * s);
    if (!(fx >= 0.0f && fx < (float)cols && fy >= 0.0f && fy < (float)rows)) continue;
    int x = (int)fx, y = (int)fy;
    float *od = &depth[y * cols + x];
    if (!*od || *od > d) { *od = d; index[y * cols + x] = i; }
  }
}

/* ------------------------------------------------------------------------------------------
 * PointIntegralImage::compute, pointintegralimage.cpp:7-44; PointAccumulator += Point,
 * pointaccumulator.h:56-59.  10 unique channels (the 4x4 outer product of (x,y,z,1) is
 * bitwise symmetric and its last row/col equals the 4-sum): n,x,y,z,xx,xy,xz,yy,yz,zz.
 * Order: scatter, then sequential prefix along image-x inside every row ("fill by column" of
 * the transposed Eigen matrix), then sequential prefix along image-y inside every column.
 * ---------------------------------------------------------------------------------------- */
void orc_integral_image(const int *index, const float *points, int rows, int cols, float *I) {
#pragma omp parallel for
  for (int r = 0; r < rows; r++)
    for (int c = 0; c < cols; c++) {
      float *a = I + 10 * ((size_t)r * cols + c);
      int idx = index[r * cols + c];
      if (idx < 0) { for (int k = 0; k < 10; k++) a[k] = 0.0f; continue; }
      const float *p = points + 4 * idx;
      a[0] = 1.0f; a[1] = p[0]; a[2] = p[1]; a[3] = p[2];
      a[4] = p[0] * p[0]; a[5] = p[0] * p[1]; a[6] = p[0] * p[2];
      a[7] = p[1] * p[1]; a[8] = p[1] * p[2]; a[9] = p[2] * p[2];
    }
#pragma omp parallel for
  for (int r = 0; r < rows; r++)
    for (int c = 1; c < cols; c++) {
      float *a = I + 10 * ((size_t)r * cols + c);
      const float *b = a - 10;
      for (int k = 0; k < 10; k++) a[k] += b[k];
    }
#pragma omp parallel for
  for (int c = 0; c < cols; c++)
    for (int r = 1; r < rows; r++) {
      float *a = I + 10 * ((size_t)r * cols + c);
      const float *b = a - 10 * (size_t)cols;
      for (int k = 0; k < 10; k++) a[k] += b[k];
    }
}

static inline int clampi(int v, int lo, int hi) { v = v < lo ? lo : v; return v > hi ? hi : v; }

/* PointIntegralImage::getRegion, pointintegralimage.cpp:53-66 (x = image column, y = image row) */
static void get_region(const float *I, int rows, int cols, int xmin, int xmax, int ymin, int ymax, float acc[10]) {
  xmin = clampi(xmin - 1, 0, cols - 1);
  xmax = clampi(xmax - 1, 0, cols - 1);
  ymin = clampi(ymin - 1, 0, rows - 1);
  ymax = clampi(ymax - 1, 0, rows - 1);
  const float *a = I + 10 * ((size_t)ymax * cols + xmax);
  const float *b = I + 10 * ((size_t)ymin * cols + xmin);
  const float *c = I + 10 * ((size_t)ymax * cols + xmin);
  const float *d = I + 10 * ((size_t)ymin * cols + xmax);
  for (int k = 0; k < 10; k++) acc[k] = ((a[k] + b[k]) - c[k]) - d[k];
}

/* ------------------------------------------------------------------------------------------
 * Eigen::SelfAdjointEigenSolver<Matrix3f>::computeDirect, Eigen 3.2.x closed form
 * (SURVEY.md Appendix A4).  C column-major 3x3 symmetric; evals ascending; evecs column-major.
 * ---------------------------------------------------------------------------------------- */
static inline void cross3(const float *a, const float *b, float *o) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}
static inline float sqnorm3(const float *a) { return (a[0] * a[0] + a[1] * a[1]) + a[2] * a[2]; }
static void unit_orthogonal(const float *s, float *o) {
  /* Eigen unitOrthogonal for 3-vectors; isMuchSmallerThan(a,b): |a| <= |b| * 1e-5 */
  const float prec = 1e-5f;
  if (!(fabsf(s[0]) <= fabsf(s[2]) * prec) || !(fabsf(s[1]) <= fabsf(s[2]) * prec)) {
    float invnm = 1.0f / sqrtf(s[0] * s[0] + s[1] * s[1]);
    o[0] = -s[1] * invnm; o[1] = s[0] * invnm; o[2] = 0.0f;
  } else {
    float invnm = 1.0f / sqrtf(s[1] * s[1] + s[2] * s[2]);
    o[0] = 0.0f; o[1] = -s[2] * invnm; o[2] = s[1] * invnm;
  }
}
/* devtrig != 0: atan2 / cos / sin evaluated in float64 and rounded to float32, as the CUDA path does (eigen_variant 2);
 * otherwise the libm float functions of the reference build */
static void eigen3_32(const float C[9], float evals[3], float evecs[9], int devtrig) {
  const float eps = FLT_EPSILON;
  float scale = 0.0f;
  for (int i = 0; i < 9; i++) { float a = fabsf(C[i]); if (a > scale) scale = a; }
  float m[9];
  for (int i = 0; i < 9; i++) m[i] = C[i] / scale;
  /* computeRoots */
  const float s_inv3 = 1.0f / 3.0f;
  const float s_sqrt3 = sqrtf(3.0f);
  float m00 = M3(m, 0, 0), m11 = M3(m, 1, 1), m22 = M3(m, 2, 2);
  float m10 = M3(m, 1, 0), m20 = M3(m, 2, 0), m21 = M3(m, 2, 1);
  float c0 = m00 * m11 * m22 + 2.0f * m10 * m20 * m21 - m00 * m21 * m21 - m11 * m20 * m20 - m22 * m10 * m10;
  float c1 = m00 * m11 - m10 * m10 + m00 * m22 - m20 * m20 + m11 * m22 - m21 * m21;
  float c2 = m00 + m11 + m22;
  float c2_over_3 = c2 * s_inv3;
  float a_over_3 = (c1 - c2 * c2_over_3) * s_inv3;
  if (a_over_3 > 0.0f) a_over_3 = 0.0f;
  float half_b = 0.5f * (c0 + c2_over_3 * (2.0f * c2_over_3 * c2_over_3 - c1));
  float q = half_b * half_b + a_over_3 * a_over_3 * a_over_3;
  if (q > 0.0f) q = 0.0f;
  float rho = sqrtf(-a_over_3);
  float theta, cos_theta, sin_theta;
  if (devtrig) {
    theta = (float)atan2((double)sqrtf(-q), (double)half_b) * s_inv3;
    cos_theta = (float)cos((double)theta);
    sin_theta = (float)sin((double)theta);
  } else {
    theta = atan2f(sqrtf(-q), half_b) * s_inv3;
    cos_theta = cosf(theta);
    sin_theta = sinf(theta);
  }
  float r0 = c2_over_3 + 2.0f * rho * cos_theta;
  float r1 = c2_over_3 - rho * (cos_theta + s_sqrt3 * sin_theta);
  float r2 = c2_over_3 - rho * (cos_theta - s_sqrt3 * sin_theta);
  float tsw;
  if (r0 >= r1) { tsw = r0; r0 = r1; r1 = tsw; }
  if (r1 >= r2) {
    tsw = r1; r1 = r2; r2 = tsw;
    if (r0 >= r1) { tsw = r0; r0 = r1; r1 = tsw; }
  }
  float ev[3] = {r0, r1, r2};
  const float safeNorm2 = eps * eps;
  if ((ev[2] - ev[0]) <= eps) {
    memset(evecs, 0, 9 * sizeof(float));
    evecs[0] = evecs[4] = evecs[8] = 1.0f;
  } else {
    float d0 = ev[2] - ev[1];
    float d1 = ev[1] - ev[0];
    int k = d0 > d1 ? 2 : 0;
    d0 = d0 > d1 ? d1 : d0;
    float tmp[9];
    memcpy(tmp, m, sizeof tmp);
    tmp[0] -= ev[k]; tmp[4] -= ev[k]; tmp[8] -= ev[k];
    float row0[3] = {M3(tmp, 0, 0), M3(tmp, 0, 1), M3(tmp, 0, 2)};
    float row1[3] = {M3(tmp, 1, 0), M3(tmp, 1, 1), M3(tmp, 1, 2)};
    float row2[3] = {M3(tmp, 2, 0), M3(tmp, 2, 1), M3(tmp, 2, 2)};
    float cr[3], n;
    float uk[3], u1[3], ul[3];
    cross3(row0, row1, cr);
    n = sqnorm3(cr);
    if (!(n > safeNorm2)) {
      cross3(row0, row2, cr);
      n = sqnorm3(cr);
      if (!(n > safeNorm2)) {
        cross3(row1, row2, cr);
        n = sqnorm3(cr);
        if (!(n > safeNorm2)) {
          /* NumericalIssue: Eigen returns with eigenvectors left untouched (uninitialised);
             the oracle defines them as identity */
          memset(evecs, 0, 9 * sizeof(float));
          evecs[0] = evecs[4] = evecs[8] = 1.0f;
          for (int i = 0; i < 3; i++) evals[i] = ev[i] * scale;
          return;
        }
      }
    }
    { float sn = sqrtf(n); uk[0] = cr[0] / sn; uk[1] = cr[1] / sn; uk[2] = cr[2] / sn; }
    memcpy(tmp, m, sizeof tmp);
    tmp[0] -= ev[1]; tmp[4] -= ev[1]; tmp[8] -= ev[1];
    if (d0 <= eps) {
      unit_orthogonal(uk, u1);
    } else {
      float r0v[3] = {M3(tmp, 0, 0), M3(tmp, 0, 1), M3(tmp, 0, 2)};
      float r1v[3] = {M3(tmp, 1, 0), M3(tmp, 1, 1), M3(tmp, 1, 2)};
      float r2v[3] = {M3(tmp, 2, 0), M3(tmp, 2, 1), M3(tmp, 2, 2)};
      float nr0 = sqrtf(sqnorm3(r0v));
      float r0n[3] = {r0v[0] / nr0, r0v[1] / nr0, r0v[2] / nr0};
      int have = 1;
      cross3(uk, r0n, cr);
      n = sqnorm3(cr);
      if (!(n > safeNorm2)) {
        cross3(uk, r1v, cr);
        n = sqnorm3(cr);
        if (!(n > safeNorm2)) {
          cross3(uk, r2v, cr);
          n = sqnorm3(cr);
          if (!(n > safeNorm2)) { unit_orthogonal(uk, u1); have = 0; }
        }
      }
      if (have) { float sn = sqrtf(n); u1[0] = cr[0] / sn; u1[1] = cr[1] / sn; u1[2] = cr[2] / sn; }
      /* make sure u1 is orthogonal to uk: u1 = normalize(uk x (u1 x uk)) */
      float t1[3], t2[3];
      cross3(u1, uk, t1);
      cross3(uk, t1, t2);
      float sn = sqrtf(sqnorm3(t2));
      u1[0] = t2[0] / sn; u1[1] = t2[1] / sn; u1[2] = t2[2] / sn;
    }
    {
      float t[3];
      cross3(uk, u1, t);
      float sn = sqrtf(sqnorm3(t));
      ul[0] = t[0] / sn; ul[1] = t[1] / sn; ul[2] = t[2] / sn;
    }
    int l = (k == 2) ? 0 : 2;
    for (int i = 0; i < 3; i++) { M3(evecs, i, k) = uk[i]; M3(evecs, i, 1) = u1[i]; M3(evecs, i, l) = ul[i]; }
  }
  for (int i = 0; i < 3; i++) evals[i] = ev[i] * scale;
}
void orc_eigen3(const float C[9], float evals[3], float evecs[9]) { eigen3_32(C, evals, evecs, 0); }
void orc_eigen3_devtrig(const float C[9], float evals[3], float evecs[9]) { eigen3_32(C, evals, evecs, 1); }

/* ------------------------------------------------------------------------------------------
 * The same call as Eigen >= 3.3 implements it (recalled from Eigen/src/Eigenvalues/SelfAdjointEigenSolver.h of 3.3.x,
 * direct_selfadjoint_eigenvalues<SolverType, 3, false>; UNPINNED like the 3.2 variant above: no Eigen in this image).
 * Differences from 3.2: the matrix is shifted by trace / 3 before scaling, the roots come out of computeRoots already
 * sorted, and the eigenvectors are taken from the kernel of (A - lambda I) through the cross products of its most
 * significant column (extract_kernel) instead of the row cross products with a safeNorm test.  The reference pins no
 * Eigen version (CMakeLists.txt:158 asks for >= 3.1.2), so which of the two its users run depends on their distribution;
 * tests/test_oracle.py and DESIGN.md section 2 report how far apart the two are on the bench inputs.
 * ---------------------------------------------------------------------------------------- */
static void extract_kernel33(const float *mat /* column-major 3x3 */, float *res, float *representative) {
  int i0 = 0;
  float best = fabsf(M3(mat, 0, 0));
  for (int i = 1; i < 3; i++)
    if (fabsf(M3(mat, i, i)) > best) { best = fabsf(M3(mat, i, i)); i0 = i; }
  const int i1 = (i0 + 1) % 3, i2 = (i0 + 2) % 3;
  float col0[3] = {M3(mat, 0, i0), M3(mat, 1, i0), M3(mat, 2, i0)};
  float col1[3] = {M3(mat, 0, i1), M3(mat, 1, i1), M3(mat, 2, i1)};
  float col2[3] = {M3(mat, 0, i2), M3(mat, 1, i2), M3(mat, 2, i2)};
  for (int i = 0; i < 3; i++) representative[i] = col0[i];
  float c0[3], c1[3];
  cross3(col0, col1, c0);
  cross3(col0, col2, c1);
  float n0 = sqnorm3(c0), n1 = sqnorm3(c1);
  if (n0 > n1) { float sn = sqrtf(n0); for (int i = 0; i < 3; i++) res[i] = c0[i] / sn; }
  else { float sn = sqrtf(n1); for (int i = 0; i < 3; i++) res[i] = c1[i] / sn; }
}
void orc_eigen3_v33(const float C[9], float evals[3], float evecs[9]) {
  const float eps = FLT_EPSILON;
  /* shift to the mean eigenvalue, scale the (lower-triangle view of the) matrix into [-1, 1] */
  float shift = ((M3(C, 0, 0) + M3(C, 1, 1)) + M3(C, 2, 2)) / 3.0f;
  float m[9];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) M3(m, r, c) = r >= c ? M3(C, r, c) : M3(C, c, r);
  m[0] -= shift; m[4] -= shift; m[8] -= shift;
  float scale = 0.0f;
  for (int i = 0; i < 9; i++) { float a = fabsf(m[i]); if (a > scale) scale = a; }
  if (scale > 0.0f)
    for (int i = 0; i < 9; i++) m[i] = m[i] / scale;
  /* computeRoots (3.3): roots sorted by construction */
  const float s_inv3 = 1.0f / 3.0f;
  const float s_sqrt3 = sqrtf(3.0f);
  float m00 = M3(m, 0, 0), m11 = M3(m, 1, 1), m22 = M3(m, 2, 2);
  float m10 = M3(m, 1, 0), m20 = M3(m, 2, 0), m21 = M3(m, 2, 1);
  float c0 = m00 * m11 * m22 + 2.0f * m10 * m20 * m21 - m00 * m21 * m21 - m11 * m20 * m20 - m22 * m10 * m10;
  float c1 = m00 * m11 - m10 * m10 + m00 * m22 - m20 * m20 + m11 * m22 - m21 * m21;
  float c2 = m00 + m11 + m22;
  float c2_over_3 = c2 * s_inv3;
  float a_over_3 = (c2 * c2_over_3 - c1) * s_inv3;
  if (a_over_3 < 0.0f) a_over_3 = 0.0f;
  float half_b = 0.5f * (c0 + c2_over_3 * (2.0f * c2_over_3 * c2_over_3 - c1));
  float q = a_over_3 * a_over_3 * a_over_3 - half_b * half_b;
  if (q < 0.0f) q = 0.0f;
  float rho = sqrtf(a_over_3);
  float theta = atan2f(sqrtf(q), half_b) * s_inv3;
  float cos_theta = cosf(theta);
  float sin_theta = sinf(theta);
  float ev[3];
  ev[0] = c2_over_3 - rho * (cos_theta + s_sqrt3 * sin_theta);
  ev[1] = c2_over_3 - rho * (cos_theta - s_sqrt3 * sin_theta);
  ev[2] = c2_over_3 + 2.0f * rho * cos_theta;
  if ((ev[2] - ev[0]) <= eps) {
    memset(evecs, 0, 9 * sizeof(float));
    evecs[0] = evecs[4] = evecs[8] = 1.0f;
  } else {
    float d0 = ev[2] - ev[1];
    float d1 = ev[1] - ev[0];
    int k = 0, l = 2;
    if (d0 > d1) { k = 2; l = 0; d0 = d1; }
    float tmp[9], vk[3], vl[3], dummy[3];
    memcpy(tmp, m, sizeof tmp);
    tmp[0] -= ev[k]; tmp[4] -= ev[k]; tmp[8] -= ev[k];
    extract_kernel33(tmp, vk, vl);
    if (d0 <= 2.0f * eps * d1) {
      /* the other two eigenvalues are numerically the same: ortho-normalise the representative saved above */
      float dot = (vk[0] * vl[0] + vk[1] * vl[1]) + vk[2] * vl[2];
      for (int i = 0; i < 3; i++) vl[i] = vl[i] - dot * vl[i];
      float sn = sqrtf(sqnorm3(vl));
      for (int i = 0; i < 3; i++) vl[i] = vl[i] / sn;
    } else {
      memcpy(tmp, m, sizeof tmp);
      tmp[0] -= ev[l]; tmp[4] -= ev[l]; tmp[8] -= ev[l];
      extract_kernel33(tmp, vl, dummy);
    }
    for (int i = 0; i < 3; i++) { M3(evecs, i, k) = vk[i]; M3(evecs, i, l) = vl[i]; }
    /* col(1) = col(2).cross(col(0)).normalized() */
    float a2[3] = {M3(evecs, 0, 2), M3(evecs, 1, 2), M3(evecs, 2, 2)}, a0[3] = {M3(evecs, 0, 0), M3(evecs, 1, 0), M3(evecs, 2, 0)}, t[3];
    cross3(a2, a0, t);
    float sn = sqrtf(sqnorm3(t));
    for (int i = 0; i < 3; i++) M3(evecs, i, 1) = t[i] / sn;
  }
  for (int i = 0; i < 3; i++) evals[i] = ev[i] * scale + shift;
}
/* 0: Eigen 3.2.x with libm (the reference build; the variant the CUDA path follows), 1: Eigen >= 3.3, 2: Eigen 3.2.x with
 * the CUDA path's float64 trig (test yardstick: every other operation of the CUDA path is meant to match it bit for bit) */
static int g_eigen_variant = 0;
void orc_set_eigen_variant(int v) { g_eigen_variant = v; }
static void eigen3_dispatch(const float C[9], float evals[3], float evecs[9]) {
  if (g_eigen_variant == 1) orc_eigen3_v33(C, evals, evecs);
  else eigen3_32(C, evals, evecs, g_eigen_variant == 2);
}

/* ------------------------------------------------------------------------------------------
 * StatsCalculatorIntegralImage::compute, statscalculatorintegralimage.cpp:14-82.
 * statsM: 16 floats/point (the Stats 4x4: eigenvectors in the 3x3 block, mean in column 3),
 * defaults Stats() = identity, eigenvalues 0, n 0 (stats.h:21-27); curvature as
 * Stats::curvature() returns it (stats.h:98-103): (float)(e0 / (double)(e0+e1+e2) + 1e-9)).
 * ---------------------------------------------------------------------------------------- */
static inline float stats_curvature(const float *e) {
  return (float)((double)e[0] / ((double)((e[0] + e[1]) + e[2]) + 1e-9));
}
void orc_stats(const float *I, const int *index, const int *interval, const float *points,
               int rows, int cols, int n, const orc_stats_params *p,
               float *normals, float *statsM, float *eigvals, int *statsN, float *curvature) {
  for (int i = 0; i < n; i++) {
    memset(normals + 4 * i, 0, 4 * sizeof(float));
    mat4_identity(statsM + 16 * i);
    eigvals[3 * i] = eigvals[3 * i + 1] = eigvals[3 * i + 2] = 0.0f;
    statsN[i] = 0;
    curvature[i] = stats_curvature(eigvals + 3 * i); /* = 0 */
  }
#pragma omp parallel for
  for (int r = 0; r < rows; r++)
    for (int c = 0; c < cols; c++) {
      int idx = index[r * cols + c], k = interval[r * cols + c];
      if (idx < 0 || k < 0) continue;
      if (k < p->minImageRadius) k = p->minImageRadius;
      if (k > p->maxImageRadius) k = p->maxImageRadius;
      float acc[10];
      get_region(I, rows, cols, c - k, c + k, r - k, r + k, acc);
      if ((int)acc[0] < p->minPoints) continue;
      /* PointAccumulator::mean / covariance, pointaccumulator.h:65-86 */
      float d = 1.0f / acc[0];
      float mu[3] = {acc[1] * d, acc[2] * d, acc[3] * d};
      float C[9];
      M3(C, 0, 0) = acc[4] * d - mu[0] * mu[0];
      M3(C, 1, 0) = M3(C, 0, 1) = acc[5] * d - mu[0] * mu[1];
      M3(C, 2, 0) = M3(C, 0, 2) = acc[6] * d - mu[0] * mu[2];
      M3(C, 1, 1) = acc[7] * d - mu[1] * mu[1];
      M3(C, 2, 1) = M3(C, 1, 2) = acc[8] * d - mu[1] * mu[2];
      M3(C, 2, 2) = acc[9] * d - mu[2] * mu[2];
      float ev[3], U[9];
      eigen3_dispatch(C, ev, U);
      if (ev[0] < 0.0f) ev[0] = 0.0f;
      float *S = statsM + 16 * idx;
      memset(S, 0, 16 * sizeof(float));
      for (int rr = 0; rr < 3; rr++)
        for (int cc = 0; cc < 3; cc++) M4(S, rr, cc) = M3(U, rr, cc);
      M4(S, 0, 3) = mu[0]; M4(S, 1, 3) = mu[1]; M4(S, 2, 3) = mu[2]; M4(S, 3, 3) = 1.0f;
      eigvals[3 * idx] = ev[0]; eigvals[3 * idx + 1] = ev[1]; eigvals[3 * idx + 2] = ev[2];
      statsN[idx] = (int)acc[0];
      float curv = stats_curvature(ev);
      curvature[idx] = curv;
      float *nrm = normals + 4 * idx;
      const float *pt = points + 4 * idx;
      nrm[0] = M3(U, 0, 0); nrm[1] = M3(U, 1, 0); nrm[2] = M3(U, 2, 0); nrm[3] = 0.0f;
      if (curv < p->curvatureThreshold) {
        /* normal.dot(point): 4 lanes, w lane contributes 0*1 */
        if (dot4(nrm[0], nrm[1], nrm[2], nrm[3], pt[0], pt[1], pt[2], pt[3]) > 0) {
          nrm[0] = -nrm[0]; nrm[1] = -nrm[1]; nrm[2] = -nrm[2];
        }
      } else {
        nrm[0] = nrm[1] = nrm[2] = 0.0f;
      }
    }
}

/* Point/NormalInformationMatrixCalculator::compute, informationmatrixcalculator.cpp:9-58.
 * omegaP/omegaN: full 4x4 column-major per point (last row/col zero). */
void orc_information(const float *normals, const float *statsM, const float *eigvals, const float *curvature,
                     int n, const orc_stats_params *p, float *omegaP, float *omegaN) {
#pragma omp parallel for
  for (int i = 0; i < n; i++) {
    float *OP = omegaP + 16 * i, *ON = omegaN + 16 * i;
    memset(OP, 0, 16 * sizeof(float));
    memset(ON, 0, 16 * sizeof(float));
    const float *nr = normals + 4 * i;
    float sq = ((nr[0] * nr[0] + nr[1] * nr[1]) + nr[2] * nr[2]) + nr[3] * nr[3];
    if (!(sq > 0)) continue;
    const float *S = statsM + 16 * i;
    float dg[3];
    int flat = curvature[i] < p->omegaCurvatureThreshold;
    if (flat) {
      dg[0] = p->flatOmegaP[0]; dg[1] = p->flatOmegaP[1]; dg[2] = p->flatOmegaP[2];
    } else {
      dg[0] = 1.0f / eigvals[3 * i]; dg[1] = 1.0f / eigvals[3 * i + 1]; dg[2] = 1.0f / eigvals[3 * i + 2];
    }
    /* (U * D) * U^T */
    float UD[9];
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) M3(UD, r, c) = M4(S, r, c) * dg[c];
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++)
        M4(OP, r, c) = dot3(M3(UD, r, 0), M3(UD, r, 1), M3(UD, r, 2), M4(S, c, 0), M4(S, c, 1), M4(S, c, 2));
    const float *dn = flat ? p->flatOmegaN : p->nonFlatOmegaN;
    M4(ON, 0, 0) = dn[0]; M4(ON, 1, 1) = dn[1]; M4(ON, 2, 2) = dn[2];
  }
}

/* Cloud::transformInPlace, cloud.cpp:173-186 (+ TransformableVector, StatsVector,
 * InformationMatrixVector::transformInPlace) */
void orc_cloud_transform(const float T[16], int n, float *points, float *normals, float *statsM,
                         float *omegaP, float *omegaN) {
  float m[16];
  memcpy(m, T, sizeof m);
  fix_last_row(m);
  int ident = 1;
  for (int r = 0; r < 4; r++)
    for (int c = 0; c < 4; c++)
      if (M4(m, r, c) != (r == c ? 1.0f : 0.0f)) ident = 0;
  if (ident) return;
  float R[16];
  memcpy(R, m, sizeof R);
  for (int i = 0; i < 4; i++) { M4(R, 3, i) = 0.0f; M4(R, i, 3) = 0.0f; }
  float Rt[16];
  for (int r = 0; r < 4; r++)
    for (int c = 0; c < 4; c++) M4(Rt, r, c) = M4(R, c, r);
  for (int i = 0; i < n; i++) {
    float o[3];
    float *p = points + 4 * i;
    xform3(m, p[0], p[1], p[2], p[3], o);
    p[0] = o[0]; p[1] = o[1]; p[2] = o[2]; p[3] = 1.0f;
    float *q = normals + 4 * i;
    xform3(m, q[0], q[1], q[2], q[3], o);
    q[0] = o[0]; q[1] = o[1]; q[2] = o[2]; q[3] = 0.0f;
    if (statsM) mat4_mul(m, statsM + 16 * i, statsM + 16 * i);
    if (omegaP) {
      float t[16];
      mat4_mul(R, omegaP + 16 * i, t);
      mat4_mul(t, Rt, omegaP + 16 * i);
      mat4_mul(R, omegaN + 16 * i, t);
      mat4_mul(t, Rt, omegaN + 16 * i);
    }
  }
}

/* DepthImageConverterIntegralImage::compute, depthimageconverterintegralimage.cpp:15-55 */
int orc_depth_to_cloud(const float *depth, int rows, int cols, const float K[9], float minD, float maxD,
                       const orc_stats_params *p, const float sensorOffset[16],
                       float *points, float *normals, float *statsM, float *eigvals, int *statsN,
                       float *curvature, float *omegaP, float *omegaN, int *index, int *interval,
                       float *integral) {
  float I4[16], KRt[16], iKRt[16];
  mat4_identity(I4);
  orc_update_matrices(K, I4, KRt, iKRt);
  int n = orc_unproject(depth, rows, cols, iKRt, minD, maxD, points, index);
  orc_project_intervals(depth, rows, cols, K, minD, maxD, p->worldRadius, interval);
  orc_integral_image(index, points, rows, cols, integral);
  orc_stats(integral, index, interval, points, rows, cols, n, p, normals, statsM, eigvals, statsN, curvature);
  orc_information(normals, statsM, eigvals, curvature, n, p, omegaP, omegaN);
  orc_cloud_transform(sensorOffset, n, points, normals, statsM, omegaP, omegaN);
  return n;
}

/* ------------------------------------------------------------------------------------------
 * MultiPointProjector (see pwn_oracle.h for the layout that is restated)
 * ---------------------------------------------------------------------------------------- */
void orc_multi_image_size(const orc_multi *m, int *rows, int *cols) { /* computeImageSize, multipointprojector.cpp:7-18 */
  int r = 0, c = 0;
  for (int i = 0; i < m->n; i++) {
    if (m->width[i] > r) r = m->width[i];
    c += m->height[i];
  }
  *rows = r;
  *cols = c;
}
/* child projector matrices for a rig pose T: setTransform(T * sensorOffset_i), multipointprojector.cpp:207-215 */
static void multi_child_matrices(const orc_multi *m, const float T[16], int i, float KRt[16], float iKRt[16]) {
  float Tc[16];
  orc_iso_mul(T, m->offset[i], Tc);
  /* PointProjector::setTransform rewrites the last row (pointprojector.h:17-20) */
  fix_last_row(Tc);
  orc_update_matrices(m->K[i], Tc, KRt, iKRt);
}
int orc_multi_unproject(const orc_multi *m, const float T[16], const float *depth, int rows, int cols,
                        float *points, int *index) {
  int count = 0, colOff = 0;
  for (int i = 0; i < rows * cols; i++) index[i] = -1;
  for (int i = 0; i < m->n; i++) {
    float KRt[16], iKRt[16];
    multi_child_matrices(m, T, i, KRt, iKRt);
    for (int r = 0; r < rows && r < m->width[i]; r++)
      for (int v = 0; v < m->height[i] && colOff + v < cols; v++) {
        float d = depth[r * cols + colOff + v];
        if (d < m->minD[i] || d > m->maxD[i]) continue;
        float *p = points + 4 * count;
        xform3(iKRt, r * d, v * d, d, 1.0f, p); /* _unProject(p, x = u = row, y = v) */
        p[3] = 1.0f;
        index[r * cols + colOff + v] = count++;
      }
    colOff += m->height[i];
  }
  return count;
}
void orc_multi_intervals(const orc_multi *m, const float *depth, int rows, int cols, float worldRadius, int *interval) {
  int colOff = 0;
  for (int i = 0; i < rows * cols; i++) interval[i] = -1;
  for (int i = 0; i < m->n; i++) {
    const float *K = m->K[i];
    float p0 = dot3(M3(K, 0, 0), M3(K, 0, 1), M3(K, 0, 2), worldRadius, worldRadius, 0.0f);
    float p1 = dot3(M3(K, 1, 0), M3(K, 1, 1), M3(K, 1, 2), worldRadius, worldRadius, 0.0f);
    for (int r = 0; r < rows && r < m->width[i]; r++)
      for (int v = 0; v < m->height[i] && colOff + v < cols; v++) {
        float d = depth[r * cols + colOff + v];
        if (d < m->minD[i] || d > m->maxD[i]) continue;
        float s = 1.0f / d;
        float a = p0 * s, b = p1 * s;
        interval[r * cols + colOff + v] = (a > b) ? (int)a : (int)b;
      }
    colOff += m->height[i];
  }
}
void orc_multi_project(const orc_multi *m, const float T[16], const float *points, int n, int rows, int cols,
                       int *index, float *depth) {
  float KRt[ORC_MAX_CAMERAS][16], iKRt[16];
  for (int i = 0; i < m->n; i++) multi_child_matrices(m, T, i, KRt[i], iKRt);
  for (int i = 0; i < rows * cols; i++) { depth[i] = 0.0f; index[i] = -1; }
  for (int pi = 0; pi < n; pi++) {
    const float *p = points + 4 * pi;
    int X = -1, Y = -1, colOff = 0;
    float F = 0.0f;
    for (int i = 0; i < m->n; i++) {
      float ip[3];
      xform3(KRt[i], p[0], p[1], p[2], p[3], ip);
      float d = ip[2];
      if (!(d < m->minD[i] || d > m->maxD[i])) {
        float s = 1.0f / d;
        float fx = roundf(ip[0] * s), fy = roundf(ip[1] * s);
        if (!(d < 0.0f) && fx >= 0.0f && fx < (float)m->width[i] && fy >= 0.0f && fy < (float)m->height[i]) {
          X = (int)fx;
          Y = (int)fy + colOff;
          F = d;
          break;
        }
      }
      colOff += m->height[i];
    }
    if (X < 0 || X >= rows || Y < 0 || Y >= cols) continue;
    float *od = &depth[X * cols + Y];
    if (!*od || *od > F) { *od = F; index[X * cols + Y] = pi; }
  }
}
int orc_multi_depth_to_cloud(const orc_multi *m, const float *depth, int rows, int cols, const orc_stats_params *p,
                             const float sensorOffset[16], float *points, float *normals, float *statsM, float *eigvals,
                             int *statsN, float *curvature, float *omegaP, float *omegaN, int *index, int *interval,
                             float *integral) {
  float I4[16];
  mat4_identity(I4);
  int n = orc_multi_unproject(m, I4, depth, rows, cols, points, index);
  orc_multi_intervals(m, depth, rows, cols, p->worldRadius, interval);
  orc_integral_image(index, points, rows, cols, integral);
  orc_stats(integral, index, interval, points, rows, cols, n, p, normals, statsM, eigvals, statsN, curvature);
  orc_information(normals, statsM, eigvals, curvature, n, p, omegaP, omegaN);
  orc_cloud_transform(sensorOffset, n, points, normals, statsM, omegaP, omegaN);
  return n;
}

/* ------------------------------------------------------------------------------------------
 * CorrespondenceFinder::compute, correspondencefinder.cpp:20-118
 * ---------------------------------------------------------------------------------------- */
int orc_correspond(const int *refIndex, const int *curIndex, int rows, int cols,
                   const float *refPoints, const float *refNormals, const float *refCurv,
                   const float *curPoints, const float *curNormals, const float *curCurv,
                   const float Tin[16], const orc_corr_params *p, int numThreads,
                   int *corr, int *corrImage) {
  float T[16];
  memcpy(T, Tin, sizeof T);
  fix_last_row(T);
  if (numThreads < 1) numThreads = 1;
  float squaredThreshold = p->inlierDistanceThreshold * p->inlierDistanceThreshold;
  float minCurvatureRatio = 1.0f / p->inlierCurvatureRatioThreshold;
  float maxCurvatureRatio = p->inlierCurvatureRatioThreshold;
  int *localIndex = (int *)malloc(sizeof(int) * numThreads);
  int *localOffset = (int *)malloc(sizeof(int) * numThreads);
  int rowsPerThread = rows / numThreads;
  int iterationsPerThread = (rows * cols) / numThreads;
  for (int i = 0; i < numThreads; i++) localIndex[i] = localOffset[i] = i * iterationsPerThread;
  if (corrImage)
    for (int i = 0; i < rows * cols; i++) corrImage[i] = -1;
#pragma omp parallel for schedule(static, 1)
  for (int t = 0; t < numThreads; t++) {
    int rMin = t * rowsPerThread, rMax = rMin + rowsPerThread;
    if (rMax > rows) rMax = rows;
    int ci = localIndex[t];
    for (int r = rMin; r < rMax; r++)
      for (int c = 0; c < cols; c++) {
        int ri = refIndex[r * cols + c], cidx = curIndex[r * cols + c];
        if (ri < 0 || cidx < 0) continue;
        const float *cn = curNormals + 4 * cidx, *rn0 = refNormals + 4 * ri;
        const float *cp = curPoints + 4 * cidx, *rp0 = refPoints + 4 * ri;
        if (dot4(cn[0], cn[1], cn[2], cn[3], cn[0], cn[1], cn[2], cn[3]) == 0.0f ||
            dot4(rn0[0], rn0[1], rn0[2], rn0[3], rn0[0], rn0[1], rn0[2], rn0[3]) == 0.0f)
          continue;
        float rp[3], rn[3];
        xform3(T, rp0[0], rp0[1], rp0[2], 1.0f, rp);
        xform3(T, rn0[0], rn0[1], rn0[2], 0.0f, rn);
        if (dot4(cn[0], cn[1], cn[2], 0.0f, rn[0], rn[1], rn[2], 0.0f) < p->inlierNormalAngularThreshold) continue;
        float dx = cp[0] - rp[0], dy = cp[1] - rp[1], dz = cp[2] - rp[2];
        if (dot4(dx, dy, dz, 0.0f, dx, dy, dz, 0.0f) > squaredThreshold) continue;
        float rc = refCurv[ri], cc = curCurv[cidx];
        if (rc < p->flatCurvatureThreshold) rc = p->flatCurvatureThreshold;
        if (cc < p->flatCurvatureThreshold) cc = p->flatCurvatureThreshold;
        float ratio = (float)(((double)rc + 1e-5) / ((double)cc + 1e-5));
        if (ratio < minCurvatureRatio || ratio > maxCurvatureRatio) continue;
        corr[2 * ci] = ri;
        corr[2 * ci + 1] = cidx;
        ci++;
        if (corrImage) corrImage[r * cols + c] = ri;
      }
    localIndex[t] = ci;
  }
  int k = 0;
  for (int t = 0; t < numThreads; t++)
    for (int i = localOffset[t]; i < localIndex[t]; i++) {
      corr[2 * k] = corr[2 * i];
      corr[2 * k + 1] = corr[2 * i + 1];
      k++;
    }
  for (int i = k; i < rows * cols; i++) corr[2 * i] = corr[2 * i + 1] = -1;
  free(localIndex);
  free(localOffset);
  return k;
}

/* ------------------------------------------------------------------------------------------
 * Linearizer::update, linearizer.cpp:17-115.  One correspondence's contribution:
 * Htt(9) Htr(9) Hrr(9) bt(3) br(3), chi2 and kscale.  skew() is bm_se3.h:54-66 (S = -2[v]x).
 * Returns 0 if the correspondence is dropped (non-robust outlier).
 * ---------------------------------------------------------------------------------------- */
typedef struct { float Htt[9], Htr[9], Hrr[9], bt[3], br[3], err; } lin_term;

static void skew3(const float *v, float *S) {
  float tx = 2 * v[0], ty = 2 * v[1], tz = 2 * v[2];
  memset(S, 0, 9 * sizeof(float));
  M3(S, 0, 1) = tz; M3(S, 1, 0) = -tz;
  M3(S, 0, 2) = -ty; M3(S, 2, 0) = ty;
  M3(S, 1, 2) = tx; M3(S, 2, 1) = -tx;
}
static void mat3_mul(const float *A, const float *B, float *C) { /* C = A*B */
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++)
      M3(C, r, c) = dot3(M3(A, r, 0), M3(A, r, 1), M3(A, r, 2), M3(B, 0, c), M3(B, 1, c), M3(B, 2, c));
}
static void mat3_tmul(const float *A, const float *B, float *C) { /* C = A^T*B */
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++)
      M3(C, r, c) = dot3(M3(A, 0, r), M3(A, 1, r), M3(A, 2, r), M3(B, 0, c), M3(B, 1, c), M3(B, 2, c));
}
static int lin_one(const float *T, const float *rp0, const float *rn0, const float *cp, const float *cn,
                   const float *OP4, const float *ON4, float maxChi2, int robust, lin_term *o) {
  float rp[3], rn[3], OP[9], ON[9];
  xform3(T, rp0[0], rp0[1], rp0[2], 1.0f, rp);
  xform3(T, rn0[0], rn0[1], rn0[2], 0.0f, rn);
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) { M3(OP, r, c) = M4(OP4, r, c); M3(ON, r, c) = M4(ON4, r, c); }
  float pe[3] = {rp[0] - cp[0], rp[1] - cp[1], rp[2] - cp[2]};
  float ne[3] = {rn[0] - cn[0], rn[1] - cn[1], rn[2] - cn[2]};
  float ep[3], en[3];
  for (int r = 0; r < 3; r++) {
    ep[r] = dot3(M3(OP, r, 0), M3(OP, r, 1), M3(OP, r, 2), pe[0], pe[1], pe[2]);
    en[r] = dot3(M3(ON, r, 0), M3(ON, r, 1), M3(ON, r, 2), ne[0], ne[1], ne[2]);
  }
  float localError = dot3(pe[0], pe[1], pe[2], ep[0], ep[1], ep[2]) + dot3(ne[0], ne[1], ne[2], en[0], en[1], en[2]);
  float kscale = 1;
  if (localError > maxChi2) {
    if (robust) kscale = sqrtf(maxChi2 / localError);
    else return 0;
  }
  o->err = kscale * localError;
  float Sp[9], Sn[9], A[9], B1[9], B2[9];
  skew3(rp, Sp);
  skew3(rn, Sn);
  memcpy(o->Htt, OP, sizeof OP);
  mat3_mul(OP, Sp, o->Htr);
  mat3_tmul(Sp, OP, A);
  mat3_mul(A, Sp, B1);
  mat3_tmul(Sn, ON, A);
  mat3_mul(A, Sn, B2);
  for (int i = 0; i < 9; i++) o->Hrr[i] = B1[i] + B2[i];
  for (int r = 0; r < 3; r++) {
    o->bt[r] = kscale * ep[r];
    float a = dot3(M3(Sp, 0, r), M3(Sp, 1, r), M3(Sp, 2, r), ep[0], ep[1], ep[2]);
    float b = dot3(M3(Sn, 0, r), M3(Sn, 1, r), M3(Sn, 2, r), en[0], en[1], en[2]);
    o->br[r] = kscale * (a + b);
  }
  return 1;
}
static void assemble_H(const float *Htt, const float *Htr, const float *Hrr, const float *bt, const float *br,
                       float *H, float *b) {
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) {
      M6(H, r, c) = M3(Htt, r, c);
      M6(H, r, c + 3) = M3(Htr, r, c);
      M6(H, r + 3, c + 3) = M3(Hrr, r, c);
      M6(H, c + 3, r) = M3(Htr, r, c);
    }
  for (int r = 0; r < 3; r++) { b[r] = bt[r]; b[r + 3] = br[r]; }
}
void orc_linearize(const int *corr, int numCorr,
                   const float *refPoints, const float *refNormals,
                   const float *curPoints, const float *curNormals,
                   const float *curOmegaP, const float *curOmegaN,
                   const float Tin[16], float inlierMaxChi2, int robustKernel, int numThreads,
                   float H[36], float b[6], float *error, int *inliers) {
  float T[16];
  memcpy(T, Tin, sizeof T);
  fix_last_row(T);
  if (numThreads < 1) numThreads = 1;
  lin_term *part = (lin_term *)calloc(numThreads, sizeof(lin_term));
  int *pin = (int *)calloc(numThreads, sizeof(int));
  int iterationsPerThread = numCorr / numThreads;
#pragma omp parallel for schedule(static, 1)
  for (int t = 0; t < numThreads; t++) {
    int imin = iterationsPerThread * t, imax = imin + iterationsPerThread;
    if (imax > numCorr) imax = numCorr;
    lin_term acc;
    memset(&acc, 0, sizeof acc);
    int inl = 0;
    for (int i = imin; i < imax; i++) {
      int ri = corr[2 * i], ci = corr[2 * i + 1];
      lin_term o;
      if (!lin_one(T, refPoints + 4 * ri, refNormals + 4 * ri, curPoints + 4 * ci, curNormals + 4 * ci,
                   curOmegaP + 16 * ci, curOmegaN + 16 * ci, inlierMaxChi2, robustKernel, &o))
        continue;
      inl++;
      acc.err += o.err;
      for (int k = 0; k < 9; k++) { acc.Htt[k] += o.Htt[k]; acc.Htr[k] += o.Htr[k]; acc.Hrr[k] += o.Hrr[k]; }
      for (int k = 0; k < 3; k++) { acc.bt[k] += o.bt[k]; acc.br[k] += o.br[k]; }
    }
    part[t] = acc;
    pin[t] = inl;
  }
  lin_term s;
  memset(&s, 0, sizeof s);
  int inl = 0;
  for (int t = 0; t < numThreads; t++) {
    for (int k = 0; k < 9; k++) { s.Htt[k] += part[t].Htt[k]; s.Htr[k] += part[t].Htr[k]; s.Hrr[k] += part[t].Hrr[k]; }
    for (int k = 0; k < 3; k++) { s.bt[k] += part[t].bt[k]; s.br[k] += part[t].br[k]; }
    s.err += part[t].err;
    inl += pin[t];
  }
  assemble_H(s.Htt, s.Htr, s.Hrr, s.bt, s.br, H, b);
  *error = s.err;
  *inliers = inl;
  free(part);
  free(pin);
}
void orc_linearize_f64(const int *corr, int numCorr,
                       const float *refPoints, const float *refNormals,
                       const float *curPoints, const float *curNormals,
                       const float *curOmegaP, const float *curOmegaN,
                       const float Tin[16], float inlierMaxChi2, int robustKernel,
                       double H[36], double b[6], double *error, int *inliers) {
  float T[16];
  memcpy(T, Tin, sizeof T);
  fix_last_row(T);
  double Htt[9] = {0}, Htr[9] = {0}, Hrr[9] = {0}, bt[3] = {0}, br[3] = {0}, err = 0;
  int inl = 0;
  for (int i = 0; i < numCorr; i++) {
    int ri = corr[2 * i], ci = corr[2 * i + 1];
    lin_term o;
    if (!lin_one(T, refPoints + 4 * ri, refNormals + 4 * ri, curPoints + 4 * ci, curNormals + 4 * ci,
                 curOmegaP + 16 * ci, curOmegaN + 16 * ci, inlierMaxChi2, robustKernel, &o))
      continue;
    inl++;
    err += o.err;
    for (int k = 0; k < 9; k++) { Htt[k] += o.Htt[k]; Htr[k] += o.Htr[k]; Hrr[k] += o.Hrr[k]; }
    for (int k = 0; k < 3; k++) { bt[k] += o.bt[k]; br[k] += o.br[k]; }
  }
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) {
      M6(H, r, c) = M3(Htt, r, c);
      M6(H, r, c + 3) = M3(Htr, r, c);
      M6(H, r + 3, c + 3) = M3(Hrr, r, c);
      M6(H, c + 3, r) = M3(Htr, r, c);
    }
  for (int r = 0; r < 3; r++) { b[r] = bt[r]; b[r + 3] = br[r]; }
  *error = err;
  *inliers = inl;
}

/* ------------------------------------------------------------------------------------------
 * Eigen::LDLT<Matrix6f>::compute + solve (Eigen 3.2 ldlt_inplace<Lower>::unblocked with
 * diagonal pivoting), used as H.ldlt().solve(-b) at aligner.cpp:110.  x = H^-1 b here.
 * ---------------------------------------------------------------------------------------- */
void orc_ldlt_solve6(const float Hin[36], const float bin[6], float x[6]) {
  const int N = 6;
  float m[36];
  int tr[6];
  memcpy(m, Hin, sizeof m);
  for (int k = 0; k < N; k++) {
    int big = k;
    float bv = fabsf(M6(m, k, k));
    for (int i = k + 1; i < N; i++) {
      float a = fabsf(M6(m, i, i));
      if (a > bv) { bv = a; big = i; }
    }
    tr[k] = big;
    if (big != k) {
      float t;
      for (int j = 0; j < k; j++) { t = M6(m, k, j); M6(m, k, j) = M6(m, big, j); M6(m, big, j) = t; }
      for (int i = big + 1; i < N; i++) { t = M6(m, i, k); M6(m, i, k) = M6(m, i, big); M6(m, i, big) = t; }
      t = M6(m, k, k); M6(m, k, k) = M6(m, big, big); M6(m, big, big) = t;
      for (int i = k + 1; i < big; i++) { t = M6(m, i, k); M6(m, i, k) = M6(m, big, i); M6(m, big, i) = t; }
    }
    if (k > 0) {
      float temp[6];
      for (int j = 0; j < k; j++) temp[j] = M6(m, j, j) * M6(m, k, j);
      float s = 0.0f;
      for (int j = 0; j < k; j++) s += M6(m, k, j) * temp[j];
      M6(m, k, k) -= s;
      for (int i = k + 1; i < N; i++) {
        float s2 = 0.0f;
        for (int j = 0; j < k; j++) s2 += M6(m, i, j) * temp[j];
        M6(m, i, k) -= s2;
      }
    }
    float akk = M6(m, k, k);
    if (fabsf(akk) > 0.0f)
      for (int i = k + 1; i < N; i++) M6(m, i, k) /= akk;
  }
  float y[6];
  memcpy(y, bin, sizeof y);
  for (int k = 0; k < N; k++) { float t = y[k]; y[k] = y[tr[k]]; y[tr[k]] = t; }
  for (int i = 0; i < N; i++) {         /* L y' = y, unit lower */
    float s = y[i];
    for (int j = 0; j < i; j++) s -= M6(m, i, j) * y[j];
    y[i] = s;
  }
  for (int i = 0; i < N; i++) {         /* D */
    float d = M6(m, i, i);
    y[i] = (fabsf(d) > FLT_MIN) ? y[i] / d : 0.0f;
  }
  for (int i = N - 1; i >= 0; i--) {    /* L^T */
    float s = y[i];
    for (int j = i + 1; j < N; j++) s -= M6(m, j, i) * y[j];
    y[i] = s;
  }
  for (int k = N - 1; k >= 0; k--) { float t = y[k]; y[k] = y[tr[k]]; y[tr[k]] = t; }
  memcpy(x, y, sizeof y);
}

/* ------------------------------------------------------------------------------------------
 * small dense helpers for priors and statistics (host-side, tiny)
 * ---------------------------------------------------------------------------------------- */
static void mat6_mul(const float *A, const float *B, float *C) {
  float t[36];
  for (int c = 0; c < 6; c++)
    for (int r = 0; r < 6; r++) {
      float s = 0.0f;
      for (int k = 0; k < 6; k++) s += M6(A, r, k) * M6(B, k, c);
      M6(t, r, c) = s;
    }
  memcpy(C, t, sizeof t);
}
static void mat6_transpose(const float *A, float *At) {
  float t[36];
  for (int r = 0; r < 6; r++)
    for (int c = 0; c < 6; c++) M6(t, r, c) = M6(A, c, r);
  memcpy(At, t, sizeof t);
}
/* general 6x6 inverse: Gauss-Jordan with partial pivoting in float64 (Eigen uses PartialPivLU
   in float32 for sizes > 4; tolerance-level parity only) */
static void mat6_inverse(const float *A, float *Ai) {
  double a[6][12];
  for (int r = 0; r < 6; r++)
    for (int c = 0; c < 6; c++) { a[r][c] = M6(A, r, c); a[r][c + 6] = (r == c); }
  for (int k = 0; k < 6; k++) {
    int piv = k;
    for (int r = k + 1; r < 6; r++)
      if (fabs(a[r][k]) > fabs(a[piv][k])) piv = r;
    if (piv != k)
      for (int c = 0; c < 12; c++) { double t = a[k][c]; a[k][c] = a[piv][c]; a[piv][c] = t; }
    double d = a[k][k];
    for (int c = 0; c < 12; c++) a[k][c] /= d;
    for (int r = 0; r < 6; r++)
      if (r != k) {
        double f = a[r][k];
        if (f != 0.0)
          for (int c = 0; c < 12; c++) a[r][c] -= f * a[k][c];
      }
  }
  for (int r = 0; r < 6; r++)
    for (int c = 0; c < 6; c++) M6(Ai, r, c) = (float)a[r][c + 6];
}

/* SE3Prior, se3_prior.cpp:8-71 */
static void prior_error(const orc_prior *pr, const float *mean, const float *invT, float e[6]) {
  float t[16];
  if (pr->kind == 0) {
    orc_iso_mul(invT, mean, t);
  } else {
    float u[16];
    orc_iso_mul(invT, pr->refInv, u);
    orc_iso_mul(u, mean, t);
  }
  orc_t2v(t, e);
}
static void prior_jacobian(const orc_prior *pr, const float *invT, float J[36]) {
  float epsilon = 1e-3f, iEps = 0.5f / epsilon;
  for (int i = 0; i < 6; i++) {
    float up[6] = {0}, dn[6] = {0}, Tu[16], Td[16], A[16], eu[6], ed[6];
    up[i] = epsilon;
    dn[i] = -epsilon;
    orc_v2t(up, Tu);
    orc_v2t(dn, Td);
    orc_iso_mul(Tu, invT, A);
    prior_error(pr, pr->mean, A, eu);
    orc_iso_mul(Td, invT, A);
    prior_error(pr, pr->mean, A, ed);
    for (int r = 0; r < 6; r++) M6(J, r, i) = iEps * (eu[r] - ed[r]);
  }
}
static void prior_jacobianZ(const orc_prior *pr, const float *invT, float J[36]) {
  float epsilon = 1e-3f, iEps = 0.5f / epsilon;
  for (int i = 0; i < 6; i++) {
    float up[6] = {0}, dn[6] = {0}, Tu[16], Td[16], mu[16], md[16], eu[6], ed[6];
    up[i] = epsilon;
    dn[i] = -epsilon;
    orc_v2t(up, Tu);
    orc_v2t(dn, Td);
    orc_iso_mul(pr->mean, Tu, mu);
    orc_iso_mul(pr->mean, Td, md);
    prior_error(pr, mu, invT, eu);
    prior_error(pr, md, invT, ed);
    for (int r = 0; r < 6; r++) M6(J, r, i) = iEps * (eu[r] - ed[r]);
  }
}
/* aligner.cpp:97-108 */
static void add_priors(const orc_align_params *p, const float *invT, float *H, float *b) {
  for (int j = 0; j < p->numPriors; j++) {
    const orc_prior *pr = &p->priors[j];
    float e[6], J[36], Jz[36], iJz[36], iJzT[36], info[36], Jt[36], A[36], Hp[36];
    prior_error(pr, pr->mean, invT, e);
    prior_jacobian(pr, invT, J);
    prior_jacobianZ(pr, invT, Jz);
    mat6_inverse(Jz, iJz);
    mat6_transpose(iJz, iJzT);
    mat6_mul(iJzT, pr->info, A);
    mat6_mul(A, iJz, info);
    mat6_transpose(J, Jt);
    mat6_mul(Jt, info, A);
    mat6_mul(A, J, Hp);
    for (int i = 0; i < 36; i++) H[i] += Hp[i];
    for (int r = 0; r < 6; r++) {
      float s = 0.0f;
      for (int k = 0; k < 6; k++) s += M6(A, r, k) * e[k];
      b[r] += s;
    }
  }
}

/* cyclic Jacobi eigen-decomposition of a symmetric n x n matrix in float64 (n <= 6);
   stands in for Eigen::JacobiSVD at aligner.cpp:172-173,190-198 (tolerance-level parity) */
static void jacobi_sym(int n, double *A /* n*n col-major, destroyed */, double *V, double *w) {
  for (int i = 0; i < n * n; i++) V[i] = 0;
  for (int i = 0; i < n; i++) V[i * n + i] = 1;
  for (int sweep = 0; sweep < 60; sweep++) {
    double off = 0, diag = 0;
    for (int p = 0; p < n; p++) {
      diag += A[p * n + p] * A[p * n + p];
      for (int q = p + 1; q < n; q++) off += A[q * n + p] * A[q * n + p];
    }
    /* converged to double precision (the old absolute 1e-300 test never fired and all 60 sweeps ran) */
    if (off <= 1e-32 * (diag + off)) break;
    for (int p = 0; p < n; p++)
      for (int q = p + 1; q < n; q++) {
        double apq = A[q * n + p];
        if (fabs(apq) < 1e-300) continue;
        double app = A[p * n + p], aqq = A[q * n + q];
        double tau = (aqq - app) / (2 * apq);
        double t = (tau >= 0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1 + tau * tau));
        double c = 1 / sqrt(1 + t * t), s = t * c;
        for (int k = 0; k < n; k++) {
          double akp = A[p * n + k], akq = A[q * n + k];
          A[p * n + k] = c * akp - s * akq;
          A[q * n + k] = s * akp + c * akq;
        }
        for (int k = 0; k < n; k++) {
          double apk = A[k * n + p], aqk = A[k * n + q];
          A[k * n + p] = c * apk - s * aqk;
          A[k * n + q] = s * apk + c * aqk;
        }
        for (int k = 0; k < n; k++) {
          double vkp = V[p * n + k], vkq = V[q * n + k];
          V[p * n + k] = c * vkp - s * vkq;
          V[q * n + k] = s * vkp + c * vkq;
        }
      }
  }
  for (int i = 0; i < n; i++) w[i] = A[i * n + i];
}
static void sym_pinv6(const float *H, float *Hi) {
  double A[36], V[36], w[6];
  for (int r = 0; r < 6; r++)
    for (int c = 0; c < 6; c++) A[c * 6 + r] = 0.5 * ((double)M6(H, r, c) + (double)M6(H, c, r));
  jacobi_sym(6, A, V, w);
  double wmax = 0;
  for (int i = 0; i < 6; i++) if (fabs(w[i]) > wmax) wmax = fabs(w[i]);
  for (int r = 0; r < 6; r++)
    for (int c = 0; c < 6; c++) {
      double s = 0;
      for (int k = 0; k < 6; k++)
        if (fabs(w[k]) > wmax * 6 * (double)FLT_EPSILON) s += V[k * 6 + r] * V[k * 6 + c] / w[k];
      M6(Hi, r, c) = (float)s;
    }
}
static float sym_eig_ratio3(const float *O, int off) {
  double A[9], V[9], w[3];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) A[c * 3 + r] = 0.5 * ((double)M6(O, off + r, off + c) + (double)M6(O, off + c, off + r));
  jacobi_sym(3, A, V, w);
  double mx = 0, mn = 1e300;
  for (int i = 0; i < 3; i++) { double a = fabs(w[i]); if (a > mx) mx = a; if (a < mn) mn = a; }
  return (float)(mx / mn);
}

/* Aligner::_computeStatistics tail, aligner.cpp:172-198; unscented.h:23-65 */
static void compute_statistics(const float *H_lin, const float *T, float *mean, float *Omega, float *tr, float *rr) {
  float H[36], Sigma[36];
  memcpy(H, H_lin, sizeof H);
  for (int i = 0; i < 6; i++) M6(H, i, i) += 1.0f;
  sym_pinv6(H, Sigma);
  const int dim = 6;
  const double alpha = 1e-3, beta = 2.;
  const double lambda = alpha * alpha * dim;
  const double wi = 1. / (2. * (dim + lambda));
  double wm[13], wc[13];
  float samples[13][6];
  memset(samples, 0, sizeof samples);
  wm[0] = lambda / (dim + lambda);
  wc[0] = lambda / (dim + lambda) + (1. - alpha * alpha + beta);
  /* LLT of Sigma * (dim + lambda), float32 */
  float A[36], L[36];
  memset(L, 0, sizeof L);
  float sc = (float)(dim + lambda);
  for (int i = 0; i < 36; i++) A[i] = Sigma[i] * sc;
  for (int j = 0; j < 6; j++) {
    float s = M6(A, j, j);
    for (int k = 0; k < j; k++) s -= M6(L, j, k) * M6(L, j, k);
    float d = sqrtf(s);
    M6(L, j, j) = d;
    for (int i = j + 1; i < 6; i++) {
      float t = M6(A, i, j);
      for (int k = 0; k < j; k++) t -= M6(L, i, k) * M6(L, j, k);
      M6(L, i, j) = t / d;
    }
  }
  int k = 1;
  for (int i = 0; i < dim; i++) {
    for (int r = 0; r < 6; r++) { samples[k][r] = M6(L, r, i); samples[k + 1][r] = -M6(L, r, i); }
    wm[k] = wc[k] = wi;
    wm[k + 1] = wc[k + 1] = wi;
    k += 2;
  }
  for (int i = 0; i < 13; i++) {
    float X[16], Xi[16], Y[16];
    orc_v2t(samples[i], X);
    orc_iso_inverse(X, Xi);
    orc_iso_mul(T, Xi, Y);
    orc_t2v(Y, samples[i]);
  }
  for (int r = 0; r < 6; r++) mean[r] = 0;
  for (int i = 0; i < 13; i++)
    for (int r = 0; r < 6; r++) mean[r] += (float)(wm[i] * (double)samples[i][r]);
  float cov[36];
  memset(cov, 0, sizeof cov);
  for (int i = 0; i < 13; i++) {
    float dl[6];
    for (int r = 0; r < 6; r++) dl[r] = samples[i][r] - mean[r];
    for (int r = 0; r < 6; r++)
      for (int c = 0; c < 6; c++) M6(cov, r, c) += (float)(wc[i] * (double)(dl[r] * dl[c]));
  }
  mat6_inverse(cov, Omega);
  *tr = sym_eig_ratio3(Omega, 0);
  *rr = sym_eig_ratio3(Omega, 3);
}

/* ------------------------------------------------------------------------------------------
 * Aligner::align, aligner.cpp:49-150
 * ---------------------------------------------------------------------------------------- */
/* test knob: accumulate the Linearizer sums of orc_align in float64 (same float32 terms, exact
   summation) -- the yardstick that separates the GPU's error from the reference's own float32
   summation noise.  0 = reference behaviour. */
static int g_accumulate_f64 = 0;
void orc_set_accumulate_f64(int on) { g_accumulate_f64 = on; }
/* OpenMP team size of every parallel region of this library (the reference runs its `#pragma omp parallel for` loops with
 * the runtime's default team; OMP_NUM_THREADS is only read when libgomp initialises, so callers that choose the thread
 * count later -- bench.py under torch.distributed.run, which exports OMP_NUM_THREADS=1 -- must call this).  Returns the
 * team size now in force (omp_get_max_threads). */
int orc_set_threads(int n) {
  if (n > 0) omp_set_num_threads(n);
  return omp_get_max_threads();
}
static void align_linearize(const int *corr, int numCorr, const float *refPoints, const float *refNormals,
                            const float *curPoints, const float *curNormals, const float *curOmegaP,
                            const float *curOmegaN, const float *invT, const orc_align_params *p, float *H, float *b,
                            float *err, int *inl) {
  if (!g_accumulate_f64) {
    orc_linearize(corr, numCorr, refPoints, refNormals, curPoints, curNormals, curOmegaP, curOmegaN, invT,
                  p->inlierMaxChi2, p->robustKernel, p->numThreads, H, b, err, inl);
    return;
  }
  double Hd[36], bd[6], ed;
  orc_linearize_f64(corr, numCorr, refPoints, refNormals, curPoints, curNormals, curOmegaP, curOmegaN, invT,
                    p->inlierMaxChi2, p->robustKernel, Hd, bd, &ed, inl);
  for (int i = 0; i < 36; i++) H[i] = (float)Hd[i];
  for (int i = 0; i < 6; i++) b[i] = (float)bd[i];
  *err = (float)ed;
}

/* aligner.cpp:92-111: H + I + 1000 I, the priors at invT, dx = LDLT^-1 (-b), invT = v2t(dx) invT */
static void gn_solve(const orc_align_params *p, const float *H, const float *b, float *invT) {
  float Hd[36], nb[6], dx[6], dT[16];
  memcpy(Hd, H, sizeof Hd);
  for (int d = 0; d < 6; d++) M6(Hd, d, d) = M6(Hd, d, d) + 1.0f;
  for (int d = 0; d < 6; d++) M6(Hd, d, d) = M6(Hd, d, d) + 1000.0f;
  memcpy(nb, b, sizeof nb);
  if (p->numPriors) add_priors(p, invT, Hd, nb);
  for (int d = 0; d < 6; d++) nb[d] = -nb[d];
  orc_ldlt_solve6(Hd, nb, dx);
  orc_v2t(dx, dT);
  orc_iso_mul(dT, invT, invT);
}
/* aligner.cpp:115-117: T = invT^-1, T = v2t(t2v(T)), fixLastRow */
static void gn_finish(const float *invT, float *T) {
  orc_iso_inverse(invT, T);
  float v[6];
  orc_t2v(T, v);
  orc_v2t(v, T);
  fix_last_row(T);
}

void orc_align(int nRef, const float *refPoints, const float *refNormals, const float *refCurv,
               int nCur, const float *curPoints, const float *curNormals, const float *curCurv,
               const float *curOmegaP, const float *curOmegaN,
               const orc_align_params *p, orc_align_result *res,
               int *refIndex, float *refDepth, int *curIndex, float *curDepth, int *corr,
               float *trace) {
  float KRt[16], iKRt[16], T[16], invT[16], tmp[16];
  float H[36], b[6], err = 0;
  int inl = 0, numCorr = 0;
  memset(H, 0, sizeof H);
  memset(b, 0, sizeof b);
  if (p->multi) {
    orc_multi_project(p->multi, p->curSensorOffset, curPoints, nCur, p->rows, p->cols, curIndex, curDepth);
  } else {
    orc_update_matrices(p->K, p->curSensorOffset, KRt, iKRt);
    orc_project(curPoints, nCur, p->rows, p->cols, KRt, p->minD, p->maxD, curIndex, curDepth);
  }
  memcpy(T, p->initialGuess, sizeof T);
  for (int i = 0; i < p->outerIterations; i++) {
    fix_last_row(T);
    orc_iso_mul(T, p->refSensorOffset, tmp);
    if (p->multi) {
      fix_last_row(tmp);
      orc_multi_project(p->multi, tmp, refPoints, nRef, p->rows, p->cols, refIndex, refDepth);
    } else {
      orc_update_matrices(p->K, tmp, KRt, iKRt);
      orc_project(refPoints, nRef, p->rows, p->cols, KRt, p->minD, p->maxD, refIndex, refDepth);
    }
    orc_iso_inverse(T, invT);
    numCorr = orc_correspond(refIndex, curIndex, p->rows, p->cols, refPoints, refNormals, refCurv,
                             curPoints, curNormals, curCurv, invT, &p->corr, p->numThreads, corr, NULL);
    if (trace) memcpy(trace + ORC_TRACE_STRIDE * i, T, 16 * sizeof(float));
    for (int k = 0; k < p->innerIterations; k++) {
      fix_last_row(invT);
      align_linearize(corr, numCorr, refPoints, refNormals, curPoints, curNormals, curOmegaP, curOmegaN, invT, p, H, b,
                      &err, &inl);
      if (trace && k == 0) {
        float *tr = trace + ORC_TRACE_STRIDE * i;
        memcpy(tr + 16, H, 36 * sizeof(float));
        memcpy(tr + 52, b, 6 * sizeof(float));
        tr[58] = err; tr[59] = (float)inl; tr[60] = (float)numCorr;
      }
      gn_solve(p, H, b, invT);
    }
    gn_finish(invT, T);
  }
  res->error = err;
  res->inliers = inl;
  res->numCorrespondences = numCorr;
  memcpy(res->T, T, sizeof res->T);
  /* _computeStatistics: one more linearisation at the final T with the last correspondences */
  orc_iso_inverse(T, invT);
  fix_last_row(invT);
  align_linearize(corr, numCorr, refPoints, refNormals, curPoints, curNormals, curOmegaP, curOmegaN, invT, p, H, b,
                  &err, &inl);
  memcpy(res->H, H, sizeof res->H);
  memcpy(res->b, b, sizeof res->b);
  compute_statistics(H, T, res->mean, res->omega, &res->translationalRatio, &res->rotationalRatio);
}

void orc_compute_statistics(const float H[36], const float T[16], float mean[6], float Omega[36], float *tr, float *rr) {
  compute_statistics(H, T, mean, Omega, tr, rr);
}

/* orc_align's outer iteration (inner = 1) from its linearisation on */
void orc_gn_step(const float H[36], const float b[6], const float T[16], const orc_prior *priors, int numPriors,
                 float Tnext[16]) {
  orc_align_params p;
  memset(&p, 0, sizeof p);
  p.numPriors = numPriors;
  p.priors = priors;
  float Tc[16], invT[16];
  memcpy(Tc, T, sizeof Tc);
  fix_last_row(Tc);
  orc_iso_inverse(Tc, invT);
  fix_last_row(invT);
  gn_solve(&p, H, b, invT);
  gn_finish(invT, Tnext);
}

/* PwnMatcherBase::matchClouds, pwn_tracker2/pwn_matcher_base.cpp:167-196.  NB: the reference
 * computes diff = abs(cur-ref) & mask as a BITWISE and of float bit patterns with 255.0f. */
void orc_image_stats(const float *curDepth, const float *refDepth, int n, float inlierDepthThreshold,
                     int *nonZeros, int *inliers, int *outliers, float *reprojectionDistance) {
  int nz = 0, inl = 0;
  float sum = 0;
  union { float f; uint32_t u; } m255, a, o;
  m255.f = 255.0f;
  for (int i = 0; i < n; i++) {
    uint16_t c = (curDepth[i] < FLT_MAX) ? (uint16_t)(1000.0f * curDepth[i]) : 0;
    uint16_t r = (refDepth[i] < FLT_MAX) ? (uint16_t)(1000.0f * refDepth[i]) : 0;
    int mask = (c > 0) && (r > 0);
    a.f = fabsf((float)c - (float)r);
    o.u = mask ? (a.u & m255.u) : 0u;
    float d = o.f;
    if (mask) nz++;
    if (mask && d < inlierDepthThreshold) inl++;
    sum += d;
  }
  *nonZeros = nz;
  *inliers = inl;
  *outliers = nz - inl;
  *reprojectionDistance = sum / nz;
}

/* ------------------------------------------------------------------------------------------
 * Gaussian3f sensor model and Merger (local-map maintenance)
 * ---------------------------------------------------------------------------------------- */
static void mat3_mulf(const float *A, const float *B, float *C) { /* C = A*B, canonical dot order */
  float o[9];
  for (int c = 0; c < 3; c++)
    for (int r = 0; r < 3; r++)
      M3(o, r, c) = dot3(M3(A, r, 0), M3(A, r, 1), M3(A, r, 2), M3(B, 0, c), M3(B, 1, c), M3(B, 2, c));
  memcpy(C, o, sizeof o);
}
static void mat3_mul_bt(const float *A, const float *B, float *C) { /* C = A*B^T */
  float o[9];
  for (int c = 0; c < 3; c++)
    for (int r = 0; r < 3; r++)
      M3(o, r, c) = dot3(M3(A, r, 0), M3(A, r, 1), M3(A, r, 2), M3(B, c, 0), M3(B, c, 1), M3(B, c, 2));
  memcpy(C, o, sizeof o);
}
static void mat3_vec(const float *A, const float *v, float *o) {
  float t[3];
  for (int r = 0; r < 3; r++) t[r] = dot3(M3(A, r, 0), M3(A, r, 1), M3(A, r, 2), v[0], v[1], v[2]);
  o[0] = t[0]; o[1] = t[1]; o[2] = t[2];
}
/* Gaussian::_updateMoments / _updateInfo, basemath/gaussian.h:76-90 */
static void gauss_update_moments(float *g, int *f) {
  if (*f & ORC_GAUSS_MOMENTS) return;
  mat3_inverse(g + 15, g + 3);
  mat3_vec(g + 3, g + 12, g);
  *f |= ORC_GAUSS_MOMENTS;
}
static void gauss_update_info(float *g, int *f) {
  if (*f & ORC_GAUSS_INFO) return;
  mat3_inverse(g + 3, g + 15);
  mat3_vec(g + 15, g, g + 12);
  *f |= ORC_GAUSS_INFO;
}
/* pinholepointprojector.cpp:93-133 */
int orc_unproject_gaussians(const float *depth, int rows, int cols, const float K[9], const float iKRt[16],
                            float minD, float maxD, float baseline, float alpha, float *points, int *index,
                            float *gauss, int *gflags) {
  float iK[9];
  mat3_inverse(K, iK);
  const float fB = baseline * M3(K, 0, 0);
  int count = 0;
  for (int r = 0; r < rows; r++)
    for (int c = 0; c < cols; c++) {
      float z = depth[r * cols + c];
      if (z < minD || z > maxD) { index[r * cols + c] = -1; continue; }
      float *p = points + 4 * count;
      xform3(iKRt, c * z, r * z, z, 1.0f, p);
      p[3] = 1.0f;
      float zVariation = (alpha * z * z) / (fB + z * alpha);
      float J[9] = {z, 0.0f, 0.0f, 0.0f, z, 0.0f, (float)c, (float)r, 1.0f}; /* column-major [z 0 c; 0 z r; 0 0 1] */
      mat3_mulf(iK, J, J);
      float JD[9];
      const float dg[3] = {3.0f, 3.0f, zVariation};
      for (int j = 0; j < 3; j++)
        for (int i = 0; i < 3; i++) M3(JD, i, j) = M3(J, i, j) * dg[j];
      float *g = gauss + (size_t)ORC_GAUSS_FLOATS * count;
      memset(g, 0, sizeof(float) * ORC_GAUSS_FLOATS);
      g[0] = p[0]; g[1] = p[1]; g[2] = p[2];
      mat3_mul_bt(JD, J, g + 3);
      gflags[count] = ORC_GAUSS_MOMENTS;
      index[r * cols + c] = count++;
    }
  return count;
}
/* gaussian3.h:26-36 */
void orc_gaussians_transform(const float T[16], int n, float *gauss, int *gflags) {
  float m[16];
  memcpy(m, T, sizeof m);
  fix_last_row(m);
  int ident = 1;
  for (int r = 0; r < 4; r++)
    for (int c = 0; c < 4; c++)
      if (M4(m, r, c) != (r == c ? 1.0f : 0.0f)) ident = 0;
  if (ident) return;
  float R[9], t[3];
  for (int r = 0; r < 3; r++) {
    for (int c = 0; c < 3; c++) M3(R, r, c) = M4(m, r, c);
    t[r] = M4(m, r, 3);
  }
  for (int i = 0; i < n; i++) {
    float *g = gauss + (size_t)ORC_GAUSS_FLOATS * i;
    gauss_update_moments(g, &gflags[i]);
    float mean[3], RC[9];
    mat3_vec(R, g, mean);
    g[0] = mean[0] + t[0]; g[1] = mean[1] + t[1]; g[2] = mean[2] + t[2];
    mat3_mulf(R, g + 3, RC);
    mat3_mul_bt(RC, R, g + 3);
    gflags[i] = ORC_GAUSS_MOMENTS;
  }
}
/* merger.cpp:15-119 */
int orc_merge(int n, float *points, float *normals, float *statsM, float *omegaP, float *omegaN, float *gauss,
              int *gflags, int rows, int cols, const float K[9], const float T[16], float minD, float maxD,
              float distanceThreshold, float normalThreshold, float maxPointDepth, int *collapsedOut) {
  float KRt[16], iKRt[16];
  orc_update_matrices(K, T, KRt, iKRt);
  int *indexImage = (int *)malloc(sizeof(int) * rows * cols);
  float *depthImage = (float *)malloc(sizeof(float) * rows * cols);
  int *collapsed = (int *)malloc(sizeof(int) * (n > 0 ? n : 1));
  orc_project(points, n, rows, cols, KRt, minD, maxD, indexImage, depthImage);
  for (int i = 0; i < n; i++) collapsed[i] = -1;
  for (int i = 0; i < n; i++) {
    const float *p = points + 4 * i, *cn = normals + 4 * i;
    int r = -1, c = -1;
    float ip[3];
    xform3(KRt, p[0], p[1], p[2], p[3], ip);
    float depth = ip[2];
    if (!(depth < minD || depth > maxD)) { /* _project, pinholepointprojector.h:224-233 */
      float s = 1.0f / depth;
      c = (int)roundf(ip[0] * s);
      r = (int)roundf(ip[1] * s);
    }
    if (depth < 0 || depth > maxPointDepth || r < 0 || r >= rows || c < 0 || c >= cols) continue;
    float targetZ = depthImage[r * cols + c];
    int targetIndex = indexImage[r * cols + c];
    if (targetIndex < 0) continue;
    const float *tn = normals + 4 * targetIndex;
    if (targetIndex == i) {
      collapsed[i] = i;
    } else if (fabsf(depth - targetZ) < distanceThreshold &&
               dot4(cn[0], cn[1], cn[2], cn[3], tn[0], tn[1], tn[2], tn[3]) > normalThreshold) {
      float *tg = gauss + (size_t)ORC_GAUSS_FLOATS * targetIndex, *cg = gauss + (size_t)ORC_GAUSS_FLOATS * i;
      gauss_update_info(tg, &gflags[targetIndex]); /* Gaussian::addInformation, gaussian.h:49-55 */
      gauss_update_info(cg, &gflags[i]);
      for (int k = 0; k < 9; k++) tg[15 + k] += cg[15 + k];
      for (int k = 0; k < 3; k++) tg[12 + k] += cg[12 + k];
      gflags[targetIndex] &= ~ORC_GAUSS_MOMENTS;
      collapsed[i] = targetIndex;
    }
  }
  int k = 0;
  for (int i = 0; i < n; i++) {
    int ci = collapsed[i];
    if (ci == i) {
      float *g = gauss + (size_t)ORC_GAUSS_FLOATS * i;
      gauss_update_moments(g, &gflags[i]);
      points[4 * i] = g[0]; points[4 * i + 1] = g[1]; points[4 * i + 2] = g[2];
    }
    if (ci < 0 || ci == i) {
      if (k != i) {
        memcpy(points + 4 * k, points + 4 * i, sizeof(float) * 4);
        memcpy(normals + 4 * k, normals + 4 * i, sizeof(float) * 4);
        if (statsM) memcpy(statsM + 16 * k, statsM + 16 * i, sizeof(float) * 16);
        if (omegaP) memcpy(omegaP + 16 * k, omegaP + 16 * i, sizeof(float) * 16);
        if (omegaN) memcpy(omegaN + 16 * k, omegaN + 16 * i, sizeof(float) * 16);
        memcpy(gauss + (size_t)ORC_GAUSS_FLOATS * k, gauss + (size_t)ORC_GAUSS_FLOATS * i, sizeof(float) * ORC_GAUSS_FLOATS);
        gflags[k] = gflags[i];
      }
      k++;
    }
  }
  if (collapsedOut) memcpy(collapsedOut, collapsed, sizeof(int) * n);
  free(indexImage); free(depthImage); free(collapsed);
  return k;
}

/* ---- exported for oracle/shim (the Eigen stand-in the reference's own sources are compiled against): the numerical
 * kernels of Eigen that stay "unpinned" are these very restatements ---- */
void orc_sym_pinv6(const float H[36], float Hi[36]) { sym_pinv6(H, Hi); }
void orc_mat6_inverse(const float A[36], float Ai[36]) { mat6_inverse(A, Ai); }
void orc_sym_singular_values3(const float A[9], float sv[3]) {
  double M[9], V[9], w[3];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) M[c * 3 + r] = 0.5 * ((double)A[c * 3 + r] + (double)A[r * 3 + c]);
  jacobi_sym(3, M, V, w);
  for (int i = 0; i < 3; i++) w[i] = fabs(w[i]);
  for (int i = 0; i < 3; i++)
    for (int j = i + 1; j < 3; j++)
      if (w[j] > w[i]) { double t = w[i]; w[i] = w[j]; w[j] = t; }
  for (int i = 0; i < 3; i++) sv[i] = (float)w[i];
}

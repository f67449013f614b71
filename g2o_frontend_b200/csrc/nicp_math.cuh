// nicp_math.cuh -- small fixed-size float32 math shared by host and device code.
//
// Everything that decides an index, a gate or a stored cloud attribute is evaluated with
// explicitly rounded operations (__fmul_rn/__fadd_rn on the device: never contracted into FMA,
// in either build), in the one evaluation order SURVEY.md Appendix A fixes for the Eigen
// expressions of pwn_core:  ((a0*b0 + a1*b1) + a2*b2) + a3*b3.
// Only the Linearizer's H/b term (corr_linearize.cu) uses ordinary operators and may be
// contracted in the default build; the --fmad=false build is bit-reproducible end to end.
//
// Matrices are column-major like Eigen: M(r,c) = m[c*R + r].
#pragma once
#include <cfloat>
#include <cmath>
#include <cstring>

#if defined(__CUDACC__)
#define NICP_HD __host__ __device__ __forceinline__
#else
#define NICP_HD inline
#endif

namespace nicp {

#if defined(__CUDA_ARCH__)
NICP_HD float fmul(float a, float b) { return __fmul_rn(a, b); }
NICP_HD float fadd(float a, float b) { return __fadd_rn(a, b); }
NICP_HD float fsub(float a, float b) { return __fsub_rn(a, b); }
NICP_HD float fdiv(float a, float b) { return __fdiv_rn(a, b); }
NICP_HD float fsqrt(float a) { return __fsqrt_rn(a); }
NICP_HD float frcp(float a) { return __frcp_rn(a); }  // correctly rounded 1/a == 1.0f / a, fewer instructions than fdiv
#else
// host: compiled with -ffp-contract=off
NICP_HD float fmul(float a, float b) { return a * b; }
NICP_HD float fadd(float a, float b) { return a + b; }
NICP_HD float fsub(float a, float b) { return a - b; }
NICP_HD float fdiv(float a, float b) { return a / b; }
NICP_HD float fsqrt(float a) { return sqrtf(a); }
NICP_HD float frcp(float a) { return 1.0f / a; }
#endif

#define NM4(m, r, c) ((m)[(c) * 4 + (r)])
#define NM3(m, r, c) ((m)[(c) * 3 + (r)])
#define NM6(m, r, c) ((m)[(c) * 6 + (r)])

NICP_HD float dot3(float a0, float a1, float a2, float b0, float b1, float b2) {
  return fadd(fadd(fmul(a0, b0), fmul(a1, b1)), fmul(a2, b2));
}
NICP_HD float dot4(float a0, float a1, float a2, float a3, float b0, float b1, float b2, float b3) {
  return fadd(fadd(fadd(fmul(a0, b0), fmul(a1, b1)), fmul(a2, b2)), fmul(a3, b3));
}

// 3x4 affine part of a column-major 4x4, kept in registers / constant memory
struct Affine {
  float r[3][4];  // r[i][j] = M(i,j)
};
NICP_HD Affine affine_from(const float *m) {
  Affine a;
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 4; j++) a.r[i][j] = NM4(m, i, j);
  return a;
}
// rows 0..2 of M * (x,y,z,1)
// (the product with the homogeneous 1 is exact, so the translation entry is added as it is)
NICP_HD void xform_point(const Affine &a, float x, float y, float z, float &ox, float &oy, float &oz) {
  ox = fadd(dot3(a.r[0][0], a.r[0][1], a.r[0][2], x, y, z), a.r[0][3]);
  oy = fadd(dot3(a.r[1][0], a.r[1][1], a.r[1][2], x, y, z), a.r[1][3]);
  oz = fadd(dot3(a.r[2][0], a.r[2][1], a.r[2][2], x, y, z), a.r[2][3]);
}
// rows 0..2 of M * (x,y,z,0): the translation column contributes an exact zero
NICP_HD void xform_normal(const Affine &a, float x, float y, float z, float &ox, float &oy, float &oz) {
  ox = dot3(a.r[0][0], a.r[0][1], a.r[0][2], x, y, z);
  oy = dot3(a.r[1][0], a.r[1][1], a.r[1][2], x, y, z);
  oz = dot3(a.r[2][0], a.r[2][1], a.r[2][2], x, y, z);
}

NICP_HD void mat4_identity(float *m) {
  for (int i = 0; i < 16; i++) m[i] = 0.0f;
  m[0] = m[5] = m[10] = m[15] = 1.0f;
}
NICP_HD void fix_last_row(float *T) {
  NM4(T, 3, 0) = 0.f; NM4(T, 3, 1) = 0.f; NM4(T, 3, 2) = 0.f; NM4(T, 3, 3) = 1.f;
}

// ---- bm_se3.h -----------------------------------------------------------------------------
// quat2mat (bm_se3.h:9-21) + v2t (:36-43)
NICP_HD void v2t(const float *v, float *T) {
  float qx = v[3], qy = v[4], qz = v[5];
  float qw = fsqrt(fsub(1.f, fadd(fadd(fmul(qx, qx), fmul(qy, qy)), fmul(qz, qz))));
  float ww = fmul(qw, qw), xx = fmul(qx, qx), yy = fmul(qy, qy), zz = fmul(qz, qz);
  mat4_identity(T);
  NM4(T, 0, 0) = fsub(fsub(fadd(ww, xx), yy), zz);
  NM4(T, 0, 1) = fmul(2.f, fsub(fmul(qx, qy), fmul(qw, qz)));
  NM4(T, 0, 2) = fmul(2.f, fadd(fmul(qx, qz), fmul(qw, qy)));
  NM4(T, 1, 0) = fmul(2.f, fadd(fmul(qx, qy), fmul(qz, qw)));
  NM4(T, 1, 1) = fsub(fadd(fsub(ww, xx), yy), zz);
  NM4(T, 1, 2) = fmul(2.f, fsub(fmul(qy, qz), fmul(qx, qw)));
  NM4(T, 2, 0) = fmul(2.f, fsub(fmul(qx, qz), fmul(qy, qw)));
  NM4(T, 2, 1) = fmul(2.f, fadd(fmul(qy, qz), fmul(qx, qw)));
  NM4(T, 2, 2) = fadd(fsub(fsub(ww, xx), yy), zz);
  NM4(T, 0, 3) = v[0];
  NM4(T, 1, 3) = v[1];
  NM4(T, 2, 3) = v[2];
}
// mat2quat (bm_se3.h:24-34: Eigen::Quaternion(R), normalize, sign) + t2v (:45-52)
NICP_HD void t2v(const float *T, float *v) {
  float q[4];  // x y z w
  float t = fadd(fadd(NM4(T, 0, 0), NM4(T, 1, 1)), NM4(T, 2, 2));
  if (t > 0.f) {
    t = fsqrt(fadd(t, 1.0f));
    q[3] = fmul(0.5f, t);
    t = fdiv(0.5f, t);
    q[0] = fmul(fsub(NM4(T, 2, 1), NM4(T, 1, 2)), t);
    q[1] = fmul(fsub(NM4(T, 0, 2), NM4(T, 2, 0)), t);
    q[2] = fmul(fsub(NM4(T, 1, 0), NM4(T, 0, 1)), t);
  } else {
    // i = index of the largest diagonal entry (ties -> lowest), j = (i+1)%3, k = (j+1)%3; written out per case so
    // that every array index is a compile-time constant (the matrices stay in registers on the device)
    int i = 0;
    if (NM4(T, 1, 1) > NM4(T, 0, 0)) i = 1;
    if (NM4(T, 2, 2) > (i == 1 ? NM4(T, 1, 1) : NM4(T, 0, 0))) i = 2;
#define NICP_T2V_CASE(I, J, K)                                                                      \
  {                                                                                                 \
    t = fsqrt(fadd(fsub(fsub(NM4(T, I, I), NM4(T, J, J)), NM4(T, K, K)), 1.0f));                    \
    q[I] = fmul(0.5f, t);                                                                           \
    t = fdiv(0.5f, t);                                                                              \
    q[3] = fmul(fsub(NM4(T, K, J), NM4(T, J, K)), t);                                               \
    q[J] = fmul(fadd(NM4(T, J, I), NM4(T, I, J)), t);                                               \
    q[K] = fmul(fadd(NM4(T, K, I), NM4(T, I, K)), t);                                               \
  }
    if (i == 0) NICP_T2V_CASE(0, 1, 2)
    else if (i == 1) NICP_T2V_CASE(1, 2, 0)
    else NICP_T2V_CASE(2, 0, 1)
#undef NICP_T2V_CASE
  }
  float nrm = fsqrt(fadd(fadd(fadd(fmul(q[0], q[0]), fmul(q[1], q[1])), fmul(q[2], q[2])), fmul(q[3], q[3])));
  for (int i = 0; i < 4; i++) q[i] = fdiv(q[i], nrm);
  v[0] = NM4(T, 0, 3);
  v[1] = NM4(T, 1, 3);
  v[2] = NM4(T, 2, 3);
  if (q[3] < 0) { v[3] = -q[0]; v[4] = -q[1]; v[5] = -q[2]; }
  else          { v[3] =  q[0]; v[4] =  q[1]; v[5] =  q[2]; }
}
// Eigen Isometry3f::inverse(): R' = R^T, t' = -(R^T t).  Safe when Ti aliases T.
NICP_HD void iso_inverse(const float *T, float *Ti) {
  float o[16];
  mat4_identity(o);
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) NM4(o, r, c) = NM4(T, c, r);
  for (int r = 0; r < 3; r++)
    NM4(o, r, 3) = -dot3(NM4(o, r, 0), NM4(o, r, 1), NM4(o, r, 2), NM4(T, 0, 3), NM4(T, 1, 3), NM4(T, 2, 3));
  for (int i = 0; i < 16; i++) Ti[i] = o[i];
}
// Isometry * Isometry.  Safe when C aliases A or B.
NICP_HD void iso_mul(const float *A, const float *B, float *C) {
  float o[16];
  mat4_identity(o);
  for (int r = 0; r < 3; r++) {
    for (int c = 0; c < 3; c++)
      NM4(o, r, c) = dot3(NM4(A, r, 0), NM4(A, r, 1), NM4(A, r, 2), NM4(B, 0, c), NM4(B, 1, c), NM4(B, 2, c));
    NM4(o, r, 3) = fadd(dot3(NM4(A, r, 0), NM4(A, r, 1), NM4(A, r, 2), NM4(B, 0, 3), NM4(B, 1, 3), NM4(B, 2, 3)), NM4(A, r, 3));
  }
  for (int i = 0; i < 16; i++) C[i] = o[i];
}

// R * Om * R^T for the 3x3 blocks, R = the rotation of the 4x4 M (InformationMatrixVector::transformInPlace,
// informationmatrix.h:111-121)
NICP_HD void rotate_sym(const float *M, const float *Om /*3x3 col-major*/, float *out) {
  float t[9];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++)
      NM3(t, r, c) = dot3(NM4(M, r, 0), NM4(M, r, 1), NM4(M, r, 2), NM3(Om, 0, c), NM3(Om, 1, c), NM3(Om, 2, c));
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++)
      NM3(out, r, c) = dot3(NM3(t, r, 0), NM3(t, r, 1), NM3(t, r, 2), NM4(M, c, 0), NM4(M, c, 1), NM4(M, c, 2));
}

// ---- PinholePointProjector::_updateMatrices (pinholepointprojector.cpp:17-31) ---------------
NICP_HD float cof3(const float *m, int i, int j) {
  int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
  return fsub(fmul(NM3(m, i1, j1), NM3(m, i2, j2)), fmul(NM3(m, i1, j2), NM3(m, i2, j1)));
}
// Eigen 3x3 inverse: cofactors / determinant
NICP_HD void mat3_inverse(const float *m, float *inv) {
  float c00 = cof3(m, 0, 0), c10 = cof3(m, 1, 0), c20 = cof3(m, 2, 0);
  float det = fadd(fadd(fmul(c00, NM3(m, 0, 0)), fmul(c10, NM3(m, 1, 0))), fmul(c20, NM3(m, 2, 0)));
  float invdet = fdiv(1.0f, det);
  NM3(inv, 0, 0) = fmul(c00, invdet);
  NM3(inv, 0, 1) = fmul(c10, invdet);
  NM3(inv, 0, 2) = fmul(c20, invdet);
  NM3(inv, 1, 0) = fmul(cof3(m, 0, 1), invdet);
  NM3(inv, 1, 1) = fmul(cof3(m, 1, 1), invdet);
  NM3(inv, 1, 2) = fmul(cof3(m, 2, 1), invdet);
  NM3(inv, 2, 0) = fmul(cof3(m, 0, 2), invdet);
  NM3(inv, 2, 1) = fmul(cof3(m, 1, 2), invdet);
  NM3(inv, 2, 2) = fmul(cof3(m, 2, 2), invdet);
}
// KRt = [K R^-1, K t_inv], for a projector whose pose is T
NICP_HD void compute_KRt(const float *K, const float *T, float *KRt) {
  float t[16];
  iso_inverse(T, t);
  mat4_identity(KRt);
  for (int r = 0; r < 3; r++) {
    for (int c = 0; c < 3; c++)
      NM4(KRt, r, c) = dot3(NM3(K, r, 0), NM3(K, r, 1), NM3(K, r, 2), NM4(t, 0, c), NM4(t, 1, c), NM4(t, 2, c));
    NM4(KRt, r, 3) = dot3(NM3(K, r, 0), NM3(K, r, 1), NM3(K, r, 2), NM4(t, 0, 3), NM4(t, 1, 3), NM4(t, 2, 3));
  }
}
// iKRt = [R K^-1, t]
NICP_HD void compute_iKRt(const float *K, const float *T, float *iKRt) {
  float iK[9];
  mat3_inverse(K, iK);
  mat4_identity(iKRt);
  for (int r = 0; r < 3; r++) {
    for (int c = 0; c < 3; c++)
      NM4(iKRt, r, c) = dot3(NM4(T, r, 0), NM4(T, r, 1), NM4(T, r, 2), NM3(iK, 0, c), NM3(iK, 1, c), NM3(iK, 2, c));
    NM4(iKRt, r, 3) = NM4(T, r, 3);
  }
}

// ---- Eigen::LDLT<Matrix6f> compute + solve (Eigen 3.2 unblocked, diagonal pivoting) ----------
// x = H^-1 b (aligner.cpp:110 calls it with -b)
NICP_HD void ldlt_solve6(const float *Hin, const float *bin, float *x) {
  // Every loop has compile-time bounds and every array index is a compile-time constant after unrolling; the
  // data-dependent pivot is applied as predicated swaps against each candidate row.  (On the device this keeps
  // the 6x6 in registers: the solving thread is a single thread on the critical path of every iteration.)
  const int N = 6;
  float m[36];
  int tr[6];
#pragma unroll
  for (int i = 0; i < 36; i++) m[i] = Hin[i];
#pragma unroll
  for (int k = 0; k < N; k++) {
    int big = k;
    float bv = fabsf(NM6(m, k, k));
#pragma unroll
    for (int i = k + 1; i < N; i++) {
      float a = fabsf(NM6(m, i, i));
      if (a > bv) { bv = a; big = i; }
    }
    tr[k] = big;
    // symmetric row/column swap k <-> big in the lower triangle
#pragma unroll
    for (int cand = k + 1; cand < N; cand++) {
      if (cand == big) {
        float t;
#pragma unroll
        for (int j = 0; j < k; j++) { t = NM6(m, k, j); NM6(m, k, j) = NM6(m, cand, j); NM6(m, cand, j) = t; }
#pragma unroll
        for (int i = cand + 1; i < N; i++) { t = NM6(m, i, k); NM6(m, i, k) = NM6(m, i, cand); NM6(m, i, cand) = t; }
        t = NM6(m, k, k); NM6(m, k, k) = NM6(m, cand, cand); NM6(m, cand, cand) = t;
#pragma unroll
        for (int i = k + 1; i < cand; i++) { t = NM6(m, i, k); NM6(m, i, k) = NM6(m, cand, i); NM6(m, cand, i) = t; }
      }
    }
    if (k > 0) {
      float temp[6];
#pragma unroll
      for (int j = 0; j < k; j++) temp[j] = fmul(NM6(m, j, j), NM6(m, k, j));
      float s = 0.0f;
#pragma unroll
      for (int j = 0; j < k; j++) s = fadd(s, fmul(NM6(m, k, j), temp[j]));
      NM6(m, k, k) = fsub(NM6(m, k, k), s);
#pragma unroll
      for (int i = k + 1; i < N; i++) {
        float s2 = 0.0f;
#pragma unroll
        for (int j = 0; j < k; j++) s2 = fadd(s2, fmul(NM6(m, i, j), temp[j]));
        NM6(m, i, k) = fsub(NM6(m, i, k), s2);
      }
    }
    float akk = NM6(m, k, k);
    if (fabsf(akk) > 0.0f) {
#pragma unroll
      for (int i = k + 1; i < N; i++) NM6(m, i, k) = fdiv(NM6(m, i, k), akk);
    }
  }
  float y[6];
#pragma unroll
  for (int i = 0; i < N; i++) y[i] = bin[i];
  // y = P b: transpositions applied in order
#pragma unroll
  for (int k = 0; k < N; k++) {
#pragma unroll
    for (int cand = k + 1; cand < N; cand++)
      if (cand == tr[k]) { float t = y[k]; y[k] = y[cand]; y[cand] = t; }
  }
#pragma unroll
  for (int i = 0; i < N; i++) {
    float s = y[i];
#pragma unroll
    for (int j = 0; j < i; j++) s = fsub(s, fmul(NM6(m, i, j), y[j]));
    y[i] = s;
  }
#pragma unroll
  for (int i = 0; i < N; i++) {
    float d = NM6(m, i, i);
    y[i] = (fabsf(d) > FLT_MIN) ? fdiv(y[i], d) : 0.0f;
  }
#pragma unroll
  for (int i = N - 1; i >= 0; i--) {
    float s = y[i];
#pragma unroll
    for (int j = i + 1; j < N; j++) s = fsub(s, fmul(NM6(m, j, i), y[j]));
    y[i] = s;
  }
  // x = P^T y: transpositions in reverse order
#pragma unroll
  for (int k = N - 1; k >= 0; k--) {
#pragma unroll
    for (int cand = k + 1; cand < N; cand++)
      if (cand == tr[k]) { float t = y[k]; y[k] = y[cand]; y[cand] = t; }
  }
#pragma unroll
  for (int i = 0; i < N; i++) x[i] = y[i];
}

}  // namespace nicp

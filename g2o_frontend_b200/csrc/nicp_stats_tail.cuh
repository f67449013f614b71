// nicp_stats_tail.cuh -- the dense tail of Aligner::_computeStatistics (aligner.cpp:172-198, unscented.h:23-65):
// Sigma = pinv(H + I), 13 sigma points (alpha 1e-3, beta 2), remap t2v(T * v2t(s)^-1), rebuild mean / covariance,
// Omega = cov^-1, eigen-ratios of Omega's two 3x3 blocks.
//
// ONE implementation for the host and the device: a single alignment finishes it on the host (3.8 us, no kernel on the
// critical path), a batch runs it on the device, one thread per pair, right after the statistics linearisation -- and a
// pair must get the same omega bits either way.  Every operation is therefore spelled out with explicitly rounded
// wrappers (float: nicp_math.cuh; double: below); no contraction, no library call except IEEE sqrt.
// JacobiSVD / Matrix6f::inverse() of the reference are replaced by a float64 cyclic Jacobi and a float64 Gauss-Jordan
// (tolerance-level parity, like the oracle: DESIGN.md section 5).
#pragma once
#include <cstring>
#include "nicp_math.cuh"

namespace nicp {

#if defined(__CUDA_ARCH__)
NICP_HD double dmul(double a, double b) { return __dmul_rn(a, b); }
NICP_HD double dadd(double a, double b) { return __dadd_rn(a, b); }
NICP_HD double dsub(double a, double b) { return __dsub_rn(a, b); }
NICP_HD double ddiv(double a, double b) { return __ddiv_rn(a, b); }
NICP_HD double dsqrt(double a) { return __dsqrt_rn(a); }
#else
NICP_HD double dmul(double a, double b) { return a * b; }
NICP_HD double dadd(double a, double b) { return a + b; }
NICP_HD double dsub(double a, double b) { return a - b; }
NICP_HD double ddiv(double a, double b) { return a / b; }
NICP_HD double dsqrt(double a) { return sqrt(a); }
#endif

// cyclic Jacobi eigen-decomposition of a symmetric N x N matrix (row-major A is destroyed; V rows = eigenvectors)
template <int N>
NICP_HD void jacobi_sym(double *A, double *V, double *w) {
  for (int i = 0; i < N * N; i++) V[i] = 0.0;
  for (int i = 0; i < N; i++) V[i * N + i] = 1.0;
  for (int sweep = 0; sweep < 60; sweep++) {
    double off = 0.0, diag = 0.0;
    for (int p = 0; p < N; p++) {
      diag = dadd(diag, dmul(A[p * N + p], A[p * N + p]));
      for (int q = p + 1; q < N; q++) off = dadd(off, dmul(A[q * N + p], A[q * N + p]));
    }
    if (off <= dmul(1e-32, dadd(diag, off))) break;  // converged to double precision
    for (int p = 0; p < N; p++)
      for (int q = p + 1; q < N; q++) {
        const double apq = A[q * N + p];
        if (fabs(apq) < 1e-300) continue;
        const double app = A[p * N + p], aqq = A[q * N + q];
        const double tau = ddiv(dsub(aqq, app), dmul(2.0, apq));
        const double t = ddiv(tau >= 0.0 ? 1.0 : -1.0, dadd(fabs(tau), dsqrt(dadd(1.0, dmul(tau, tau)))));
        const double c = ddiv(1.0, dsqrt(dadd(1.0, dmul(t, t)))), s = dmul(t, c);
        for (int k = 0; k < N; k++) {
          const double akp = A[p * N + k], akq = A[q * N + k];
          A[p * N + k] = dsub(dmul(c, akp), dmul(s, akq));
          A[q * N + k] = dadd(dmul(s, akp), dmul(c, akq));
        }
        for (int k = 0; k < N; k++) {
          const double apk = A[k * N + p], aqk = A[k * N + q];
          A[k * N + p] = dsub(dmul(c, apk), dmul(s, aqk));
          A[k * N + q] = dadd(dmul(s, apk), dmul(c, aqk));
        }
        for (int k = 0; k < N; k++) {
          const double vkp = V[p * N + k], vkq = V[q * N + k];
          V[p * N + k] = dsub(dmul(c, vkp), dmul(s, vkq));
          V[q * N + k] = dadd(dmul(s, vkp), dmul(c, vkq));
        }
      }
  }
  for (int i = 0; i < N; i++) w[i] = A[i * N + i];
}

// pseudo-inverse of the symmetrised 6x6 H (JacobiSVD + threshold in the reference, aligner.cpp:172-173)
NICP_HD void stats_sym_pinv6(const float *H, float *Hi) {
  double A[36], V[36], w[6];
  for (int r = 0; r < 6; r++)
    for (int c = 0; c < 6; c++) A[c * 6 + r] = dmul(0.5, dadd((double)NM6(H, r, c), (double)NM6(H, c, r)));
  jacobi_sym<6>(A, V, w);
  double wmax = 0.0;
  for (int i = 0; i < 6; i++)
    if (fabs(w[i]) > wmax) wmax = fabs(w[i]);
  const double thr = dmul(dmul(wmax, 6.0), (double)FLT_EPSILON);
  for (int r = 0; r < 6; r++)
    for (int c = 0; c < 6; c++) {
      double s = 0.0;
      for (int k = 0; k < 6; k++)
        if (fabs(w[k]) > thr) s = dadd(s, ddiv(dmul(V[k * 6 + r], V[k * 6 + c]), w[k]));
      NM6(Hi, r, c) = (float)s;
    }
}

// general 6x6 inverse: float64 Gauss-Jordan with partial pivoting (Matrix6f::inverse() in the reference, aligner.cpp:190)
NICP_HD void stats_mat6_inverse(const float *A, float *Ai) {
  double a[6][12];
  for (int r = 0; r < 6; r++)
    for (int c = 0; c < 6; c++) {
      a[r][c] = (double)NM6(A, r, c);
      a[r][c + 6] = (r == c) ? 1.0 : 0.0;
    }
  for (int k = 0; k < 6; k++) {
    int piv = k;
    for (int r = k + 1; r < 6; r++)
      if (fabs(a[r][k]) > fabs(a[piv][k])) piv = r;
    if (piv != k)
      for (int c = 0; c < 12; c++) { const double t = a[k][c]; a[k][c] = a[piv][c]; a[piv][c] = t; }
    const double d = a[k][k];
    for (int c = 0; c < 12; c++) a[k][c] = ddiv(a[k][c], d);
    for (int r = 0; r < 6; r++)
      if (r != k) {
        const double f = a[r][k];
        if (f != 0.0)
          for (int c = 0; c < 12; c++) a[r][c] = dsub(a[r][c], dmul(f, a[k][c]));
      }
  }
  for (int r = 0; r < 6; r++)
    for (int c = 0; c < 6; c++) NM6(Ai, r, c) = (float)a[r][c + 6];
}

// largest / smallest |eigenvalue| of the symmetrised 3x3 block of O at (off, off) (aligner.cpp:192-198)
NICP_HD float stats_sym_eig_ratio3(const float *O, int off) {
  double A[9], V[9], w[3];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) A[c * 3 + r] = dmul(0.5, dadd((double)NM6(O, off + r, off + c), (double)NM6(O, off + c, off + r)));
  jacobi_sym<3>(A, V, w);
  double mx = 0.0, mn = 1e300;
  for (int i = 0; i < 3; i++) {
    const double a = fabs(w[i]);
    if (a > mx) mx = a;
    if (a < mn) mn = a;
  }
  return (float)ddiv(mx, mn);
}

// x, or the quiet NaN 0x7fc00000 if x is any NaN.  A weak or degenerate H makes NaNs in the tail (a sigma point with
// |q| > 1 takes sqrt of a negative number in v2t; a direction dropped by the pseudo-inverse makes the Cholesky divide
// 0 by 0), and x86 and sm_100a arithmetic give those NaNs different sign and payload bits: one NaN for the record keeps
// the host's single-alignment record and the device's batch record byte-identical.
NICP_HD float canonical_nan(float x) {
  if (x == x) return x;
#if defined(__CUDA_ARCH__)
  return __int_as_float(0x7fc00000);
#else
  const unsigned int q = 0x7fc00000u;
  float f;
  memcpy(&f, &q, sizeof f);
  return f;
#endif
}

// H_lin: the linearisation at the final T (column-major 6x6); T column-major 4x4.  Omega (36), two ratios; every NaN
// among them is canonical_nan's.
NICP_HD void compute_statistics_tail(const float *H_lin, const float *T, float *Omega, float *tr, float *rr) {
  float H[36], Sigma[36];
  for (int i = 0; i < 36; i++) H[i] = H_lin[i];
  for (int i = 0; i < 6; i++) NM6(H, i, i) = fadd(NM6(H, i, i), 1.0f);
  stats_sym_pinv6(H, Sigma);
  const int dim = 6;
  const double alpha = 1e-3, beta = 2.0;
  const double lambda = dmul(dmul(alpha, alpha), (double)dim);
  const double wi = ddiv(1.0, dmul(2.0, dadd((double)dim, lambda)));
  double wm[13], wc[13];
  float samples[13][6];
  for (int i = 0; i < 13; i++)
    for (int r = 0; r < 6; r++) samples[i][r] = 0.0f;
  wm[0] = ddiv(lambda, dadd((double)dim, lambda));
  wc[0] = dadd(ddiv(lambda, dadd((double)dim, lambda)), dadd(dsub(1.0, dmul(alpha, alpha)), beta));
  // Cholesky factor of (dim + lambda) * Sigma (LLT, unscented.h:38-42), float32
  float A[36], L[36];
  for (int i = 0; i < 36; i++) L[i] = 0.0f;
  const float sc = (float)dadd((double)dim, lambda);
  for (int i = 0; i < 36; i++) A[i] = fmul(Sigma[i], sc);
  for (int j = 0; j < 6; j++) {
    float s = NM6(A, j, j);
    for (int k = 0; k < j; k++) s = fsub(s, fmul(NM6(L, j, k), NM6(L, j, k)));
    const float d = fsqrt(s);
    NM6(L, j, j) = d;
    for (int i = j + 1; i < 6; i++) {
      float t = NM6(A, i, j);
      for (int k = 0; k < j; k++) t = fsub(t, fmul(NM6(L, i, k), NM6(L, j, k)));
      NM6(L, i, j) = fdiv(t, d);
    }
  }
  int k = 1;
  for (int i = 0; i < dim; i++) {
    for (int r = 0; r < 6; r++) {
      samples[k][r] = NM6(L, r, i);
      samples[k + 1][r] = -NM6(L, r, i);
    }
    wm[k] = wc[k] = wi;
    wm[k + 1] = wc[k + 1] = wi;
    k += 2;
  }
  for (int i = 0; i < 13; i++) {
    float X[16], Xi[16], Y[16];
    v2t(samples[i], X);
    iso_inverse(X, Xi);
    iso_mul(T, Xi, Y);
    t2v(Y, samples[i]);
  }
  float mean[6] = {0, 0, 0, 0, 0, 0};
  for (int i = 0; i < 13; i++)
    for (int r = 0; r < 6; r++) mean[r] = fadd(mean[r], (float)dmul(wm[i], (double)samples[i][r]));
  float cov[36];
  for (int i = 0; i < 36; i++) cov[i] = 0.0f;
  for (int i = 0; i < 13; i++) {
    float dl[6];
    for (int r = 0; r < 6; r++) dl[r] = fsub(samples[i][r], mean[r]);
    for (int r = 0; r < 6; r++)
      for (int c = 0; c < 6; c++) NM6(cov, r, c) = fadd(NM6(cov, r, c), (float)dmul(wc[i], (double)fmul(dl[r], dl[c])));
  }
  stats_mat6_inverse(cov, Omega);
  *tr = canonical_nan(stats_sym_eig_ratio3(Omega, 0));
  *rr = canonical_nan(stats_sym_eig_ratio3(Omega, 3));
  for (int i = 0; i < 36; i++) Omega[i] = canonical_nan(Omega[i]);
}

}  // namespace nicp

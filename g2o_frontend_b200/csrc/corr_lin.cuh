// corr_lin.cuh -- the fused CorrespondenceFinder::compute + Linearizer::update kernels: k_corr_lin_group and
// k_corr_lin_tiled.
//
//   CorrespondenceFinder::compute   correspondencefinder.cpp:20-118
//   Linearizer::update              linearizer.cpp:17-115
//   PwnMatcherBase::matchClouds     pwn_tracker2/pwn_matcher_base.cpp:167-196 (image statistics, MODE 1)
//
// k_corr_lin_group: one warp owns a 96-pixel tile (3 pixels per lane) of a GROUP of pairs that share their current cloud
// -- the shape of loop-closure candidate verification, where one frame is matched against many candidates
// (pwn_closer.cpp:92-105).  The current side of the tile (index image, point, normal + curvature, Omega_P / Omega_N) is
// loaded ONCE and kept in registers / shared memory while the warp walks the pairs of the group; per pair it only fetches
// the reference z-buffer words and the reference point / normal gathers, so the current cloud stops being re-read (and
// its addresses re-computed) for every pair.
// k_corr_lin_tiled: one warp owns a 96-pixel tile of one pair (lone pairs, single alignments).
// Both kernels compute a (pair, tile) with the same term, lane / pixel mapping and butterfly, so its partial row has the
// same bits whichever kernel and whichever group computed it.
//
// The Linearizer term runs its point half and its normal half in the two lanes of Blackwell's packed FP32 instructions
// (fma.rn.f32x2 / mul / add -> FFMA2 / FMUL2 / FADD2, sm_100): Omega_P / Omega_N are stored interleaved (Omega3) so a
// 128-bit load leaves (P_ij, N_ij) in an aligned register pair.  Measured on a B200 (tools/microbench/fp32_pipes.cu):
// FFMA2 issues at half the rate of FFMA for twice the work, i.e. the same FP32 rate for half the issue slots, and the
// kernel was bound by issue slots (profiles/r2_summary.md).  Every operation of the term is spelled out (no contraction
// left to the compiler), so both builds and every instantiation produce the same H and b bits.
#pragma once
#include "nicp_internal.cuh"

namespace nicp {

// ---- packed FP32 pairs ------------------------------------------------------------------------------------------
typedef unsigned long long f32x2;  // (lo, hi)
__device__ __forceinline__ f32x2 pk(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ float lo_of(f32x2 v) {
  float a, b;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
  return a;
}
__device__ __forceinline__ float hi_of(f32x2 v) {
  float a, b;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
  return b;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

// accumulators of one (pair, tile): scalar sums for what only the point half feeds, packed (point, normal) sums for Hrr / br
struct TermAcc {
  float htt[6];    // sum Omega_P (xx xy xz yy yz zz)
  float htr[9];    // sum Omega_P * S_p, row-major
  f32x2 hrr[6];    // (S_p^T Omega_P S_p, S_n^T Omega_N S_n) upper triangle
  float bt[3];
  f32x2 br[3];
  float err, inl;
};
__device__ __forceinline__ void term_clear(TermAcc &A) {
#pragma unroll
  for (int i = 0; i < 6; i++) { A.htt[i] = 0.0f; A.hrr[i] = 0ull; }
#pragma unroll
  for (int i = 0; i < 9; i++) A.htr[i] = 0.0f;
#pragma unroll
  for (int i = 0; i < 3; i++) { A.bt[i] = 0.0f; A.br[i] = 0ull; }
  A.err = 0.0f;
  A.inl = 0.0f;
}

// one correspondence (linearizer.cpp:56-89), executed by every lane of the warp: `w` is 1 for the lanes whose pixel was
// accepted and 0 for the others, whose Omega is multiplied away (everything below is linear in Omega, and every input is
// finite -- the shared-memory slots are zero-filled at kernel start), so there is no divergent control flow around the
// accumulators.  R = transformed reference (point, normal) per axis, packed; E0..E2 = the errors (rp - cp, rn - cn) per
// axis, packed;
// A=(a,g) B=(b,h) C=(c,i) D=(d,j) E=(e,k) F=(f,l) with Omega_P = [a b c; b d e; c e f], Omega_N = [g h i; h j k; i k l].
template <bool ROBUST, bool MASKED = true>
__device__ __forceinline__ void term_add_e(TermAcc &acc, float w, f32x2 Rx, f32x2 Ry, f32x2 Rz, f32x2 E0, f32x2 E1, f32x2 E2,
                                           f32x2 A, f32x2 B, f32x2 C, f32x2 D, f32x2 E, f32x2 F, float maxChi2) {
  if (MASKED) {  // (w == 1 for every caller with MASKED = false: the product with 1 is exact, the bits do not change)
    const f32x2 W = pk(w, w);
    A = mul2(A, W); B = mul2(B, W); C = mul2(C, W); D = mul2(D, W); E = mul2(E, W); F = mul2(F, W);
  }
  // Omega e, rows: (a e0 + b e1) + c e2 ...
  f32x2 W0 = fma2(C, E2, fma2(B, E1, mul2(A, E0)));
  f32x2 W1 = fma2(E, E2, fma2(D, E1, mul2(B, E0)));
  f32x2 W2 = fma2(F, E2, fma2(E, E1, mul2(C, E0)));
  const f32x2 chi2 = fma2(E2, W2, fma2(E1, W1, mul2(E0, W0)));
  float chi = __fadd_rn(lo_of(chi2), hi_of(chi2));
  float ks = 1.0f;
  if (ROBUST) {
    // sqrt(maxChi2 / chi) (linearizer.cpp:66-71) as r * rsqrt(r): two special-function results and a select, where sqrtf
    // brings a divergent region with its own slow-path call into every pixel slot; 2 ulp from the rounded square root
    // (the scale only weighs outlier terms in b and the error; H / b tolerance 1e-4).  chi = 0: inf * 0 is selected away.
    const float r = __fdividef(maxChi2, chi);
    float rs;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rs) : "f"(r));
    ks = chi > maxChi2 ? __fmul_rn(r, rs) : 1.0f;
  } else {
    // without the robust kernel such a correspondence is skipped altogether (linearizer.cpp:66-71): multiplied away
    const float keep = chi > maxChi2 ? 0.0f : 1.0f;
    const f32x2 K2 = pk(keep, keep);
    A = mul2(A, K2); B = mul2(B, K2); C = mul2(C, K2); D = mul2(D, K2); E = mul2(E, K2); F = mul2(F, K2);
    W0 = mul2(W0, K2); W1 = mul2(W1, K2); W2 = mul2(W2, K2);
    chi = __fmul_rn(chi, keep);
    w = __fmul_rn(w, keep);
  }
  acc.inl = __fadd_rn(acc.inl, w);
  acc.err = __fmaf_rn(ks, chi, acc.err);
  // skew(v) = -2 [v]x (bm_se3.h:54-66): P = 2 v, NP = -2 v
  const f32x2 two = pk(2.0f, 2.0f), mtwo = pk(-2.0f, -2.0f);
  const f32x2 PX = mul2(Rx, two), PY = mul2(Ry, two), PZ = mul2(Rz, two);
  const f32x2 NX = mul2(Rx, mtwo), NY = mul2(Ry, mtwo), NZ = mul2(Rz, mtwo);
  // M = Omega S (point half: Omega_P S_p, normal half: Omega_N S_n)
  const f32x2 m00 = fma2(C, PY, mul2(B, NZ)), m01 = fma2(A, PZ, mul2(C, NX)), m02 = fma2(B, PX, mul2(A, NY));
  const f32x2 m10 = fma2(E, PY, mul2(D, NZ)), m11 = fma2(B, PZ, mul2(E, NX)), m12 = fma2(D, PX, mul2(B, NY));
  const f32x2 m20 = fma2(F, PY, mul2(E, NZ)), m21 = fma2(C, PZ, mul2(F, NX)), m22 = fma2(E, PX, mul2(C, NY));
  acc.htt[0] = __fadd_rn(acc.htt[0], lo_of(A)); acc.htt[1] = __fadd_rn(acc.htt[1], lo_of(B));
  acc.htt[2] = __fadd_rn(acc.htt[2], lo_of(C)); acc.htt[3] = __fadd_rn(acc.htt[3], lo_of(D));
  acc.htt[4] = __fadd_rn(acc.htt[4], lo_of(E)); acc.htt[5] = __fadd_rn(acc.htt[5], lo_of(F));
  acc.htr[0] = __fadd_rn(acc.htr[0], lo_of(m00)); acc.htr[1] = __fadd_rn(acc.htr[1], lo_of(m01));
  acc.htr[2] = __fadd_rn(acc.htr[2], lo_of(m02)); acc.htr[3] = __fadd_rn(acc.htr[3], lo_of(m10));
  acc.htr[4] = __fadd_rn(acc.htr[4], lo_of(m11)); acc.htr[5] = __fadd_rn(acc.htr[5], lo_of(m12));
  acc.htr[6] = __fadd_rn(acc.htr[6], lo_of(m20)); acc.htr[7] = __fadd_rn(acc.htr[7], lo_of(m21));
  acc.htr[8] = __fadd_rn(acc.htr[8], lo_of(m22));
  // Hrr = S^T M, upper triangle; S^T rows: (0,-tz,ty) (tz,0,-tx) (-ty,tx,0) with t = 2 v
  acc.hrr[0] = fma2(NZ, m10, fma2(PY, m20, acc.hrr[0]));
  acc.hrr[1] = fma2(NZ, m11, fma2(PY, m21, acc.hrr[1]));
  acc.hrr[2] = fma2(NZ, m12, fma2(PY, m22, acc.hrr[2]));
  acc.hrr[3] = fma2(NX, m21, fma2(PZ, m01, acc.hrr[3]));
  acc.hrr[4] = fma2(NX, m22, fma2(PZ, m02, acc.hrr[4]));
  acc.hrr[5] = fma2(NY, m02, fma2(PX, m12, acc.hrr[5]));
  acc.bt[0] = __fmaf_rn(ks, lo_of(W0), acc.bt[0]);
  acc.bt[1] = __fmaf_rn(ks, lo_of(W1), acc.bt[1]);
  acc.bt[2] = __fmaf_rn(ks, lo_of(W2), acc.bt[2]);
  const f32x2 KS = pk(ks, ks);
  acc.br[0] = fma2(KS, fma2(PY, W2, mul2(NZ, W1)), acc.br[0]);
  acc.br[1] = fma2(KS, fma2(PZ, W0, mul2(NX, W2)), acc.br[1]);
  acc.br[2] = fma2(KS, fma2(PX, W1, mul2(NY, W0)), acc.br[2]);
}
// the same from the current point / normal (per-pair kernel)
template <bool ROBUST, bool MASKED = true>
__device__ __forceinline__ void term_add(TermAcc &acc, float w, f32x2 Rx, f32x2 Ry, f32x2 Rz, float4 cp, float4 cn, f32x2 A, f32x2 B,
                                         f32x2 C, f32x2 D, f32x2 E, f32x2 F, float maxChi2) {
  term_add_e<ROBUST, MASKED>(acc, w, Rx, Ry, Rz, sub2(Rx, pk(cp.x, cn.x)), sub2(Ry, pk(cp.y, cn.y)), sub2(Rz, pk(cp.z, cn.z)), A, B, C,
                             D, E, F, maxChi2);
}

// the 32 reduction slots of a (pair, tile) from the accumulators (slot layout: A_* in nicp_internal.cuh)
__device__ __forceinline__ void term_slots(const TermAcc &A, float (&v)[kAccum]) {
#pragma unroll
  for (int i = 0; i < 6; i++) v[A_HTT + i] = A.htt[i];
#pragma unroll
  for (int i = 0; i < 9; i++) v[A_HTR + i] = A.htr[i];
#pragma unroll
  for (int i = 0; i < 6; i++) v[A_HRR + i] = __fadd_rn(lo_of(A.hrr[i]), hi_of(A.hrr[i]));
#pragma unroll
  for (int i = 0; i < 3; i++) v[A_BT + i] = A.bt[i];
#pragma unroll
  for (int i = 0; i < 3; i++) v[A_BR + i] = __fadd_rn(lo_of(A.br[i]), hi_of(A.br[i]));
  v[A_ERR] = A.err;
  v[A_INL] = A.inl;
}

// transposing warp reduction of 32 values: afterwards lane j holds the warp total of v[j] in v[0]
__device__ __forceinline__ float warp_transpose_reduce(float (&v)[kAccum], int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool upper = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < off; i++) {
      float mine = upper ? v[i + off] : v[i];
      float send = upper ? v[i] : v[i + off];
      v[i] = mine + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

// One warp per tile of kTilePixels pixels in both kernels: lane l owns pixels base + k * 32 + l of pixel slots k = 0..2.
// A (pair, tile) row depends on that mapping, so it is the same constant for both kernels and the host launch code.
constexpr int kTileLanes = 32, kTileSlots = 3, kTilePixels = kTileLanes * kTileSlots;

// per-lane slots (lane l, pixel slot k -> [k * 32 + l]): nothing here is shared between lanes except T; shared memory is
// used as a register file extension -- for what must survive the walk over the pairs of the group, and as the landing
// zone of the reference gathers, which are issued with cp.async one pair AHEAD of the pair being computed (no registers
// are held while they are in flight)
struct GroupSmem {      // the current side of the tile and T of every pair
  float4 om[3][kTilePixels];  // Omega_P / Omega_N of the current point (Omega3 layout), cp.async
  float4 c0[kTilePixels];     // current point / normal interleaved like nicp_cloud::pn: (px, nx, py, ny)
  float4 c1[kTilePixels];     // (pz, nz, 1, curvature clamped to flatCurvatureThreshold, or -1 for a zero normal (MODE 0))
  float4 T[kMaxGroup][4];     // state->invT of every pair of the group (column-major), fetched by lane g in the prologue
};
struct GatherStage {    // nicp_cloud::pn records of the pair being computed / the next pair, cp.async
  float4 p0[kTilePixels];     // reference (px, nx, py, ny)
  float4 p1[kTilePixels];     // reference (pz, nz, 1, curvature)
};

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
  unsigned int sa = (unsigned int)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}
__device__ __forceinline__ const float4 *shfl_ptr(const float4 *p, int src) {
  unsigned long long v = reinterpret_cast<unsigned long long>(p);
  unsigned int lo = __shfl_sync(0xffffffffu, (unsigned int)v, src), hi = __shfl_sync(0xffffffffu, (unsigned int)(v >> 32), src);
  return reinterpret_cast<const float4 *>(((unsigned long long)hi << 32) | lo);
}

// ---- grouped kernel: one warp walks the pairs of a group over one tile ----
// MODE 0: correspondence gates + linearise at state->invT; the correspondence image is written only when asked for.
// MODE 1: linearise over the stored correspondence image (inner iterations > 0, _computeStatistics) and, if imgStats,
//         accumulate the matchClouds image statistics (slots 29..31).
// Software pipeline over the pairs of the group (one exposed memory round trip per GROUP, not per pair):
//   while pair g is computed out of shared memory, the point / normal gathers of pair g + 1 are landing there (cp.async)
//   and the z-buffer words of pair g + 2 are on their way into registers.  No address is loaded inside the loop: the
//   slot buffers are affine in the slot index (SlotBases), the cloud pointers and T of all pairs are fetched by lane g
//   in the prologue and handed out with shuffles / shared memory.
// Registers are handed out 32 per thread at a time, so anything from 129 to 160 leaves 12 resident one-warp CTAs per SM:
// with that room the three pixel slots run as ONE straight-line block (every slot executed, weights 0 / 1) and the
// compiler interleaves them -- more independent instructions per warp at 3 warps per scheduler (158 registers +
// straight-line 873 us per 256-pair launch, 144 + skipping empty slots 905 us; profiles/r2_summary.md section 3).
template <int MODE, bool ROBUST>
__global__ void __launch_bounds__(kTileLanes, 12) k_corr_lin_group(const PairDesc *__restrict__ desc, const PairGroup *__restrict__ groups,
                                                                   SlotBases B, int epoch, int writeCorr, AlignConsts ac, int numPixels,
                                                                   int imgStats, float imgThreshold, int groupFast, int curEpoch) {
  constexpr int TK = kTileSlots, NT = kTileLanes, TILE = kTilePixels;
  __shared__ GroupSmem S;
  __shared__ GatherStage stage[2];
  // group-fastest block order: the CTAs resident together work on the same tile of different groups, so the reference
  // z-buffer rows and the tile's current-cloud lines they touch stay close in L2
  const int groupId = groupFast ? blockIdx.x : blockIdx.y;
  const int tileId = groupFast ? blockIdx.y : blockIdx.x;
  const int lane = threadIdx.x & 31;
  const int base = tileId * TILE;
  const bool wantZ = MODE == 0 || imgStats;  // the reference z-buffer words are needed (index / depth)
  PairGroup G;
  {
    const uint4 *gp = reinterpret_cast<const uint4 *>(groups + groupId);
    const uint4 g0 = __ldg(gp), g1 = __ldg(gp + 1), g2 = __ldg(gp + 2);
    G.first = (int)g0.x; G.count = (int)g0.y; G.curSlot = (int)g0.z; G.pad = 0;
    G.curPoints = reinterpret_cast<const float4 *>(((unsigned long long)g1.y << 32) | g1.x);
    G.curNormals = reinterpret_cast<const float4 *>(((unsigned long long)g1.w << 32) | g1.z);
    G.curOmega = reinterpret_cast<const float4 *>(((unsigned long long)g2.y << 32) | g2.x);
    G.curPN = reinterpret_cast<const float4 *>(((unsigned long long)g2.w << 32) | g2.z);
  }

  // what identifies the reference side of a pixel for one pair: the z-buffer word (MODE 0: index + epoch; MODE 1 with
  // image statistics: depth) and / or the stored correspondence (MODE 1)
  struct RefKey {
    unsigned long long z[TK];
    int ri[TK];
  };
  auto load_key = [&](int g, RefKey &key) {
    const size_t off = (size_t)(G.first + g) * (size_t)B.slotPixels;
#pragma unroll
    for (int k = 0; k < TK; k++) {
      const int pix = base + k * NT + lane;
      key.z[k] = kEmptyZ;
      key.ri[k] = -1;
      if (pix < numPixels) {
        if (wantZ) key.z[k] = __ldg(B.refZ + off + pix);
        if (MODE == 1) key.ri[k] = __ldg(B.corrImage + off + pix);
      }
    }
  };
  auto issue_gathers = [&](const float4 *refPN, const int (&ri)[TK], const bool (&curOk)[TK], int st) {
#pragma unroll
    for (int k = 0; k < TK; k++) {
      if (ri[k] >= 0 && curOk[k]) {  // the two halves of the point's 32-byte sector
        cp_async16(&stage[st].p0[k * NT + lane], refPN + 2 * (size_t)ri[k]);
        cp_async16(&stage[st].p1[k * NT + lane], refPN + 2 * (size_t)ri[k] + 1);
      }
    }
  };

  // every shared-memory slot of this lane holds finite values from the start (the per-pixel code below is branch free
  // and multiplies what a rejected lane read by zero)
  {
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < TK; k++) {
      S.om[0][k * NT + lane] = z4; S.om[1][k * NT + lane] = z4; S.om[2][k * NT + lane] = z4;
      stage[0].p0[k * NT + lane] = z4; stage[1].p0[k * NT + lane] = z4;
      stage[0].p1[k * NT + lane] = z4; stage[1].p1[k * NT + lane] = z4;
    }
  }
  // ---- prologue: current side of the tile (once per group), keys of pairs 0 and 1, pointers and T of every pair ----
  const int *__restrict__ curIndex = B.curIndex + (size_t)G.curSlot * (size_t)B.slotPixels;
  int ci[TK];
#pragma unroll
  for (int k = 0; k < TK; k++) {
    const int pix = base + k * NT + lane;
    ci[k] = pix < numPixels ? __ldg(curIndex + pix) : -1;
  }
  RefKey keyNext;  // keys of the pair whose gathers are issued next
  if (G.count > 0) load_key(0, keyNext);
  else {
#pragma unroll
    for (int k = 0; k < TK; k++) { keyNext.z[k] = kEmptyZ; keyNext.ri[k] = -1; }
  }
  // lane g fetches what pair g of the group needs: its cloud pointers (kept, handed out by shuffle) and its T (to shared
  // memory); count <= kMaxGroup
  const float4 *myRefPN = nullptr;
  if (lane < G.count) {
    myRefPN = desc[G.first + lane].refPN;
    const float4 *tp = reinterpret_cast<const float4 *>(B.state[G.first + lane].invT);
    S.T[lane][0] = __ldg(tp);
    S.T[lane][1] = __ldg(tp + 1);
    S.T[lane][2] = __ldg(tp + 2);
    S.T[lane][3] = __ldg(tp + 3);
  }
  // nothing of the current cloud projects into this tile: every pair of the group gets a row of zeros (MODE 1 with image
  // statistics still has to look at the reference z-buffer)
  if (!(MODE == 1 && imgStats) && !__any_sync(0xffffffffu, ci[0] >= 0 || ci[1] >= 0 || ci[2] >= 0)) {
    for (int g = 0; g < G.count; g++) {
      B.partials[(size_t)(G.first + g) * (size_t)B.partialStride + (size_t)tileId * kAccum + lane] = 0.0f;
      if (MODE == 0 && writeCorr) {
        int *__restrict__ corrImage = B.corrImage + (size_t)(G.first + g) * (size_t)B.slotPixels;
#pragma unroll
        for (int k = 0; k < TK; k++) {
          const int pix = base + k * NT + lane;
          if (pix < numPixels) corrImage[pix] = -1;
        }
      }
    }
    return;
  }
  unsigned long long zc[TK];
  if (MODE == 1 && imgStats) {
    const unsigned long long *__restrict__ zcur = B.curZ + (size_t)G.curSlot * (size_t)B.slotPixels;
#pragma unroll
    for (int k = 0; k < TK; k++) {
      const int pix = base + k * NT + lane;
      zc[k] = pix < numPixels ? __ldg(zcur + pix) : kEmptyZ;
    }
  }
  bool curOk[TK];
  int riCur[TK];                 // reference indices of the pair being computed
  unsigned long long zCur[TK];   // its z-buffer words (image statistics)
  {
    float4 c0l[TK], c1l[TK];
#pragma unroll
    for (int k = 0; k < TK; k++) {
      curOk[k] = ci[k] >= 0;
      c0l[k] = make_float4(0.f, 0.f, 0.f, 0.f);
      c1l[k] = make_float4(0.f, 0.f, 1.f, 0.f);
      if (curOk[k]) {
        const float4 *om = G.curOmega + 3 * (size_t)ci[k];
        cp_async16(&S.om[0][k * NT + lane], om);
        cp_async16(&S.om[1][k * NT + lane], om + 1);
        cp_async16(&S.om[2][k * NT + lane], om + 2);
        c0l[k] = __ldg(G.curPN + 2 * (size_t)ci[k]);
        c1l[k] = __ldg(G.curPN + 2 * (size_t)ci[k] + 1);
      }
    }
    // gathers of pair 0 ride in the same cp.async group as Omega
#pragma unroll
    for (int k = 0; k < TK; k++) {
      riCur[k] = MODE == 0 ? z_index(keyNext.z[k], epoch) : keyNext.ri[k];
      zCur[k] = keyNext.z[k];
    }
    issue_gathers(shfl_ptr(myRefPN, 0), riCur, curOk, 0);
    cp_async_commit();
    if (1 < G.count) load_key(1, keyNext);
    // what the gates need from the current side (correspondencefinder.cpp:69, :87-93), prepared once per group
#pragma unroll
    for (int k = 0; k < TK; k++) {
      if (MODE == 0) {
        // a zero current normal rejects the pixel for every pair (the pixel still counts as "both indices valid")
        const float nx = c0l[k].y, ny = c0l[k].w, nz = c1l[k].y;
        if (dot3(nx, ny, nz, nx, ny, nz) == 0.0f) c1l[k].w = -1.0f;  // curvature >= 0
        else if (c1l[k].w < ac.flatCurvature) c1l[k].w = ac.flatCurvature;
      }
      S.c0[k * NT + lane] = c0l[k];
      S.c1[k * NT + lane] = c1l[k];
    }
  }
  unsigned short c16[TK];
#pragma unroll
  for (int k = 0; k < TK; k++) {
    c16[k] = 0;
    if (MODE == 1 && imgStats) {
      const float dc = z_depth(zc[k], curEpoch, FLT_MAX);
      c16[k] = dc < FLT_MAX ? (unsigned short)(int)fmul(1000.0f, dc) : 0;
    }
  }
  __syncwarp();  // S.T of every pair visible to every lane

  // ---- the pairs of the group ----
  for (int g = 0; g < G.count; g++) {
    const int st = g & 1;
    // pair g + 1: decode its keys (loaded one iteration ago), send its gathers into the other stage; pair g + 2: keys
    int riNext[TK];
    unsigned long long zNext[TK];
#pragma unroll
    for (int k = 0; k < TK; k++) {
      riNext[k] = -1;
      zNext[k] = kEmptyZ;
    }
    if (g + 1 < G.count) {
#pragma unroll
      for (int k = 0; k < TK; k++) {
        riNext[k] = MODE == 0 ? z_index(keyNext.z[k], epoch) : keyNext.ri[k];
        zNext[k] = keyNext.z[k];
      }
      issue_gathers(shfl_ptr(myRefPN, g + 1), riNext, curOk, st ^ 1);
      if (g + 2 < G.count) load_key(g + 2, keyNext);
    }
    cp_async_commit();         // (an empty group when there is no next pair)
    cp_async_wait_group<1>();  // everything but the group just committed has landed: Omega and the gathers of pair g

    // state->invT of pair g (column-major, broadcast reads from shared memory), the rotation entries duplicated into both
    // halves of a packed register
    const float4 t0 = S.T[g][0], t1 = S.T[g][1], t2 = S.T[g][2], t3 = S.T[g][3];
    const f32x2 T00 = pk(t0.x, t0.x), T01 = pk(t1.x, t1.x), T02 = pk(t2.x, t2.x);
    const f32x2 T10 = pk(t0.y, t0.y), T11 = pk(t1.y, t1.y), T12 = pk(t2.y, t2.y);
    const f32x2 T20 = pk(t0.z, t0.z), T21 = pk(t1.z, t1.z), T22 = pk(t2.z, t2.z);
    const float T03 = t3.x, T13 = t3.y, T23 = t3.z;
    const f32x2 ONE = pk(ac.one, ac.one);
    auto sum2 = [&](f32x2 a, f32x2 b) { return fma2(b, ONE, a); };  // a + b, exactly rounded, never contracted
    int *__restrict__ corrImage = B.corrImage + (size_t)(G.first + g) * (size_t)B.slotPixels;

    // a tile where no lane has a pixel of this pair contributes a row of zeros (decided before any sum is live)
    bool ok0[TK];
#pragma unroll
    for (int k = 0; k < TK; k++) ok0[k] = riCur[k] >= 0 && curOk[k];
    const bool tileAny = __any_sync(0xffffffffu, ok0[0] || ok0[1] || ok0[2]) || (MODE == 1 && imgStats);
    float tot = 0.0f;
    if (tileAny) {
      float midx = 0.0f, imgSum = 0.0f, imgNz = 0.0f, imgInl = 0.0f;
      if (MODE == 1 && imgStats) {
#pragma unroll
        for (int k = 0; k < TK; k++) {
          // DepthImage_convert_32FC1_to_16UC1 + mask + bitwise (abs diff & 255.0f) (pwn_matcher_base.cpp:167-190)
          const float dr = z_depth(zCur[k], epoch, FLT_MAX);
          const unsigned short r16 = dr < FLT_MAX ? (unsigned short)(int)fmul(1000.0f, dr) : 0;
          if (c16[k] > 0 && r16 > 0) {
            const float df = fabsf(fsub((float)c16[k], (float)r16));
            const float dm = __uint_as_float(__float_as_uint(df) & 0x437F0000u);
            imgNz += 1.0f;
            if (dm < imgThreshold) imgInl += 1.0f;
            imgSum += dm;
          }
        }
      }
      // ---- per pixel, STRAIGHT-LINE for every lane: transform, gates in the reference's order, Linearizer term weighted
      // by 1 (accepted) or 0.  No branch surrounds the sums, so they stay in place in their registers; a lane without a
      // pixel works on the zeros / stale finite values of its slots and its Omega is multiplied away. ----
      TermAcc acc;
      term_clear(acc);
      float nc = 0.0f;
#pragma unroll
      for (int k = 0; k < TK; k++) {
        // reference and current point + normal, interleaved: (px, nx, py, ny) (pz, nz, 1, curvature)
        const ulonglong2 r0 = *reinterpret_cast<const ulonglong2 *>(&stage[st].p0[k * NT + lane]);
        const ulonglong2 r1 = *reinterpret_cast<const ulonglong2 *>(&stage[st].p1[k * NT + lane]);
        const ulonglong2 q0 = *reinterpret_cast<const ulonglong2 *>(&S.c0[k * NT + lane]);
        const ulonglong2 q1 = *reinterpret_cast<const ulonglong2 *>(&S.c1[k * NT + lane]);
        const f32x2 Px = r0.x, Py = r0.y, Pz = r1.x, Cx = q0.x, Cy = q0.y, Cz = q1.x;
        // T (p, 1) in the low halves and T (n, 0) in the high halves, row by row in the order of xform_point /
        // xform_normal: ((m0 v0 + m1 v1) + m2 v2) [+ m3]; products and sums rounded separately, so each half is bit for
        // bit what the scalar functions return.  The sums are written b * 1 + a with a run-time 1: ptxas contracts
        // mul.rn.f32x2 followed by add.rn.f32x2 into one FFMA2 (unlike the scalar .rn forms), which rounds once.
        f32x2 Rx = sum2(sum2(mul2(T00, Px), mul2(T01, Py)), mul2(T02, Pz));
        f32x2 Ry = sum2(sum2(mul2(T10, Px), mul2(T11, Py)), mul2(T12, Pz));
        f32x2 Rz = sum2(sum2(mul2(T20, Px), mul2(T21, Py)), mul2(T22, Pz));
        Rx = pk(fadd(lo_of(Rx), T03), hi_of(Rx));
        Ry = pk(fadd(lo_of(Ry), T13), hi_of(Ry));
        Rz = pk(fadd(lo_of(Rz), T23), hi_of(Rz));
        const f32x2 E0 = sub2(Rx, Cx), E1 = sub2(Ry, Cy), E2 = sub2(Rz, Cz);  // (rp - cp, rn - cn)
        bool good = ok0[k];
        if (MODE == 0) {
          midx += ok0[k] ? 1.0f : 0.0f;
          const float rnx0 = hi_of(Px), rny0 = hi_of(Py), rnz0 = hi_of(Pz);
          const float cc = hi_of(q1.y);  // current curvature, already clamped; -1 = zero current normal
          // correspondencefinder.cpp:69 zero normals, :78 normal angle, :84 distance, :87-99 curvature ratio
          good = good && !(cc < 0.0f) && dot3(rnx0, rny0, rnz0, rnx0, rny0, rnz0) != 0.0f;
          good = good && !(dot3(hi_of(Cx), hi_of(Cy), hi_of(Cz), hi_of(Rx), hi_of(Ry), hi_of(Rz)) < ac.normalThreshold);
          const float dx = lo_of(E0), dy = lo_of(E1), dz = lo_of(E2);  // (rp - cp)^2 = (cp - rp)^2 bit for bit
          good = good && !(dot3(dx, dy, dz, dx, dy, dz) > ac.squaredThreshold);
          float rc = hi_of(r1.y);
          if (rc < ac.flatCurvature) rc = ac.flatCurvature;
          // (rc + 1e-5) / (cc + 1e-5) in double, rounded to float; identical operands give exactly 1.  A float32
          // pre-test decides unless the quotient lies within 1e-4 (relative) of a threshold.
          const float q = __fdividef(rc + 1e-5f, cc + 1e-5f);
          const float lo = ac.minRatio * (1.0f - 1e-4f), hi = ac.maxRatio * (1.0f + 1e-4f);
          const float loIn = ac.minRatio * (1.0f + 1e-4f), hiIn = ac.maxRatio * (1.0f - 1e-4f);
          const bool differ = rc != cc;
          good = good && !(differ && (q < lo || q > hi));
          if (good && differ && !(q > loIn && q < hiIn)) {  // rare: the exact quotient decides
            const float ratio = (float)(((double)rc + 1e-5) / ((double)cc + 1e-5));
            if (ratio < ac.minRatio || ratio > ac.maxRatio) good = false;
          }
        }
        if (MODE == 0 && writeCorr) {
          const int pix = base + k * NT + lane;
          if (pix < numPixels) corrImage[pix] = good ? riCur[k] : -1;
        }
        const float w = good ? 1.0f : 0.0f;
        nc += w;
        const ulonglong2 w0 = *reinterpret_cast<const ulonglong2 *>(&S.om[0][k * NT + lane]);
        const ulonglong2 w1 = *reinterpret_cast<const ulonglong2 *>(&S.om[1][k * NT + lane]);
        const ulonglong2 w2 = *reinterpret_cast<const ulonglong2 *>(&S.om[2][k * NT + lane]);
        term_add_e<ROBUST>(acc, w, Rx, Ry, Rz, E0, E1, E2, w0.x, w0.y, w1.x, w1.y, w2.x, w2.y, ac.maxChi2);
      }
      float v[kAccum];
      term_slots(acc, v);
      if (MODE == 0) {
        v[A_NCORR] = nc;
        v[A_MIDX] = midx;
        v[31] = 0.0f;
      } else {
        v[29] = imgSum;
        v[30] = imgNz;
        v[31] = imgInl;
      }
      tot = warp_transpose_reduce(v, lane);
    } else if (MODE == 0 && writeCorr) {
#pragma unroll
      for (int k = 0; k < TK; k++) {
        const int pix = base + k * NT + lane;
        if (pix < numPixels) corrImage[pix] = -1;
      }
    }
    B.partials[(size_t)(G.first + g) * (size_t)B.partialStride + (size_t)tileId * kAccum + lane] = tot;
#pragma unroll
    for (int k = 0; k < TK; k++) {
      riCur[k] = riNext[k];
      zCur[k] = zNext[k];
    }
  }
  cp_async_wait_group<0>();
}


// ---- per-pair kernel: one warp per (pair, tile); lone pairs and single alignments, whose groups are too small for the
// grouped kernel's prologue to pay ----
//   stage 1  every lane loads the z-buffer word / current index of its TK pixels, then issues the 4*TK gathers (float4
//            each) back to back together with the cp.async (LDGSTS) of the 48 bytes of Omega_P/Omega_N of the current
//            point into its own shared-memory slot -- two dependent round trips per tile; the Omega bytes are wasted when
//            a gate rejects the pixel -- transforms the reference point/normal, applies the gates in the reference's
//            order and writes the correspondence image when asked to.
//   stage 2  the lane that owns an accepted pixel accumulates its Linearizer term in place, with the packed term of the
//            grouped kernel operation for operation, so a (pair, tile) row has the same bits whichever kernel produced
//            it; pixel slots without any accepted lane are skipped warp-wide.
//   stage 3  transposing warp butterfly -> one partial row per tile.
// Dynamic shared memory: Omega_P / Omega_N of the tile, om[3][kTilePixels] float4.
template <int MODE>
__global__ void __launch_bounds__(kTileLanes, 18) k_corr_lin_tiled(const PairDesc *__restrict__ desc, int parity, int epoch,
                                                                   int writeCorr, AlignConsts ac, int numPixels, int imgStats,
                                                                   float imgThreshold, int pairFast, int curEpoch) {
  constexpr int TK = kTileSlots, NT = kTileLanes, TILE = kTilePixels;
  extern __shared__ __align__(16) float4 omSmem[][kTilePixels];

  // pair-fastest block order: the CTAs that are resident together work on the SAME tile of different pairs, so the
  // current-cloud data shared by the pairs of a chunk (index image, points, normals, Omega) is served by L1/L2
  const int pairId = pairFast ? blockIdx.x : blockIdx.y;
  const int tileId = pairFast ? blockIdx.y : blockIdx.x;
  const PairDesc &D = desc[pairId];
  const Affine T = affine_from(D.state->invT);
  const float4 *__restrict__ refPoints = D.refPoints;
  const float4 *__restrict__ refNormals = D.refNormals;
  const float4 *__restrict__ curPoints = D.curPoints;
  const float4 *__restrict__ curNormals = D.curNormals;
  const float4 *__restrict__ curOmega = D.curOmega;
  const int *__restrict__ curIndex = D.curIndex;
  int *__restrict__ corrImage = D.corrImage;
  const unsigned long long *__restrict__ zref = D.refZ[parity];
  const unsigned long long *__restrict__ zcur = D.curZ;

  const int lane = threadIdx.x & 31;
  const int base = tileId * TILE;
  float midx = 0.0f, imgSum = 0.0f, imgNz = 0.0f, imgInl = 0.0f;

  // ---- stage 1: loads ----
  int ri[TK], ci[TK];
  bool ok[TK];
#pragma unroll
  for (int k = 0; k < TK; k++) {
    const int pix = base + k * NT + threadIdx.x;
    ri[k] = -1;
    ci[k] = -1;
    if (pix < numPixels) {
      ci[k] = curIndex[pix];
      if (MODE == 0) {
        ri[k] = z_index(zref[pix], epoch);
      } else {
        ri[k] = corrImage[pix];
      }
    }
  }
  // MODE 1 + image statistics: the two z-buffer words are fetched with the indices (same round trip) and decoded
  // while the gathers are in flight
  unsigned long long zc[TK], zr[TK];
  if (MODE == 1 && imgStats) {
#pragma unroll
    for (int k = 0; k < TK; k++) {
      const int pix = base + k * NT + threadIdx.x;
      zc[k] = kEmptyZ;
      zr[k] = kEmptyZ;
      if (pix < numPixels) {
        zc[k] = zcur[pix];
        zr[k] = zref[pix];
      }
    }
  }
  float4 cn[TK], rn0[TK], cp[TK], rp0[TK];
#pragma unroll
  for (int k = 0; k < TK; k++) {
    ok[k] = ri[k] >= 0 && ci[k] >= 0;
    if (ok[k]) {
      const float4 *om = curOmega + 3 * (size_t)ci[k];
      cp_async16(&omSmem[0][k * NT + threadIdx.x], om);
      cp_async16(&omSmem[1][k * NT + threadIdx.x], om + 1);
      cp_async16(&omSmem[2][k * NT + threadIdx.x], om + 2);
      cn[k] = curNormals[ci[k]];
      rn0[k] = refNormals[ri[k]];
      cp[k] = curPoints[ci[k]];
      rp0[k] = refPoints[ri[k]];
    }
  }
  if (MODE == 1 && imgStats) {
#pragma unroll
    for (int k = 0; k < TK; k++) {
      const int pix = base + k * NT + threadIdx.x;
      if (pix < numPixels) {
        // DepthImage_convert_32FC1_to_16UC1 + mask + bitwise (abs diff & 255.0f) (pwn_matcher_base.cpp:167-190)
        const float dc = z_depth(zc[k], curEpoch, FLT_MAX);
        const float dr = z_depth(zr[k], epoch, FLT_MAX);
        unsigned short c16 = dc < FLT_MAX ? (unsigned short)(int)fmul(1000.0f, dc) : 0;
        unsigned short r16 = dr < FLT_MAX ? (unsigned short)(int)fmul(1000.0f, dr) : 0;
        if (c16 > 0 && r16 > 0) {
          float df = fabsf(fsub((float)c16, (float)r16));
          float dm = __uint_as_float(__float_as_uint(df) & 0x437F0000u);
          imgNz += 1.0f;
          if (dm < imgThreshold) imgInl += 1.0f;
          imgSum += dm;
        }
      }
    }
  }

  // ---- stage 1: transform + gates (results overwrite rp0 / rn0) ----
#pragma unroll
  for (int k = 0; k < TK; k++) {
    bool good = ok[k];
    if (good) {
      float rpx, rpy, rpz, rnx, rny, rnz;
      xform_point(T, rp0[k].x, rp0[k].y, rp0[k].z, rpx, rpy, rpz);
      xform_normal(T, rn0[k].x, rn0[k].y, rn0[k].z, rnx, rny, rnz);
      if (MODE == 0) {
        midx += 1.0f;
        // correspondencefinder.cpp:69 zero normals, :78 normal angle, :84 distance, :87-99 curvature ratio
        if (dot3(cn[k].x, cn[k].y, cn[k].z, cn[k].x, cn[k].y, cn[k].z) == 0.0f ||
            dot3(rn0[k].x, rn0[k].y, rn0[k].z, rn0[k].x, rn0[k].y, rn0[k].z) == 0.0f)
          good = false;
        if (good && dot3(cn[k].x, cn[k].y, cn[k].z, rnx, rny, rnz) < ac.normalThreshold) good = false;
        if (good) {
          float dx = fsub(cp[k].x, rpx), dy = fsub(cp[k].y, rpy), dz = fsub(cp[k].z, rpz);
          if (dot3(dx, dy, dz, dx, dy, dz) > ac.squaredThreshold) good = false;
        }
        if (good) {
          float rc = rn0[k].w, cc = cn[k].w;
          if (rc < ac.flatCurvature) rc = ac.flatCurvature;
          if (cc < ac.flatCurvature) cc = ac.flatCurvature;
          // (rc + 1e-5) / (cc + 1e-5) in double, rounded to float; identical operands give exactly 1
          // float32 pre-test: the float64 quotient is only needed within 1e-4 (relative) of a threshold
          if (rc != cc) {
            const float q = __fdividef(rc + 1e-5f, cc + 1e-5f);
            const float lo = ac.minRatio * (1.0f - 1e-4f), hi = ac.maxRatio * (1.0f + 1e-4f);
            const float loIn = ac.minRatio * (1.0f + 1e-4f), hiIn = ac.maxRatio * (1.0f - 1e-4f);
            if (q < lo || q > hi) {
              good = false;
            } else if (!(q > loIn && q < hiIn)) {
              const float ratio = (float)(((double)rc + 1e-5) / ((double)cc + 1e-5));
              if (ratio < ac.minRatio || ratio > ac.maxRatio) good = false;
            }
          }
        }
      }
      rp0[k].x = rpx; rp0[k].y = rpy; rp0[k].z = rpz;
      rn0[k].x = rnx; rn0[k].y = rny; rn0[k].z = rnz;
    }
    ok[k] = good;
    if (MODE == 0 && writeCorr) {
      const int pix = base + k * NT + threadIdx.x;
      if (pix < numPixels) corrImage[pix] = good ? ri[k] : -1;
    }
  }

  // ---- stage 2 ----
  cp_async_wait_all();
  TermAcc tacc;
  term_clear(tacc);
#pragma unroll
  for (int k = 0; k < TK; k++) {
    if (__any_sync(0xffffffffu, ok[k])) {
      if (ok[k]) {
        const ulonglong2 w0 = *reinterpret_cast<const ulonglong2 *>(&omSmem[0][k * NT + threadIdx.x]);
        const ulonglong2 w1 = *reinterpret_cast<const ulonglong2 *>(&omSmem[1][k * NT + threadIdx.x]);
        const ulonglong2 w2 = *reinterpret_cast<const ulonglong2 *>(&omSmem[2][k * NT + threadIdx.x]);
        const f32x2 Rx = pk(rp0[k].x, rn0[k].x), Ry = pk(rp0[k].y, rn0[k].y), Rz = pk(rp0[k].z, rn0[k].z);
        if (ac.robust)
          term_add<true, false>(tacc, 1.0f, Rx, Ry, Rz, cp[k], cn[k], w0.x, w0.y, w1.x, w1.y, w2.x, w2.y, ac.maxChi2);
        else
          term_add<false, false>(tacc, 1.0f, Rx, Ry, Rz, cp[k], cn[k], w0.x, w0.y, w1.x, w1.y, w2.x, w2.y, ac.maxChi2);
      }
    }
  }
  float acc[kAccum];
  term_slots(tacc, acc);
  acc[30] = 0.0f;
  acc[31] = 0.0f;
  if (MODE == 0) {
    acc[A_MIDX] = midx;
    float nc = 0.0f;
#pragma unroll
    for (int k = 0; k < TK; k++) nc += ok[k] ? 1.0f : 0.0f;
    acc[A_NCORR] = nc;
  } else {
    acc[29] = imgSum;
    acc[30] = imgNz;
    acc[31] = imgInl;
  }

  // ---- stage 3 ----
  D.partials[(size_t)tileId * kAccum + lane] = warp_transpose_reduce(acc, lane);
}

}  // namespace nicp

// nicp_internal.cuh -- internal structures shared by the kernels and the C-ABI layer.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <vector>

#include "../../include/nicp_b200.h"
#include "nicp_math.cuh"

namespace nicp {

void set_error(const char *fmt, ...);

#define NICP_CUDA(expr)                                                                          \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) {                                                                     \
      ::nicp::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return NICP_ERR_CUDA;                                                                      \
    }                                                                                            \
  } while (0)

#define NICP_CHECK_LAUNCH(ctx)                                                                   \
  do {                                                                                           \
    (ctx)->launches++;                                                                           \
    cudaError_t _e = cudaGetLastError();                                                         \
    if (_e != cudaSuccess) {                                                                     \
      ::nicp::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return NICP_ERR_CUDA;                                                                      \
    }                                                                                            \
  } while (0)

constexpr int kMaxCams = 8;       // NICP_MAX_CAMERAS
constexpr int kRowGroups = 16;    // first-level CTAs per pair of k_reduce_solve (align.cu); partials2 holds that many rows per slot
constexpr int kMaxGroup = 16;     // pairs per group of the grouped fused kernel (corr_lin.cuh: T of each in shared memory)
constexpr int kMaxPrepBatch = 8;  // frames per frame-preparation launch set (their scratch stays L2 resident)
constexpr int kAccum = 32;        // accumulator slots per partial (30 used)
constexpr int kIntegralCh = 10;   // n,x,y,z,xx,xy,xz,yy,yz,zz
constexpr unsigned long long kEmptyZ = 0xFFFFFFFFFFFFFFFFull;

// z-buffer word (one per pixel, filled with 64-bit atomicMin):
//   [63:60] epoch   [59:32] float bits of depth * 2^-110   [31:0] point index
// depth * 2^-110 is exact (power of two, no underflow above 1.5e-5 m) and its biased exponent stays below 32 for
// depth < 32 km, so the top four bits of the float are free.  Smaller word wins: nearest depth, then lowest index --
// the reference's sequential scatter with its strict `otherDistance > d` test (pinholepointprojector.cpp:52-64).
// The epoch makes NEWER projections smaller than anything an older iteration left in the same buffer, so the buffer
// is never cleared between iterations (the fused kernel used to spend 8 B/pixel/iteration on that): iteration `it`
// projects into buffer it&1 with epoch 15 - ((it>>1) & 15) and a word is valid only if it carries that epoch.
// A fresh buffer is all ones = epoch 15 with index -1.
constexpr int kEpochFresh = 15;
#if defined(__CUDACC__)
__device__ __forceinline__ unsigned long long z_encode(float d, int idx, int epoch) {
  unsigned int hi = __float_as_uint(__fmul_rn(d, 0x1p-110f)) | ((unsigned int)epoch << 28);
  return ((unsigned long long)hi << 32) | (unsigned int)idx;
}
// fire-and-forget 64-bit minimum into global memory (RED, no return path, no generic-address dispatch)
__device__ __forceinline__ void z_min(unsigned long long *p, unsigned long long key) {
  asm volatile("red.relaxed.gpu.global.min.u64 [%0], %1;" ::"l"(__cvta_generic_to_global(p)), "l"(key) : "memory");
}
__device__ __forceinline__ int z_index(unsigned long long v, int epoch) {
  return ((unsigned int)(v >> 60) == (unsigned int)epoch) ? (int)(unsigned int)(v & 0xFFFFFFFFull) : -1;
}
__device__ __forceinline__ float z_depth(unsigned long long v, int epoch, float emptyDepth) {
  if ((unsigned int)(v >> 60) != (unsigned int)epoch || (unsigned int)(v & 0xFFFFFFFFull) == 0xFFFFFFFFu) return emptyDepth;
  return __fmul_rn(__uint_as_float((unsigned int)(v >> 32) & 0x0FFFFFFFu), 0x1p110f);
}
#endif
inline int epoch_of_iteration(int it) { return kEpochFresh - ((it >> 1) & 15); }

// Device layout of a point's two information matrices: 3 float4 holding the upper triangles of Omega_P and Omega_N
// INTERLEAVED element by element,
//   (Pxx, Nxx, Pxy, Nxy)  (Pxz, Nxz, Pyy, Nyy)  (Pyz, Nyz, Pzz, Nzz),
// so that a 128-bit load leaves (P_ij, N_ij) in an aligned register pair: the Linearizer term of the fused kernel runs
// its point half and its normal half in the two lanes of the packed FP32 instructions (fma.rn.f32x2) without a move.
struct Omega3 {
  float4 o0, o1, o2;
};
__host__ __device__ inline Omega3 omega_pack(const float *P6, const float *N6) {
  Omega3 w;
  w.o0 = make_float4(P6[0], N6[0], P6[1], N6[1]);
  w.o1 = make_float4(P6[2], N6[2], P6[3], N6[3]);
  w.o2 = make_float4(P6[4], N6[4], P6[5], N6[5]);
  return w;
}
__host__ __device__ inline void omega_unpack(const float4 &o0, const float4 &o1, const float4 &o2, float *P6, float *N6) {
  P6[0] = o0.x; N6[0] = o0.y; P6[1] = o0.z; N6[1] = o0.w;
  P6[2] = o1.x; N6[2] = o1.y; P6[3] = o1.z; N6[3] = o1.w;
  P6[4] = o2.x; N6[4] = o2.y; P6[5] = o2.z; N6[5] = o2.w;
}

// accumulator slot layout of the fused correspondence+linearise reduction
enum {
  A_HTT = 0,   // 6: xx xy xz yy yz zz
  A_HTR = 6,   // 9: row-major (r*3+c)
  A_HRR = 15,  // 6: upper triangle
  A_BT = 21,   // 3
  A_BR = 24,   // 3
  A_ERR = 27,
  A_INL = 28,
  A_NCORR = 29,
  A_MIDX = 30   // MODE 0 only: pixels where both index images are valid
};

// per-pair pose / linear-system state, lives in device memory
struct PairState {
  float T[16];     // current estimate (reference <- current)
  float invT[16];  // working inverse used by the finder and the lineariser
  float KRt[kMaxCams][16];  // per camera: K_i * (T * referenceSensorOffset * offset_i)^-1, next reference projection
  float H[36];     // last assembled H (column-major 6x6, without damping)
  float b[6];
  float error;     // from the last LOOP linearisation (Aligner::error())
  int inliers;
  int ncorr;
  float statH[36]; // linearisation of _computeStatistics at the final T
  float statb[6];
  int img_nonzeros, img_inliers;
  float img_sum;
  float sumMidx;   // sum over outer iterations of pixels with both indices valid (roofline accounting)
  float sumMacc;   // sum over outer iterations of accepted correspondences
  int ticket;      // k_reduce_solve: how many of the kRowGroups first-level CTAs are done (0 between launches)
  int pad[3];      // sizeof % 16 == 0: T / invT of every slot can be fetched with 128-bit loads
};
static_assert(sizeof(PairState) % 16 == 0, "PairState slots must keep T / invT 16-byte aligned");

// pairs [first, first + count) of a chunk's descriptor array share their current cloud (corr_lin.cuh); count <= kMaxGroup.
// Everything the grouped kernel needs of the current side sits in the group record itself (one 48-byte load instead
// of a pointer chase through the descriptor); curSlot = the slot whose curZ / curIndex buffers the group reads.
struct PairGroup {
  int first, count, curSlot, pad;
  const float4 *curPoints;
  const float4 *curNormals;  // w = curvature
  const float4 *curOmega;    // Omega3 layout
  const float4 *curPN;       // nicp_cloud::pn of the current cloud
};
static_assert(sizeof(PairGroup) == 48, "PairGroup is fetched with three 128-bit loads");
// slot-indexed scratch of a chunk: buffer of slot i = base + i * stride (what fill_desc puts into the descriptors,
// passed by value so the grouped kernel computes the addresses instead of loading them)
struct SlotBases {
  const unsigned long long *refZ;  // reference z-buffers of the parity in use
  const unsigned long long *curZ;
  const int *curIndex;
  int *corrImage;
  float *partials;
  const PairState *state;
  long long slotPixels;            // stride of the image buffers
  long long partialStride;         // floats per slot in `partials`
};

// per-pair descriptor for the batched kernels (device memory, filled by the host per chunk)
struct PairDesc {
  const float4 *refPoints;
  const float *refPoints3;   // the same points packed at 12 bytes (projection stream), or null
  const float4 *refNormals;  // w = curvature
  const int *refN;
  const float4 *curPoints;
  const float4 *curNormals;  // w = curvature
  const float4 *curOmega;    // 3 float4 per point, Omega_P / Omega_N interleaved (Omega3 above)
  const float4 *refPN, *curPN;  // interleaved point + normal caches (nicp_cloud::pn), 2 float4 per point
  const int *curN;
  unsigned long long *refZ[2];  // double-buffered reference z-buffer (packed depth|index)
  unsigned long long *curZ;     // current z-buffer (shared by pairs with the same current cloud)
  int *curIndex;                // decoded current index image
  int *corrImage;               // accepted reference index per pixel or -1
  float *partials;              // [blocksPerPair][kAccum]
  float *partials2;             // [16][kAccum]: first-level sums of the partial rows
  PairState *state;
  float *trace;                 // may be null
  nicp_align_result *result;
  const void *priors;           // DevPrior[numPriors] (device) or null
  int numPriors;
  float guess[16];
};

// camera set of the projector: one pinhole (n == 1, offset = I, the PinholePointProjector case) or the
// children of a MultiPointProjector (multipointprojector.h:14-78).  For n > 1 the composite image is
// laid out as the Aligner executes it (pointprojector.cpp:17-40 over multipointprojector.cpp:157-205):
// row = pixel u, col = pixel v + colOff[i], first camera that sees the point wins, empty depth = 0.
struct CamSet {
  int n;
  int multi;                    // 0: plain pinhole image (row = v, col = u)
  int width[kMaxCams], height[kMaxCams], colOff[kMaxCams];
  float minD[kMaxCams], maxD[kMaxCams];
  float K[kMaxCams][9];
  float offset[kMaxCams][16];
};
// per-camera matrices for one projector pose (KRt for project, iKRt for unProject)
struct CamMats {
  Affine M[kMaxCams];
};
// geometry of a camera set as the kernels need it
struct CamGeom {
  int n, multi;
  int width[kMaxCams], height[kMaxCams], colOff[kMaxCams];
  float minD[kMaxCams], maxD[kMaxCams];
};
// everything frame prep needs for a MultiPointProjector (device memory)
struct PrepCams {
  CamGeom g;
  Affine iKRt[kMaxCams];          // child unProject matrices with the rig at identity
  float ivx[kMaxCams], ivy[kMaxCams];  // K_i * (worldRadius, worldRadius, 0), rows 0 and 1
};
// layout of the ctx->d_cams allocation
struct DeviceCams {
  CamSet set;
  CamMats curMats;
  PrepCams prep;
};

struct AlignConsts {
  float K[9];
  float refOffset[16];
  const CamSet *cams;           // device pointer (ctx->d_cams)
  int rows, cols;
  float minD, maxD;
  float squaredThreshold, normalThreshold, flatCurvature, minRatio, maxRatio;
  float maxChi2;
  int robust;
  float one;  // 1.0f as a run-time value: x * one + y is an exactly rounded sum that ptxas cannot contract with the product
              // that made x (it does contract mul.rn.f32x2 + add.rn.f32x2 into FFMA2; corr_lin.cuh)
};

}  // namespace nicp

struct nicp_cloud {
  nicp_context *ctx;
  int device;
  int capacity;
  float4 *points;
  float4 *normals;  // w = curvature
  float4 *omega;    // 3 per point (Omega3 layout)
  float *stats16;   // optional
  float *eigvals;
  int *statsN;
  int *d_n;         // device-side point count
  int n_host;       // host mirror (valid if n_known)
  bool n_known;
  bool has_stats;
  float *points3;   // cache: x,y,z packed at 12 bytes per point, the stream k_project reads (ensure_points3)
  bool points3_valid;  // every writer of `points` clears it
  float4 *pn;       // cache: point and normal of a point interleaved in one 32-byte sector, (px,nx,py,ny) (pz,nz,1,curvature):
                    // what the fused kernels gather (one sector per point instead of two, and a 128-bit load leaves
                    // (p_k, n_k) in an aligned register pair for the packed transform); ensure_pn
  bool pn_valid;    // cleared with points3_valid
  float *gauss;     // optional: Gaussian3f per point, NICP_GAUSS_FLOATS floats each (map_ops.cu)
  int *gflags;      // NICP_GAUSS_MOMENTS | NICP_GAUSS_INFO
  bool has_gauss;
};

struct nicp_context {
  int device;
  cudaStream_t stream;
  long long launches;
  int smCount;

  // frame-prep scratch
  size_t prepPixels;
  float *d_depth;
  uint16_t *d_raw;    // two staging images back to back: frame i+1 is uploaded while frame i is being converted
  size_t rawPixels;   // pixels per staging image
  cudaStream_t copyStream;
  cudaStream_t tailStream;      // a batch chunk's k_statistics + record copies, beside the next chunk's kernels
  cudaEvent_t evTail[2];        // chunk's last kernel on `stream` -> tailStream
  cudaEvent_t evRawCopied[2], evRawUsed[2];
  int rawToggle;
  float *d_integral;  // planar [10][rows][cols]
  int *d_interval;
  int *d_index;
  int lastRows, lastCols;
  // batched frame prep (nicp_raw_depth_to_cloud_batch): scratch of batchSlots frames, raw staging of 2 x batchSlots frames
  int batchSlots;
  size_t batchPixels, batchRawPixels;
  float *d_bDepth;      // [batchSlots][batchPixels]
  float *d_bIntegral;   // [batchSlots][10][batchPixels]
  uint16_t *d_bRaw;     // [2][batchSlots][batchRawPixels]
  cudaEvent_t evBRawCopied[2], evBRawUsed[2];
  int bRawToggle;
  // dynamic shared memory opted into on THIS context's device (cudaFuncAttributeMaxDynamicSharedMemorySize is per device)
  size_t rowsSmemCfg, colsSmemCfg;
  void *h_stage;      // pinned staging
  size_t stageBytes;

  // align scratch
  int slots;          // allocated slots
  size_t slotPixels;  // pixels per slot
  int blocksPerPair;            // lower bound of the partial-row allocation
  int groupSize;                // pairs per group of the grouped kernel (pairs of a group share their current cloud)
  int groupMinAvg;              // mean pairs per group from which a chunk takes the grouped kernel (else the per-pair one)
  int partialRows;              // rows of d_partials per slot
  unsigned long long *d_refZ;   // [slots][2][P]
  unsigned long long *d_curZ;   // [slots][P]
  int *d_curIndex;              // [slots][P]
  int *d_corrImage;             // [slots][P]
  float *d_partials;            // [slots][blocksPerPair][kAccum]
  float *d_partials2;           // [slots][16][kAccum]
  nicp::PairState *d_state;     // [slots]
  // descriptor staging is double buffered so that the host can fill chunk c+1 (and post-process chunk
  // c-1) while chunk c runs; d_desc / h_desc point at the set of the chunk being issued
  nicp::PairDesc *d_desc;       // [slots] + one int flag per slot
  nicp::PairDesc *h_desc;       // pinned
  unsigned char *d_descBase, *h_descBase;
  size_t descStride;
  cudaEvent_t evChunk[2];
  nicp::DeviceCams *d_cams;     // device copy of the camera set (+ derived matrices) of the call in flight
  nicp::CamSet h_cams;
  void *d_priors;               // device copy of the priors of the last nicp_align
  int priorCap;
  float *d_trace;               // [maxIter][61] for slot 0 (single align)
  int traceIters;
  nicp_align_result *d_results; // [resultCap]
  int resultCap;
  nicp_align_result *h_results; // pinned
  float *d_statHb;              // [resultCap][42]
  float *h_statHb;              // pinned

  // optional per-kernel timing (nicp_set_kernel_timing): CUDA events around the k_corr_lin<0>
  // and k_project launches of every chunk, accumulated after the final synchronisation
  bool timing;
  std::vector<cudaEvent_t> *evCorr;  // pairs (start, stop)
  std::vector<cudaEvent_t> *evProj;
  size_t evCorrUsed, evProjUsed;
  double msCorr, msProj;
  long long nCorr, nProj;

  // CUDA graph of the last single-pair nicp_align (36 kernels + memsets + copies replayed as one graph launch when
  // every baked-in value -- thresholds, K, offsets, iteration counts, image size, buffers -- is unchanged)
  int graphsEnabled;
  static constexpr int kGraphCache = 4;   // e.g. the three levels of a pyramid + one tracker configuration
  cudaGraphExec_t graphExec[kGraphCache];
  bool graphValid[kGraphCache];
  unsigned long long graphUse[kGraphCache], graphClock;
  long long graphLaunches[kGraphCache];   // kernels in the captured chunk (for nicp_launch_count on replays)
  unsigned char graphKey[kGraphCache][512];

  // epoch bookkeeping of the batch path (run_align_chunk): reference-projection iterations since the reference
  // z-buffers were last cleared as a whole, chunks since the current z-buffers were; -1 = must be cleared first
  long long zIter;
  int zCurGen;

  // local-map maintenance scratch (map_ops.cu), grow-only
  void *d_mapScratch;
  size_t mapScratchBytes;

  // last single-align bookkeeping
  int lastAlignRows, lastAlignCols, lastAlignIters, lastAlignParity, lastAlignEpoch;
  float lastAlignEmptyDepth;
  bool lastAlignValid;
};

namespace nicp {
// prior_offsets of a batch: n + 1 non-decreasing entries from 0 (or NULL: no priors)
inline bool prior_offsets_valid(int n, const nicp_prior *priors, const int *prior_offsets) {
  if (!prior_offsets) return true;
  if (prior_offsets[0] != 0) return false;
  for (int i = 0; i < n; i++)
    if (prior_offsets[i + 1] < prior_offsets[i]) return false;
  return !(prior_offsets[n] > 0 && !priors);
}

// frame_prep.cu
int launch_depth_convert(nicp_context *ctx, const uint16_t *d_raw, int rows, int cols, float scale, int step,
                         float maxCov, float *d_out);
int launch_frame_prep(nicp_context *ctx, const float *d_depth, const nicp_projector *proj, const nicp_stats_params *sp,
                      const float sensorOffset[16], int keepStats, nicp_cloud *cloud, int *d_index,
                      const CamSet *cams = nullptr);
int launch_raw_prep_batch(nicp_context *ctx, int n, const uint16_t *const *d_raw, int rawRows, int rawCols, float scale, int step,
                          float maxCov, const nicp_projector *proj, const nicp_stats_params *sp, const float sensorOffset[16],
                          int keepStats, nicp_cloud *const *clouds);
int launch_rig_raw_prep_batch(nicp_context *ctx, int n, const uint16_t *const *d_raw, const int *rawRows, const int *rawCols,
                              float scale, int step, float maxCov, const nicp_projector *proj, const CamSet &cams,
                              const nicp_stats_params *sp, const float sensorOffset[16], int keepStats, nicp_cloud *const *clouds);
int launch_stats_stage(nicp_context *ctx, const float4 *d_points, int n, const int *d_index, const int *d_interval, int rows,
                       int cols, const nicp_stats_params *sp, float *d_integral, float4 *d_normals, float *d_stats16,
                       float *d_eigvals, int *d_statsN, float *d_curvature);
int launch_information_stage(nicp_context *ctx, int n, const float4 *d_normals, const float *d_stats16, const float *d_eigvals,
                             const float *d_curvature, const nicp_stats_params *sp, float *d_omegaP6, float *d_omegaN6);
int launch_unproject(nicp_context *ctx, const float *d_depth, int rows, int cols, const float iKRt[16], float minD,
                     float maxD, nicp_cloud *cloud, int *d_index);
int launch_intervals(nicp_context *ctx, const float *d_depth, const nicp_projector *proj, float worldRadius, int *d_interval);
int launch_cloud_transform(nicp_context *ctx, nicp_cloud *cloud, const float T[16]);
int launch_cloud_append(nicp_context *ctx, nicp_cloud *dst, const nicp_cloud *src, const float T[16]);
// align.cu
int launch_project_single(nicp_context *ctx, const nicp_cloud *cloud, const float KRt[16], int rows, int cols,
                          float minD, float maxD, unsigned long long *d_z);
int launch_project_cams(nicp_context *ctx, const nicp_cloud *cloud, const CamSet &cams, const float T[16], int rows,
                        int cols, unsigned long long *d_z);
int ensure_points3(nicp_context *ctx, nicp_cloud *cloud);
int ensure_pn(nicp_context *ctx, nicp_cloud *cloud);
int launch_decode_z(nicp_context *ctx, const unsigned long long *d_z, int n, int *d_index, float *d_depth,
                    float emptyDepth = FLT_MAX, int epoch = kEpochFresh);
void cam_mats_KRt(const CamSet &cams, const float T[16], CamMats &out);
CamGeom geom_of(const CamSet &c);
int run_align_chunk(nicp_context *ctx, int nPairs, const AlignConsts &ac, const CamSet &cams, const float curOffset[16], int outerIters,
                    int innerIters, float imgThreshold, int nUniqueCur, const int *curSlotOfPair, bool wantTrace,
                    int resultOffset);
int run_correspond_linearize(nicp_context *ctx, const AlignConsts &ac, bool fromCorrImage, int slot);
int partial_rows_for(const nicp_context *ctx, size_t pixels);
int launch_statistics(nicp_context *ctx, cudaStream_t s, int base, int n);
const PairGroup *device_groups(const nicp_context *ctx);
PairGroup *host_groups(nicp_context *ctx);
// map_ops.cu
int cloud_ensure_gaussians(nicp_context *ctx, nicp_cloud *cloud);
int launch_gauss_transform(nicp_context *ctx, nicp_cloud *cloud, const int *d_first, int first, const int *d_count,
                           int maxCount, const float T[16]);
int launch_gauss_append(nicp_context *ctx, nicp_cloud *dst, const nicp_cloud *src, const float T[16]);
int run_compute_gaussians(nicp_context *ctx, nicp_cloud *cloud, const float *depth, const nicp_projector *proj,
                          float baseline, float alpha, const float sensorOffset[16]);
int run_merge(nicp_context *ctx, nicp_cloud *cloud, const nicp_projector *proj, const float transform[16],
              const nicp_merge_params *mp, int n, int *collapsedHost, int *newSize);
int run_voxelize(nicp_context *ctx, nicp_cloud *cloud, float resolution, int n, int *repHost, int *newSize);
}  // namespace nicp

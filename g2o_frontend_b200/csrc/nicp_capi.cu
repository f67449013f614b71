// nicp_capi.cu -- the extern "C" boundary declared in include/nicp_b200.h.
// Host-side orchestration only: scratch management, H2D/D2H, kernel sequencing, and the tiny
// dense statistics of Aligner::_computeStatistics (aligner.cpp:152-199).  No CPU fallback: every
// compute entry point launches CUDA kernels or fails.
#include <climits>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <map>
#include <vector>

#include "nicp_internal.cuh"
#include "nicp_stats_tail.cuh"

namespace nicp {

static thread_local char g_err[512] = "";
void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
}

static int env_int(const char *name, int def) {
  const char *v = getenv(name);
  if (!v || !*v) return def;
  int x = atoi(v);
  return x > 0 ? x : def;
}

template <typename T>
static int dev_alloc(T **p, size_t count) {
  void *q = nullptr;
  cudaError_t e = cudaMalloc(&q, count * sizeof(T));
  if (e != cudaSuccess) {
    set_error("cudaMalloc(%zu bytes) failed: %s", count * sizeof(T), cudaGetErrorString(e));
    return NICP_ERR_ALLOC;
  }
  *p = reinterpret_cast<T *>(q);
  return NICP_OK;
}
template <typename T>
static void dev_free(T *&p) {
  if (p) cudaFree(p);
  p = nullptr;
}

static int ensure_prep(nicp_context *ctx, size_t pixels) {
  if (pixels <= ctx->prepPixels) return NICP_OK;
  dev_free(ctx->d_depth);
  dev_free(ctx->d_integral);
  dev_free(ctx->d_interval);
  dev_free(ctx->d_index);
  ctx->prepPixels = 0;
  int rc;
  if ((rc = dev_alloc(&ctx->d_depth, pixels))) return rc;
  if ((rc = dev_alloc(&ctx->d_integral, pixels * kIntegralCh))) return rc;
  if ((rc = dev_alloc(&ctx->d_interval, pixels))) return rc;
  if ((rc = dev_alloc(&ctx->d_index, pixels))) return rc;
  ctx->prepPixels = pixels;
  return NICP_OK;
}
static int ensure_raw(nicp_context *ctx, size_t pixels) {
  if (pixels <= ctx->rawPixels) return NICP_OK;
  dev_free(ctx->d_raw);
  ctx->rawPixels = 0;
  int rc;
  if ((rc = dev_alloc(&ctx->d_raw, 2 * pixels))) return rc;
  ctx->rawPixels = pixels;
  return NICP_OK;
}

// The captured single-pair graphs bake in device AND pinned host addresses (descriptor staging, result / statistics
// buffers, trace, z-buffers): every reallocation of one of them drops all cached graphs.
static void invalidate_graphs(nicp_context *ctx) {
  for (int g = 0; g < nicp_context::kGraphCache; g++)
    if (ctx->graphValid[g]) {
      cudaGraphExecDestroy(ctx->graphExec[g]);
      ctx->graphValid[g] = false;
    }
}

// scratch of the batched frame preparation: `slots` frames of depth + integral image, raw staging for two sub-batches
static int ensure_batch_prep(nicp_context *ctx, int slots, size_t pixels, size_t rawPixels) {
  if (slots <= ctx->batchSlots && pixels <= ctx->batchPixels && rawPixels <= ctx->batchRawPixels) return NICP_OK;
  if (slots < ctx->batchSlots) slots = ctx->batchSlots;
  if (pixels < ctx->batchPixels) pixels = ctx->batchPixels;
  if (rawPixels < ctx->batchRawPixels) rawPixels = ctx->batchRawPixels;
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->copyStream));
  dev_free(ctx->d_bDepth);
  dev_free(ctx->d_bIntegral);
  dev_free(ctx->d_bRaw);
  ctx->batchSlots = 0;
  ctx->batchPixels = ctx->batchRawPixels = 0;
  int rc;
  if ((rc = dev_alloc(&ctx->d_bDepth, (size_t)slots * pixels))) return rc;
  if ((rc = dev_alloc(&ctx->d_bIntegral, (size_t)slots * pixels * kIntegralCh))) return rc;
  if ((rc = dev_alloc(&ctx->d_bRaw, 2 * (size_t)slots * rawPixels))) return rc;
  ctx->batchSlots = slots;
  ctx->batchPixels = pixels;
  ctx->batchRawPixels = rawPixels;
  return NICP_OK;
}

static void free_align(nicp_context *ctx) {
  invalidate_graphs(ctx);
  dev_free(ctx->d_refZ);
  dev_free(ctx->d_curZ);
  dev_free(ctx->d_curIndex);
  dev_free(ctx->d_corrImage);
  dev_free(ctx->d_partials);
  dev_free(ctx->d_partials2);
  dev_free(ctx->d_state);
  dev_free(ctx->d_descBase);
  if (ctx->h_descBase) cudaFreeHost(ctx->h_descBase);
  ctx->h_descBase = nullptr;
  ctx->d_desc = nullptr;
  ctx->h_desc = nullptr;
  ctx->slots = 0;
  ctx->slotPixels = 0;
}
static int ensure_align(nicp_context *ctx, int slots, size_t pixels) {
  if (slots <= ctx->slots && pixels <= ctx->slotPixels) return NICP_OK;
  // keep the larger old dimension only while that does not make the allocation bigger than both the old one and the request:
  // many slots of small images followed by a few of large ones (a rig chunk after pinhole batches) must not multiply out
  const size_t keepSlots = std::max<size_t>(slots, ctx->slots), keepPixels = std::max(pixels, ctx->slotPixels);
  if (keepSlots * keepPixels <= std::max((size_t)slots * pixels, (size_t)ctx->slots * ctx->slotPixels)) {
    slots = (int)keepSlots;
    pixels = keepPixels;
  }
  free_align(ctx);
  int rc;
  if ((rc = dev_alloc(&ctx->d_refZ, 2 * (size_t)slots * pixels))) return rc;
  if ((rc = dev_alloc(&ctx->d_curZ, (size_t)slots * pixels))) return rc;
  if ((rc = dev_alloc(&ctx->d_curIndex, (size_t)slots * pixels))) return rc;
  if ((rc = dev_alloc(&ctx->d_corrImage, (size_t)slots * pixels))) return rc;
  ctx->partialRows = partial_rows_for(ctx, pixels);
  if ((rc = dev_alloc(&ctx->d_partials, (size_t)slots * ctx->partialRows * kAccum))) return rc;
  if ((rc = dev_alloc(&ctx->d_partials2, (size_t)slots * kRowGroups * kAccum))) return rc;
  if ((rc = dev_alloc(&ctx->d_state, (size_t)slots))) return rc;
  NICP_CUDA(cudaMemset(ctx->d_state, 0, sizeof(PairState) * (size_t)slots));  // the reduction tickets start at 0
  // two sets of: descriptors, one int flag per slot, one pair group per slot
  // descriptors | ownership flags | projection order | (16-byte aligned) pair groups
  size_t descBytes = sizeof(PairDesc) * slots + 2 * sizeof(int) * slots + 16 + sizeof(PairGroup) * slots;
  descBytes = (descBytes + 255) & ~(size_t)255;
  void *p = nullptr;
  NICP_CUDA(cudaMalloc(&p, 2 * descBytes));
  ctx->d_descBase = reinterpret_cast<unsigned char *>(p);
  NICP_CUDA(cudaMallocHost(&p, 2 * descBytes));
  ctx->h_descBase = reinterpret_cast<unsigned char *>(p);
  ctx->descStride = descBytes;
  ctx->d_desc = reinterpret_cast<PairDesc *>(ctx->d_descBase);
  ctx->h_desc = reinterpret_cast<PairDesc *>(ctx->h_descBase);
  ctx->slots = slots;
  ctx->slotPixels = pixels;
  ctx->zIter = -1;  // new z-buffers: the batch path clears them before use
  ctx->zCurGen = -1;
  return NICP_OK;
}
static int ensure_results(nicp_context *ctx, int n) {
  if (n <= ctx->resultCap) return NICP_OK;
  invalidate_graphs(ctx);
  dev_free(ctx->d_results);
  dev_free(ctx->d_statHb);
  if (ctx->h_results) cudaFreeHost(ctx->h_results);
  if (ctx->h_statHb) cudaFreeHost(ctx->h_statHb);
  ctx->h_results = nullptr;
  ctx->h_statHb = nullptr;
  ctx->resultCap = 0;
  int rc;
  if ((rc = dev_alloc(&ctx->d_results, (size_t)n))) return rc;
  if ((rc = dev_alloc(&ctx->d_statHb, (size_t)n * 42))) return rc;
  void *p = nullptr;
  NICP_CUDA(cudaMallocHost(&p, sizeof(nicp_align_result) * n));
  ctx->h_results = reinterpret_cast<nicp_align_result *>(p);
  NICP_CUDA(cudaMallocHost(&p, sizeof(float) * 42 * n));
  ctx->h_statHb = reinterpret_cast<float *>(p);
  ctx->resultCap = n;
  return NICP_OK;
}
static int ensure_trace(nicp_context *ctx, int iters) {
  if (iters <= ctx->traceIters) return NICP_OK;
  invalidate_graphs(ctx);
  dev_free(ctx->d_trace);
  int rc;
  if ((rc = dev_alloc(&ctx->d_trace, (size_t)iters * 61))) return rc;
  ctx->traceIters = iters;
  return NICP_OK;
}

static int cloud_sync_n(nicp_context *ctx, const nicp_cloud *cloud) {
  nicp_cloud *c = const_cast<nicp_cloud *>(cloud);
  if (c->n_known) return NICP_OK;
  NICP_CUDA(cudaSetDevice(ctx->device));
  NICP_CUDA(cudaMemcpyAsync(&c->n_host, c->d_n, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  c->n_known = true;
  return NICP_OK;
}

static int ensure_stats(nicp_cloud *cloud) {
  if (cloud->stats16) return NICP_OK;
  int rc;
  if ((rc = dev_alloc(&cloud->stats16, (size_t)cloud->capacity * 16))) return rc;
  if ((rc = dev_alloc(&cloud->eigvals, (size_t)cloud->capacity * 3))) return rc;
  if ((rc = dev_alloc(&cloud->statsN, (size_t)cloud->capacity))) return rc;
  return NICP_OK;
}

static CamSet camset_pinhole(const nicp_projector *proj) {
  CamSet c;
  memset(&c, 0, sizeof c);
  c.n = 1;
  c.multi = 0;
  c.width[0] = proj->cols;
  c.height[0] = proj->rows;
  c.minD[0] = proj->min_distance;
  c.maxD[0] = proj->max_distance;
  for (int i = 0; i < 9; i++) c.K[0][i] = proj->K[i];
  mat4_identity(c.offset[0]);
  return c;
}
static int camset_multi(const nicp_multi_projector *mp, CamSet &c, int &rows, int &cols) {
  memset(&c, 0, sizeof c);
  if (!mp || mp->num_cameras < 1 || mp->num_cameras > kMaxCams) {
    set_error("multi projector needs 1..%d cameras", kMaxCams);
    return NICP_ERR_INVALID;
  }
  c.n = mp->num_cameras;
  c.multi = 1;
  rows = 0;
  cols = 0;
  for (int i = 0; i < c.n; i++) {
    c.width[i] = mp->camera[i].rows;
    c.height[i] = mp->camera[i].cols;
    if (c.width[i] <= 0 || c.height[i] <= 0) return NICP_ERR_INVALID;
    c.colOff[i] = cols;
    cols += c.height[i];
    if (c.width[i] > rows) rows = c.width[i];
    c.minD[i] = mp->camera[i].min_distance;
    c.maxD[i] = mp->camera[i].max_distance;
    for (int k = 0; k < 9; k++) c.K[i][k] = mp->camera[i].K[k];
    for (int k = 0; k < 16; k++) c.offset[i][k] = mp->sensor_offset[i][k];
    fix_last_row(c.offset[i]);
  }
  return NICP_OK;
}
static int upload_cams(nicp_context *ctx, const CamSet &c) {
  ctx->h_cams = c;
  NICP_CUDA(cudaMemcpyAsync(&ctx->d_cams->set, &ctx->h_cams, sizeof(CamSet), cudaMemcpyHostToDevice, ctx->stream));
  return NICP_OK;
}

static AlignConsts make_consts(const nicp_projector *proj, const nicp_align_params *ap, const float *refOffset) {
  AlignConsts ac;
  memset(&ac, 0, sizeof ac);
  for (int i = 0; i < 9; i++) ac.K[i] = proj->K[i];
  if (refOffset) {
    for (int i = 0; i < 16; i++) ac.refOffset[i] = refOffset[i];
    fix_last_row(ac.refOffset);
  } else {
    mat4_identity(ac.refOffset);
  }
  ac.cams = nullptr;
  ac.rows = proj->rows;
  ac.cols = proj->cols;
  ac.minD = proj->min_distance;
  ac.maxD = proj->max_distance;
  // correspondencefinder.h:63-70 (_squaredThreshold), correspondencefinder.cpp:28-29
  ac.squaredThreshold = ap->inlier_distance_threshold * ap->inlier_distance_threshold;
  ac.normalThreshold = ap->inlier_normal_angular_threshold;
  ac.flatCurvature = ap->flat_curvature_threshold;
  ac.minRatio = 1.0f / ap->inlier_curvature_ratio_threshold;
  ac.maxRatio = ap->inlier_curvature_ratio_threshold;
  ac.maxChi2 = ap->inlier_max_chi2;
  ac.robust = ap->robust_kernel;
  ac.one = 1.0f;
  return ac;
}

// pair groups of the chunk staged in ctx->h_desc (descriptors already filled): descriptors [0, m) are ordered so that
// pairs sharing a current cloud are adjacent (curSlotOf[i] = descriptor that owns pair i's current z-buffer); groups of at
// most ctx->groupSize (<= kMaxGroup) pairs.
static int stage_groups(nicp_context *ctx, int m, const int *curSlotOf) {
  PairGroup *g = host_groups(ctx);
  const int maxCount = ctx->groupSize < 1 ? 1 : (ctx->groupSize > kMaxGroup ? kMaxGroup : ctx->groupSize);
  int n = 0;
  for (int i = 0; i < m;) {
    int j = i + 1;
    while (j < m && j - i < maxCount && curSlotOf[j] == curSlotOf[i]) j++;
    memset(&g[n], 0, sizeof(PairGroup));
    g[n].first = i;
    g[n].count = j - i;
    g[n].curSlot = curSlotOf[i];
    g[n].curPoints = ctx->h_desc[i].curPoints;
    g[n].curNormals = ctx->h_desc[i].curNormals;
    g[n].curOmega = ctx->h_desc[i].curOmega;
    g[n].curPN = ctx->h_desc[i].curPN;
    n++;
    i = j;
  }
  return n;
}
// stage-level calls: one pair (descriptor 0 staged), one group
static int upload_single_group(nicp_context *ctx) {
  const int zero = 0;
  stage_groups(ctx, 1, &zero);
  NICP_CUDA(cudaMemcpyAsync(const_cast<PairGroup *>(device_groups(ctx)), host_groups(ctx), sizeof(PairGroup), cudaMemcpyHostToDevice,
                            ctx->stream));
  return NICP_OK;
}

static void fill_desc(nicp_context *ctx, int slot, int curSlot, const nicp_cloud *ref, const nicp_cloud *cur,
                      const float *guess, nicp_align_result *d_result, float *d_trace) {
  PairDesc &D = ctx->h_desc[slot];
  const size_t P = ctx->slotPixels;
  D.refPoints = ref->points;
  D.refPoints3 = nullptr;
  D.refNormals = ref->normals;
  D.refN = ref->d_n;
  D.curPoints = cur->points;
  D.curNormals = cur->normals;
  D.curOmega = cur->omega;
  D.refPN = ref->pn;  // (null until ensure_pn: the grouped kernel's chunks call it)
  D.curPN = cur->pn;
  D.curN = cur->d_n;
  D.refZ[0] = ctx->d_refZ + (size_t)slot * P;
  D.refZ[1] = ctx->d_refZ + ((size_t)ctx->slots + slot) * P;
  D.curZ = ctx->d_curZ + (size_t)curSlot * P;
  D.curIndex = ctx->d_curIndex + (size_t)curSlot * P;
  D.corrImage = ctx->d_corrImage + (size_t)slot * P;
  D.partials = ctx->d_partials + (size_t)slot * ctx->partialRows * kAccum;
  D.partials2 = ctx->d_partials2 + (size_t)slot * kRowGroups * kAccum;
  D.state = ctx->d_state + slot;
  D.trace = d_trace;
  D.result = d_result;
  D.priors = nullptr;
  D.numPriors = 0;
  if (guess) {
    for (int i = 0; i < 16; i++) D.guess[i] = guess[i];
  } else {
    mat4_identity(D.guess);
  }
}

// ---- Aligner::_computeStatistics tail (aligner.cpp:172-198, unscented.h:23-65): nicp_stats_tail.cuh, shared with the device ----
static void compute_statistics(const float *H_lin, const float *T, float *Omega, float *tr, float *rr) {
  compute_statistics_tail(H_lin, T, Omega, tr, rr);
}

// after a stream synchronisation: fold the recorded event pairs into the running totals
static void collect_timing(nicp_context *ctx) {
  if (!ctx->timing) return;
  for (size_t i = 0; i + 1 < ctx->evCorrUsed; i += 2) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, (*ctx->evCorr)[i], (*ctx->evCorr)[i + 1]) == cudaSuccess) {
      ctx->msCorr += ms;
      ctx->nCorr++;
    }
  }
  for (size_t i = 0; i + 1 < ctx->evProjUsed; i += 2) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, (*ctx->evProj)[i], (*ctx->evProj)[i + 1]) == cudaSuccess) {
      ctx->msProj += ms;
      ctx->nProj++;
    }
  }
  ctx->evCorrUsed = ctx->evProjUsed = 0;
}

static void select_desc_set(nicp_context *ctx, int set) {
  ctx->d_desc = reinterpret_cast<PairDesc *>(ctx->d_descBase + (size_t)set * ctx->descStride);
  ctx->h_desc = reinterpret_cast<PairDesc *>(ctx->h_descBase + (size_t)set * ctx->descStride);
}

// single alignment: the dense tail of _computeStatistics runs here (3.8 us, nothing extra on the GPU's critical path);
// batches get it from k_statistics on the device (same function, same bits) and the records arrive complete
static void finish_results(nicp_context *ctx, int base, int n, nicp_align_result *out, bool onDevice) {
  for (int i = base; i < base + n; i++) {
    nicp_align_result r = ctx->h_results[i];
    if (!onDevice) {
      const float *Hb = ctx->h_statHb + (size_t)i * 42;
      compute_statistics(Hb, r.T, r.omega, &r.translational_eigen_ratio, &r.rotational_eigen_ratio);
    }
    out[i] = r;
  }
}

}  // namespace nicp

using namespace nicp;

namespace {
struct DevBufs {  // temporaries of a stage-level call, freed on every exit path
  std::vector<void *> p;
  ~DevBufs() {
    for (void *q : p) cudaFree(q);
  }
  template <typename T>
  int alloc(T **out, size_t count) {
    void *q = nullptr;
    cudaError_t e = cudaMalloc(&q, (count ? count : 1) * sizeof(T));
    if (e != cudaSuccess) {
      set_error("cudaMalloc(%zu bytes) failed: %s", count * sizeof(T), cudaGetErrorString(e));
      return NICP_ERR_ALLOC;
    }
    p.push_back(q);
    *out = reinterpret_cast<T *>(q);
    return NICP_OK;
  }
};
}  // namespace

// =============================================================================================
extern "C" {

const char *nicp_last_error(void) { return g_err; }

int nicp_is_verification_build(void) {
#ifdef NICP_VERIFY_BUILD
  return 1;
#else
  return 0;
#endif
}

int nicp_create(int device, nicp_context **out) {
  if (!out) return NICP_ERR_INVALID;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0) {
    set_error("no CUDA device available (%s); this library has no CPU fallback",
              e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    return NICP_ERR_CUDA;
  }
  if (device < 0 || device >= count) {
    set_error("device %d out of range (0..%d)", device, count - 1);
    return NICP_ERR_INVALID;
  }
  NICP_CUDA(cudaSetDevice(device));
  nicp_context *ctx = new nicp_context();
  memset(ctx, 0, sizeof *ctx);
  ctx->device = device;
  NICP_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  NICP_CUDA(cudaStreamCreateWithFlags(&ctx->copyStream, cudaStreamNonBlocking));
  NICP_CUDA(cudaStreamCreateWithFlags(&ctx->tailStream, cudaStreamNonBlocking));
  NICP_CUDA(cudaEventCreateWithFlags(&ctx->evTail[0], cudaEventDisableTiming));
  NICP_CUDA(cudaEventCreateWithFlags(&ctx->evTail[1], cudaEventDisableTiming));
  for (int i = 0; i < 2; i++) {
    NICP_CUDA(cudaEventCreateWithFlags(&ctx->evRawCopied[i], cudaEventDisableTiming));
    NICP_CUDA(cudaEventCreateWithFlags(&ctx->evRawUsed[i], cudaEventDisableTiming));
    NICP_CUDA(cudaEventCreateWithFlags(&ctx->evBRawCopied[i], cudaEventDisableTiming));
    NICP_CUDA(cudaEventCreateWithFlags(&ctx->evBRawUsed[i], cudaEventDisableTiming));
  }
  cudaDeviceProp prop;
  NICP_CUDA(cudaGetDeviceProperties(&prop, device));
  ctx->smCount = prop.multiProcessorCount;
  ctx->blocksPerPair = 296;  // lower bound of the partial-row allocation
  ctx->groupSize = env_int("NICP_GROUP", 16);
  {
    const char *v = getenv("NICP_GROUP_MIN_AVG");  // 0 = always the grouped kernel (tests)
    ctx->groupMinAvg = (v && *v) ? atoi(v) : 3;
    if (ctx->groupMinAvg < 0) ctx->groupMinAvg = 0;
  }
  {
    void *p = nullptr;
    NICP_CUDA(cudaMalloc(&p, sizeof(DeviceCams)));
    ctx->d_cams = reinterpret_cast<DeviceCams *>(p);
  }
  NICP_CUDA(cudaEventCreateWithFlags(&ctx->evChunk[0], cudaEventDisableTiming));
  NICP_CUDA(cudaEventCreateWithFlags(&ctx->evChunk[1], cudaEventDisableTiming));
  {
    const char *g = getenv("NICP_GRAPH");
    ctx->graphsEnabled = (g && g[0] == '0') ? 0 : 1;
    ctx->zIter = -1;
    ctx->zCurGen = -1;
  }
  ctx->evCorr = new std::vector<cudaEvent_t>();
  ctx->evProj = new std::vector<cudaEvent_t>();
  *out = ctx;
  return NICP_OK;
}

void nicp_destroy(nicp_context *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  dev_free(ctx->d_depth);
  dev_free(ctx->d_raw);
  dev_free(ctx->d_integral);
  dev_free(ctx->d_interval);
  dev_free(ctx->d_index);
  free_align(ctx);
  dev_free(ctx->d_trace);
  if (ctx->d_priors) cudaFree(ctx->d_priors);
  if (ctx->d_cams) cudaFree(ctx->d_cams);
  if (ctx->d_mapScratch) cudaFree(ctx->d_mapScratch);
  dev_free(ctx->d_results);
  dev_free(ctx->d_statHb);
  if (ctx->h_results) cudaFreeHost(ctx->h_results);
  if (ctx->h_statHb) cudaFreeHost(ctx->h_statHb);
  invalidate_graphs(ctx);
  for (cudaEvent_t e : *ctx->evCorr) cudaEventDestroy(e);
  for (cudaEvent_t e : *ctx->evProj) cudaEventDestroy(e);
  delete ctx->evCorr;
  delete ctx->evProj;
  cudaEventDestroy(ctx->evChunk[0]);
  cudaEventDestroy(ctx->evChunk[1]);
  for (int i = 0; i < 2; i++) {
    cudaEventDestroy(ctx->evRawCopied[i]);
    cudaEventDestroy(ctx->evRawUsed[i]);
    cudaEventDestroy(ctx->evBRawCopied[i]);
    cudaEventDestroy(ctx->evBRawUsed[i]);
  }
  dev_free(ctx->d_bDepth);
  dev_free(ctx->d_bIntegral);
  dev_free(ctx->d_bRaw);
  cudaStreamDestroy(ctx->copyStream);
  if (ctx->tailStream) cudaStreamDestroy(ctx->tailStream);
  if (ctx->evTail[0]) cudaEventDestroy(ctx->evTail[0]);
  if (ctx->evTail[1]) cudaEventDestroy(ctx->evTail[1]);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

int nicp_synchronize(nicp_context *ctx) {
  if (!ctx) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  return NICP_OK;
}

long long nicp_launch_count(const nicp_context *ctx) { return ctx ? ctx->launches : 0; }

int nicp_set_kernel_timing(nicp_context *ctx, int enable) {
  if (!ctx) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  ctx->timing = enable != 0;
  ctx->msCorr = ctx->msProj = 0.0;
  ctx->nCorr = ctx->nProj = 0;
  ctx->evCorrUsed = ctx->evProjUsed = 0;
  return NICP_OK;
}

int nicp_get_kernel_timing(const nicp_context *ctx, double *corr_lin_ms, long long *corr_lin_launches, double *project_ms,
                           long long *project_launches) {
  if (!ctx) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  if (corr_lin_ms) *corr_lin_ms = ctx->msCorr;
  if (corr_lin_launches) *corr_lin_launches = ctx->nCorr;
  if (project_ms) *project_ms = ctx->msProj;
  if (project_launches) *project_launches = ctx->nProj;
  return NICP_OK;
}
void *nicp_stream(nicp_context *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

void nicp_update_matrices(const float K[9], const float T[16], float KRt[16], float iKRt[16]) {
  if (KRt) compute_KRt(K, T, KRt);
  if (iKRt) compute_iKRt(K, T, iKRt);
}
void nicp_v2t(const float v[6], float T[16]) { v2t(v, T); }
void nicp_t2v(const float T[16], float v[6]) { t2v(T, v); }

// ---- clouds ----------------------------------------------------------------------------------
int nicp_cloud_create(nicp_context *ctx, int capacity, nicp_cloud **out) {
  if (!ctx || !out || capacity <= 0) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  nicp_cloud *c = new nicp_cloud();
  memset(c, 0, sizeof *c);
  c->ctx = ctx;
  c->device = ctx->device;
  c->capacity = capacity;
  int rc;
  if ((rc = dev_alloc(&c->points, (size_t)capacity)) || (rc = dev_alloc(&c->normals, (size_t)capacity)) ||
      (rc = dev_alloc(&c->omega, (size_t)capacity * 3)) || (rc = dev_alloc(&c->d_n, 1))) {
    nicp_cloud_destroy(c);
    return rc;
  }
  NICP_CUDA(cudaMemsetAsync(c->d_n, 0, sizeof(int), ctx->stream));
  c->n_host = 0;
  c->n_known = true;
  *out = c;
  return NICP_OK;
}

void nicp_cloud_destroy(nicp_cloud *c) {
  if (!c) return;
  // the owning context may already be gone: cudaFree synchronises the device by itself
  cudaSetDevice(c->device);
  dev_free(c->points);
  dev_free(c->normals);
  dev_free(c->omega);
  dev_free(c->stats16);
  dev_free(c->eigvals);
  dev_free(c->statsN);
  dev_free(c->gauss);
  dev_free(c->gflags);
  dev_free(c->points3);
  dev_free(c->pn);
  dev_free(c->d_n);
  delete c;
}

int nicp_cloud_size(const nicp_cloud *c) {
  if (!c) return -1;
  if (cloud_sync_n(c->ctx, c) != NICP_OK) return -1;
  return c->n_host;
}

int nicp_cloud_upload(nicp_context *ctx, nicp_cloud *c, int n, const float *points4, const float *normals4,
                      const float *curvature, const float *omega_p6, const float *omega_n6) {
  if (!ctx || !c || n < 0 || !points4) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  if (n > c->capacity) {
    set_error("cloud upload of %d points exceeds capacity %d", n, c->capacity);
    return NICP_ERR_INVALID;
  }
  std::vector<float> nrm((size_t)n * 4, 0.0f), om((size_t)n * 12, 0.0f);
  for (int i = 0; i < n; i++) {
    if (normals4) { nrm[4 * i] = normals4[4 * i]; nrm[4 * i + 1] = normals4[4 * i + 1]; nrm[4 * i + 2] = normals4[4 * i + 2]; }
    nrm[4 * i + 3] = curvature ? curvature[i] : 0.0f;
    // device layout: the two upper triangles interleaved (Omega3, nicp_internal.cuh)
    if (omega_p6)
      for (int k = 0; k < 6; k++) om[12 * (size_t)i + 2 * k] = omega_p6[6 * (size_t)i + k];
    if (omega_n6)
      for (int k = 0; k < 6; k++) om[12 * (size_t)i + 2 * k + 1] = omega_n6[6 * (size_t)i + k];
  }
  c->points3_valid = false; c->pn_valid = false;
  NICP_CUDA(cudaMemcpyAsync(c->points, points4, sizeof(float) * 4 * n, cudaMemcpyHostToDevice, ctx->stream));
  NICP_CUDA(cudaMemcpyAsync(c->normals, nrm.data(), sizeof(float) * 4 * n, cudaMemcpyHostToDevice, ctx->stream));
  NICP_CUDA(cudaMemcpyAsync(c->omega, om.data(), sizeof(float) * 12 * n, cudaMemcpyHostToDevice, ctx->stream));
  NICP_CUDA(cudaMemcpyAsync(c->d_n, &n, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  c->n_host = n;
  c->n_known = true;
  c->has_stats = false;
  return NICP_OK;
}

int nicp_cloud_download(nicp_context *ctx, const nicp_cloud *c, float *points4, float *normals4, float *curvature,
                        float *omega_p6, float *omega_n6) {
  if (!ctx || !c) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  int rc = cloud_sync_n(ctx, c);
  if (rc) return rc;
  const int n = c->n_host;
  if (n == 0) return NICP_OK;
  if (points4) NICP_CUDA(cudaMemcpyAsync(points4, c->points, sizeof(float) * 4 * n, cudaMemcpyDeviceToHost, ctx->stream));
  std::vector<float> nrm, om;
  if (normals4 || curvature) {
    nrm.resize((size_t)n * 4);
    NICP_CUDA(cudaMemcpyAsync(nrm.data(), c->normals, sizeof(float) * 4 * n, cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (omega_p6 || omega_n6) {
    om.resize((size_t)n * 12);
    NICP_CUDA(cudaMemcpyAsync(om.data(), c->omega, sizeof(float) * 12 * n, cudaMemcpyDeviceToHost, ctx->stream));
  }
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < n; i++) {
    if (normals4) {
      normals4[4 * i] = nrm[4 * i]; normals4[4 * i + 1] = nrm[4 * i + 1]; normals4[4 * i + 2] = nrm[4 * i + 2];
      normals4[4 * i + 3] = 0.0f;
    }
    if (curvature) curvature[i] = nrm[4 * i + 3];
    if (omega_p6)
      for (int k = 0; k < 6; k++) omega_p6[6 * (size_t)i + k] = om[12 * (size_t)i + 2 * k];
    if (omega_n6)
      for (int k = 0; k < 6; k++) omega_n6[6 * (size_t)i + k] = om[12 * (size_t)i + 2 * k + 1];
  }
  return NICP_OK;
}

int nicp_cloud_download_stats(nicp_context *ctx, const nicp_cloud *c, float *stats16, float *eigenvalues3, int *n_points) {
  if (!ctx || !c) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  if (!c->has_stats) {
    set_error("cloud was built without keep_stats");
    return NICP_ERR_INVALID;
  }
  int rc = cloud_sync_n(ctx, c);
  if (rc) return rc;
  const int n = c->n_host;
  if (stats16) NICP_CUDA(cudaMemcpyAsync(stats16, c->stats16, sizeof(float) * 16 * n, cudaMemcpyDeviceToHost, ctx->stream));
  if (eigenvalues3) NICP_CUDA(cudaMemcpyAsync(eigenvalues3, c->eigvals, sizeof(float) * 3 * n, cudaMemcpyDeviceToHost, ctx->stream));
  if (n_points) NICP_CUDA(cudaMemcpyAsync(n_points, c->statsN, sizeof(int) * n, cudaMemcpyDeviceToHost, ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  return NICP_OK;
}

int nicp_cloud_transform(nicp_context *ctx, nicp_cloud *c, const float T[16]) {
  if (!ctx || !c || !T) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  return launch_cloud_transform(ctx, c, T);
}

int nicp_cloud_append(nicp_context *ctx, nicp_cloud *dst, const nicp_cloud *src, const float T[16]) {
  if (!ctx || !dst || !src || !T || dst == src) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = cloud_sync_n(ctx, dst))) return rc;
  if ((rc = cloud_sync_n(ctx, src))) return rc;
  if (dst->n_host + src->n_host > dst->capacity) {
    set_error("cloud append: %d + %d points exceed the destination capacity %d", dst->n_host, src->n_host, dst->capacity);
    return NICP_ERR_INVALID;
  }
  if ((rc = launch_cloud_append(ctx, dst, src, T))) return rc;
  dst->n_host += src->n_host;
  dst->n_known = true;
  return NICP_OK;
}

// ---- local-map maintenance (map_ops.cu) ------------------------------------------------------------
int nicp_cloud_compute_gaussians(nicp_context *ctx, nicp_cloud *c, const float *depth, const nicp_projector *proj,
                                 float baseline, float alpha, const float sensor_offset[16]) {
  if (!ctx || !c || !depth || !proj || !sensor_offset || proj->rows <= 0 || proj->cols <= 0) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  return run_compute_gaussians(ctx, c, depth, proj, baseline, alpha, sensor_offset);
}
int nicp_cloud_has_gaussians(const nicp_cloud *c) { return c && c->has_gauss ? 1 : 0; }
int nicp_cloud_download_gaussians(nicp_context *ctx, const nicp_cloud *c, float *gauss24, int *flags) {
  if (!ctx || !c) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  if (!c->has_gauss) {
    set_error("the cloud carries no gaussians (nicp_cloud_compute_gaussians / nicp_cloud_upload_gaussians first)");
    return NICP_ERR_INVALID;
  }
  int rc;
  if ((rc = cloud_sync_n(ctx, c))) return rc;
  const size_t n = (size_t)c->n_host;
  if (gauss24 && n) NICP_CUDA(cudaMemcpyAsync(gauss24, c->gauss, sizeof(float) * NICP_GAUSS_FLOATS * n, cudaMemcpyDeviceToHost, ctx->stream));
  if (flags && n) NICP_CUDA(cudaMemcpyAsync(flags, c->gflags, sizeof(int) * n, cudaMemcpyDeviceToHost, ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  return NICP_OK;
}
int nicp_cloud_upload_gaussians(nicp_context *ctx, nicp_cloud *c, const float *gauss24, const int *flags) {
  if (!ctx || !c || !gauss24 || !flags) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = cloud_sync_n(ctx, c))) return rc;
  if ((rc = cloud_ensure_gaussians(ctx, c))) return rc;
  const size_t n = (size_t)c->n_host;
  if (n) {
    NICP_CUDA(cudaMemcpyAsync(c->gauss, gauss24, sizeof(float) * NICP_GAUSS_FLOATS * n, cudaMemcpyHostToDevice, ctx->stream));
    NICP_CUDA(cudaMemcpyAsync(c->gflags, flags, sizeof(int) * n, cudaMemcpyHostToDevice, ctx->stream));
    NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  c->has_gauss = true;
  return NICP_OK;
}
int nicp_merge(nicp_context *ctx, nicp_cloud *c, const nicp_projector *proj, const float transform[16],
               const nicp_merge_params *params, int *collapsed, int *new_size) {
  if (!ctx || !c || !proj || !transform || !params || proj->rows <= 0 || proj->cols <= 0) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  if (!c->has_gauss) {
    set_error("nicp_merge: the cloud carries no gaussians (Merger::merge fuses cloud->gaussians())");
    return NICP_ERR_INVALID;
  }
  int rc;
  if ((rc = cloud_sync_n(ctx, c))) return rc;
  if (c->n_host == 0) {
    if (new_size) *new_size = 0;
    return NICP_OK;
  }
  return run_merge(ctx, c, proj, transform, params, c->n_host, collapsed, new_size);
}
int nicp_voxelize(nicp_context *ctx, nicp_cloud *c, float resolution, int *representatives, int *new_size) {
  if (!ctx || !c || !(resolution > 0.0f)) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = cloud_sync_n(ctx, c))) return rc;
  if (c->n_host == 0) {
    if (new_size) *new_size = 0;
    return NICP_OK;
  }
  return run_voxelize(ctx, c, resolution, c->n_host, representatives, new_size);
}

// ---- depth helpers ---------------------------------------------------------------------------
int nicp_depth_prepare(nicp_context *ctx, const uint16_t *raw, int rows, int cols, float depth_scale, int step,
                       float max_depth_cov, float *out) {
  if (!ctx || !raw || !out || rows <= 0 || cols <= 0) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  if (step < 1) step = 1;
  int rc;
  size_t px = (size_t)rows * cols;
  if ((rc = ensure_raw(ctx, px))) return rc;
  if ((rc = ensure_prep(ctx, px))) return rc;
  NICP_CUDA(cudaMemcpyAsync(ctx->d_raw, raw, px * sizeof(uint16_t), cudaMemcpyHostToDevice, ctx->stream));
  if ((rc = launch_depth_convert(ctx, ctx->d_raw, rows, cols, depth_scale, step, max_depth_cov, ctx->d_depth))) return rc;
  size_t opx = (size_t)(rows / step) * (cols / step);
  NICP_CUDA(cudaMemcpyAsync(out, ctx->d_depth, opx * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  return NICP_OK;
}

// ---- frame preparation -------------------------------------------------------------------------
int nicp_unproject(nicp_context *ctx, const float *depth, int rows, int cols, const float iKRt[16], float min_distance,
                   float max_distance, nicp_cloud *cloud, int *index) {
  if (!ctx || !depth || !iKRt || !cloud || rows <= 0 || cols <= 0) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  size_t px = (size_t)rows * cols;
  if ((size_t)cloud->capacity < px) {
    set_error("cloud capacity %d smaller than the image (%zu pixels)", cloud->capacity, px);
    return NICP_ERR_INVALID;
  }
  int rc;
  if ((rc = ensure_prep(ctx, px))) return rc;
  NICP_CUDA(cudaMemcpyAsync(ctx->d_depth, depth, px * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  if ((rc = launch_unproject(ctx, ctx->d_depth, rows, cols, iKRt, min_distance, max_distance, cloud, ctx->d_index))) return rc;
  // a points-only cloud: normals / information matrices are zero
  NICP_CUDA(cudaMemsetAsync(cloud->normals, 0, sizeof(float4) * px, ctx->stream));
  NICP_CUDA(cudaMemsetAsync(cloud->omega, 0, sizeof(float4) * 3 * px, ctx->stream));
  if (index) NICP_CUDA(cudaMemcpyAsync(index, ctx->d_index, px * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  return NICP_OK;
}

int nicp_project_intervals(nicp_context *ctx, const float *depth, const nicp_projector *proj, float world_radius,
                           int *interval) {
  if (!ctx || !depth || !proj || !interval || proj->rows <= 0 || proj->cols <= 0) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  size_t px = (size_t)proj->rows * proj->cols;
  int rc;
  if ((rc = ensure_prep(ctx, px))) return rc;
  NICP_CUDA(cudaMemcpyAsync(ctx->d_depth, depth, px * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  if ((rc = launch_intervals(ctx, ctx->d_depth, proj, world_radius, ctx->d_interval))) return rc;
  NICP_CUDA(cudaMemcpyAsync(interval, ctx->d_interval, px * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  return NICP_OK;
}

static int depth_to_cloud_device(nicp_context *ctx, const nicp_projector *proj, const nicp_stats_params *sp,
                                 const float sensor_offset[16], int keep_stats, nicp_cloud *cloud, int *index) {
  size_t px = (size_t)proj->rows * proj->cols;
  int rc;
  if (keep_stats && (rc = ensure_stats(cloud))) return rc;
  float eye[16];
  mat4_identity(eye);
  if ((rc = launch_frame_prep(ctx, ctx->d_depth, proj, sp, sensor_offset ? sensor_offset : eye, keep_stats, cloud,
                              ctx->d_index)))
    return rc;
  if (index) {
    NICP_CUDA(cudaMemcpyAsync(index, ctx->d_index, px * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  return NICP_OK;
}

int nicp_depth_to_cloud(nicp_context *ctx, const float *depth, const nicp_projector *proj, const nicp_stats_params *sp,
                        const float sensor_offset[16], int keep_stats, nicp_cloud *cloud, int *index) {
  if (!ctx || !depth || !proj || !sp || !cloud || proj->rows <= 0 || proj->cols <= 0) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  size_t px = (size_t)proj->rows * proj->cols;
  if ((size_t)cloud->capacity < px) {
    set_error("cloud capacity %d smaller than the image (%zu pixels)", cloud->capacity, px);
    return NICP_ERR_INVALID;
  }
  int rc;
  if ((rc = ensure_prep(ctx, px))) return rc;
  NICP_CUDA(cudaMemcpyAsync(ctx->d_depth, depth, px * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  return depth_to_cloud_device(ctx, proj, sp, sensor_offset, keep_stats, cloud, index);
}

int nicp_raw_depth_to_cloud(nicp_context *ctx, const uint16_t *raw, int raw_rows, int raw_cols, float depth_scale, int step,
                            float max_depth_cov, const nicp_projector *proj, const nicp_stats_params *sp,
                            const float sensor_offset[16], int keep_stats, nicp_cloud *cloud, int *index) {
  if (!ctx || !raw || !proj || !sp || !cloud || raw_rows <= 0 || raw_cols <= 0) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  if (step < 1) step = 1;
  if (proj->rows != raw_rows / step || proj->cols != raw_cols / step) {
    set_error("projector image size %dx%d does not match the scaled raw image %dx%d", proj->rows, proj->cols,
              raw_rows / step, raw_cols / step);
    return NICP_ERR_INVALID;
  }
  size_t rpx = (size_t)raw_rows * raw_cols, px = (size_t)proj->rows * proj->cols;
  if ((size_t)cloud->capacity < px) {
    set_error("cloud capacity %d smaller than the image (%zu pixels)", cloud->capacity, px);
    return NICP_ERR_INVALID;
  }
  int rc;
  if ((rc = ensure_raw(ctx, rpx))) return rc;
  if ((rc = ensure_prep(ctx, px))) return rc;
  // the upload runs on its own stream into one of two staging images, so the copy of this frame overlaps the
  // kernels of the previous one (from pinned host memory; a pageable source is staged by the driver as before)
  const int b = (ctx->rawToggle ^= 1);
  uint16_t *d_raw = ctx->d_raw + (size_t)b * ctx->rawPixels;
  NICP_CUDA(cudaStreamWaitEvent(ctx->copyStream, ctx->evRawUsed[b], 0));
  NICP_CUDA(cudaMemcpyAsync(d_raw, raw, rpx * sizeof(uint16_t), cudaMemcpyHostToDevice, ctx->copyStream));
  NICP_CUDA(cudaEventRecord(ctx->evRawCopied[b], ctx->copyStream));
  NICP_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->evRawCopied[b], 0));
  if ((rc = launch_depth_convert(ctx, d_raw, raw_rows, raw_cols, depth_scale, step, max_depth_cov, ctx->d_depth)))
    return rc;
  NICP_CUDA(cudaEventRecord(ctx->evRawUsed[b], ctx->stream));
  return depth_to_cloud_device(ctx, proj, sp, sensor_offset, keep_stats, cloud, index);
}

int nicp_raw_depth_to_cloud_batch(nicp_context *ctx, int n, const uint16_t *const *raws, int raw_rows, int raw_cols,
                                  float depth_scale, int step, float max_depth_cov, const nicp_projector *proj,
                                  const nicp_stats_params *sp, const float sensor_offset[16], int keep_stats,
                                  nicp_cloud *const *clouds) {
  if (!ctx || n < 0 || !proj || !sp || raw_rows <= 0 || raw_cols <= 0) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  if (n == 0) return NICP_OK;
  if (!raws || !clouds) return NICP_ERR_INVALID;
  if (step < 1) step = 1;
  if (proj->rows != raw_rows / step || proj->cols != raw_cols / step) {
    set_error("projector image size %dx%d does not match the scaled raw image %dx%d", proj->rows, proj->cols,
              raw_rows / step, raw_cols / step);
    return NICP_ERR_INVALID;
  }
  const size_t rpx = (size_t)raw_rows * raw_cols, px = (size_t)proj->rows * proj->cols;
  for (int i = 0; i < n; i++) {
    if (!raws[i] || !clouds[i]) {
      set_error("null frame or cloud at index %d", i);
      return NICP_ERR_INVALID;
    }
    if ((size_t)clouds[i]->capacity < px) {
      set_error("cloud %d: capacity %d smaller than the image (%zu pixels)", i, clouds[i]->capacity, px);
      return NICP_ERR_INVALID;
    }
    if (clouds[i]->device != ctx->device) {
      set_error("cloud %d lives on GPU %d, the context on GPU %d", i, clouds[i]->device, ctx->device);
      return NICP_ERR_INVALID;
    }
    for (int j = 0; j < i; j++)
      if (clouds[j] == clouds[i]) {
        set_error("cloud %d and cloud %d are the same object", j, i);
        return NICP_ERR_INVALID;
      }
  }
  int sub = env_int("NICP_PREP_BATCH", kMaxPrepBatch);
  if (sub > kMaxPrepBatch) sub = kMaxPrepBatch;
  if (sub > n) sub = n;
  int rc;
  if ((rc = ensure_batch_prep(ctx, sub, px, rpx))) return rc;
  float eye[16];
  mat4_identity(eye);
  for (int base = 0; base < n; base += sub) {
    const int m = n - base < sub ? n - base : sub;
    // raw frames of sub-batch k are uploaded on the copy stream into staging set k & 1 while sub-batch k - 1 computes
    const int b = (ctx->bRawToggle ^= 1);
    uint16_t *stage = ctx->d_bRaw + (size_t)b * ctx->batchSlots * ctx->batchRawPixels;
    const uint16_t *d_raw[kMaxPrepBatch];
    NICP_CUDA(cudaStreamWaitEvent(ctx->copyStream, ctx->evBRawUsed[b], 0));
    for (int f = 0; f < m; f++) {
      uint16_t *dst = stage + (size_t)f * ctx->batchRawPixels;
      NICP_CUDA(cudaMemcpyAsync(dst, raws[base + f], rpx * sizeof(uint16_t), cudaMemcpyHostToDevice, ctx->copyStream));
      d_raw[f] = dst;
    }
    NICP_CUDA(cudaEventRecord(ctx->evBRawCopied[b], ctx->copyStream));
    NICP_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->evBRawCopied[b], 0));
    for (int f = 0; f < m; f++)
      if (keep_stats && (rc = ensure_stats(clouds[base + f]))) return rc;
    if ((rc = launch_raw_prep_batch(ctx, m, d_raw, raw_rows, raw_cols, depth_scale, step, max_depth_cov, proj, sp,
                                    sensor_offset ? sensor_offset : eye, keep_stats, clouds + base)))
      return rc;
    NICP_CUDA(cudaEventRecord(ctx->evBRawUsed[b], ctx->stream));
  }
  ctx->lastRows = 0;  // the single-frame test hooks (integral / interval image) describe no frame of a batch
  return NICP_OK;
}

// frames per launch set of nicp_multi_raw_depth_to_cloud_batch for a composite image of px pixels: a set's scratch (depth +
// integral image, 44 B per pixel and frame) stays within that of a full pinhole set (kMaxPrepBatch frames of 640x480,
// 108 MB), at least one frame.  Frames are batched so that their row and column chains fill the GPU; a composite of
// 1280 x 3840 already brings 1280 row passes and 38 400 column chains on its own, so it runs one frame per set (216 MB)
// instead of 1.7 GB for eight.
static int rig_prep_frames(size_t px) {
  const size_t f = (size_t)kMaxPrepBatch * 640 * 480 / px;
  return f < 1 ? 1 : (f > (size_t)kMaxPrepBatch ? kMaxPrepBatch : (int)f);
}

int nicp_multi_raw_depth_to_cloud_batch(nicp_context *ctx, int n, const uint16_t *const *raws, const int *raw_rows,
                                        const int *raw_cols, float depth_scale, int step, float max_depth_cov,
                                        const nicp_multi_projector *mp, const nicp_stats_params *sp,
                                        const float sensor_offset[16], int keep_stats, nicp_cloud *const *clouds) {
  if (!ctx || n < 0 || !mp || !sp) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  if (n == 0) return NICP_OK;
  if (!raws || !clouds || !raw_rows || !raw_cols) return NICP_ERR_INVALID;
  if (step < 1) step = 1;
  CamSet cams;
  int rows, cols, rc;
  if ((rc = camset_multi(mp, cams, rows, cols))) return rc;
  const int nc = cams.n;
  size_t rpx = 0;
  for (int i = 0; i < nc; i++) {
    if (raw_rows[i] <= 0 || raw_cols[i] <= 0 || raw_rows[i] / step != cams.height[i] || raw_cols[i] / step != cams.width[i]) {
      set_error("camera %d: raw image %dx%d at step %d does not scale to the projector's %dx%d (rows x cols = height x width)",
                i, raw_rows[i], raw_cols[i], step, cams.height[i], cams.width[i]);
      return NICP_ERR_INVALID;
    }
    rpx += (size_t)raw_rows[i] * raw_cols[i];
  }
  const size_t px = (size_t)rows * cols;
  for (int f = 0; f < n; f++) {
    for (int i = 0; i < nc; i++)
      if (!raws[f * nc + i]) {
        set_error("null raw image of camera %d in frame %d", i, f);
        return NICP_ERR_INVALID;
      }
    if (!clouds[f]) {
      set_error("null cloud at index %d", f);
      return NICP_ERR_INVALID;
    }
    if ((size_t)clouds[f]->capacity < px) {
      set_error("cloud %d: capacity %d smaller than the composite image (%zu pixels)", f, clouds[f]->capacity, px);
      return NICP_ERR_INVALID;
    }
    if (clouds[f]->device != ctx->device) {
      set_error("cloud %d lives on GPU %d, the context on GPU %d", f, clouds[f]->device, ctx->device);
      return NICP_ERR_INVALID;
    }
    for (int j = 0; j < f; j++)
      if (clouds[j] == clouds[f]) {
        set_error("cloud %d and cloud %d are the same object", j, f);
        return NICP_ERR_INVALID;
      }
  }
  int sub = env_int("NICP_PREP_BATCH", kMaxPrepBatch);
  if (sub > rig_prep_frames(px)) sub = rig_prep_frames(px);
  if (sub < 1) sub = 1;
  if (sub > n) sub = n;
  if ((rc = ensure_batch_prep(ctx, sub, px, rpx))) return rc;
  float eye[16];
  mat4_identity(eye);
  for (int base = 0; base < n; base += sub) {
    const int m = n - base < sub ? n - base : sub;
    // as in nicp_raw_depth_to_cloud_batch: sub-batch k is uploaded into staging set k & 1 while sub-batch k - 1 computes;
    // the cameras of a frame sit back to back in its staging slot
    const int b = (ctx->bRawToggle ^= 1);
    uint16_t *stage = ctx->d_bRaw + (size_t)b * ctx->batchSlots * ctx->batchRawPixels;
    const uint16_t *d_raw[kMaxPrepBatch * kMaxCams];
    NICP_CUDA(cudaStreamWaitEvent(ctx->copyStream, ctx->evBRawUsed[b], 0));
    for (int f = 0; f < m; f++) {
      uint16_t *dst = stage + (size_t)f * ctx->batchRawPixels;
      for (int i = 0; i < nc; i++) {
        const size_t cpx = (size_t)raw_rows[i] * raw_cols[i];
        NICP_CUDA(cudaMemcpyAsync(dst, raws[(size_t)(base + f) * nc + i], cpx * sizeof(uint16_t), cudaMemcpyHostToDevice,
                                  ctx->copyStream));
        d_raw[f * nc + i] = dst;
        dst += cpx;
      }
    }
    NICP_CUDA(cudaEventRecord(ctx->evBRawCopied[b], ctx->copyStream));
    NICP_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->evBRawCopied[b], 0));
    for (int f = 0; f < m; f++)
      if (keep_stats && (rc = ensure_stats(clouds[base + f]))) return rc;
    nicp_projector proj = mp->camera[0];
    proj.rows = rows;
    proj.cols = cols;
    if ((rc = launch_rig_raw_prep_batch(ctx, m, d_raw, raw_rows, raw_cols, depth_scale, step, max_depth_cov, &proj, cams, sp,
                                        sensor_offset ? sensor_offset : eye, keep_stats, clouds + base)))
      return rc;
    NICP_CUDA(cudaEventRecord(ctx->evBRawUsed[b], ctx->stream));
  }
  ctx->lastRows = 0;
  return NICP_OK;
}

// ---- stage-level statistics / information matrices (host buffers in, host buffers out) -----------------------------
int nicp_stats_compute(nicp_context *ctx, const float *points4, int n, const int *index_image, const int *interval_image,
                       int rows, int cols, const nicp_stats_params *sp, float *normals4, float *stats16, float *eigenvalues3,
                       int *n_points, float *curvature) {
  if (!ctx || !points4 || n < 0 || !index_image || !interval_image || rows <= 0 || cols <= 0 || !sp) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  const size_t px = (size_t)rows * cols;
  DevBufs bufs;
  float4 *d_points, *d_normals;
  int *d_index, *d_interval, *d_cnt;
  float *d_integral, *d_stats, *d_eig, *d_curv;
  int rc;
  if ((rc = bufs.alloc(&d_points, (size_t)n)) || (rc = bufs.alloc(&d_normals, (size_t)n)) || (rc = bufs.alloc(&d_index, px)) ||
      (rc = bufs.alloc(&d_interval, px)) || (rc = bufs.alloc(&d_cnt, (size_t)n)) || (rc = bufs.alloc(&d_integral, px * kIntegralCh)) ||
      (rc = bufs.alloc(&d_stats, (size_t)n * 16)) || (rc = bufs.alloc(&d_eig, (size_t)n * 3)) || (rc = bufs.alloc(&d_curv, (size_t)n)))
    return rc;
  cudaStream_t st = ctx->stream;
  if (n) NICP_CUDA(cudaMemcpyAsync(d_points, points4, sizeof(float4) * n, cudaMemcpyHostToDevice, st));
  NICP_CUDA(cudaMemcpyAsync(d_index, index_image, sizeof(int) * px, cudaMemcpyHostToDevice, st));
  NICP_CUDA(cudaMemcpyAsync(d_interval, interval_image, sizeof(int) * px, cudaMemcpyHostToDevice, st));
  if ((rc = launch_stats_stage(ctx, d_points, n, d_index, d_interval, rows, cols, sp, d_integral, d_normals, d_stats, d_eig, d_cnt,
                               d_curv)))
    return rc;
  if (n) {
    if (normals4) NICP_CUDA(cudaMemcpyAsync(normals4, d_normals, sizeof(float4) * n, cudaMemcpyDeviceToHost, st));
    if (stats16) NICP_CUDA(cudaMemcpyAsync(stats16, d_stats, sizeof(float) * 16 * n, cudaMemcpyDeviceToHost, st));
    if (eigenvalues3) NICP_CUDA(cudaMemcpyAsync(eigenvalues3, d_eig, sizeof(float) * 3 * n, cudaMemcpyDeviceToHost, st));
    if (n_points) NICP_CUDA(cudaMemcpyAsync(n_points, d_cnt, sizeof(int) * n, cudaMemcpyDeviceToHost, st));
    if (curvature) NICP_CUDA(cudaMemcpyAsync(curvature, d_curv, sizeof(float) * n, cudaMemcpyDeviceToHost, st));
  }
  NICP_CUDA(cudaStreamSynchronize(st));
  return NICP_OK;
}

int nicp_information_compute(nicp_context *ctx, int n, const float *normals4, const float *stats16, const float *eigenvalues3,
                             const float *curvature, const nicp_stats_params *sp, float *omega_p6, float *omega_n6) {
  if (!ctx || n < 0 || !sp || (n > 0 && (!normals4 || !stats16 || !eigenvalues3 || !curvature))) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  if (n == 0) return NICP_OK;
  DevBufs bufs;
  float4 *d_normals;
  float *d_stats, *d_eig, *d_curv, *d_op = nullptr, *d_on = nullptr;
  int rc;
  if ((rc = bufs.alloc(&d_normals, (size_t)n)) || (rc = bufs.alloc(&d_stats, (size_t)n * 16)) || (rc = bufs.alloc(&d_eig, (size_t)n * 3)) ||
      (rc = bufs.alloc(&d_curv, (size_t)n)))
    return rc;
  if (omega_p6 && (rc = bufs.alloc(&d_op, (size_t)n * 6))) return rc;
  if (omega_n6 && (rc = bufs.alloc(&d_on, (size_t)n * 6))) return rc;
  cudaStream_t st = ctx->stream;
  NICP_CUDA(cudaMemcpyAsync(d_normals, normals4, sizeof(float4) * n, cudaMemcpyHostToDevice, st));
  NICP_CUDA(cudaMemcpyAsync(d_stats, stats16, sizeof(float) * 16 * n, cudaMemcpyHostToDevice, st));
  NICP_CUDA(cudaMemcpyAsync(d_eig, eigenvalues3, sizeof(float) * 3 * n, cudaMemcpyHostToDevice, st));
  NICP_CUDA(cudaMemcpyAsync(d_curv, curvature, sizeof(float) * n, cudaMemcpyHostToDevice, st));
  if ((rc = launch_information_stage(ctx, n, d_normals, d_stats, d_eig, d_curv, sp, d_op, d_on))) return rc;
  if (omega_p6) NICP_CUDA(cudaMemcpyAsync(omega_p6, d_op, sizeof(float) * 6 * n, cudaMemcpyDeviceToHost, st));
  if (omega_n6) NICP_CUDA(cudaMemcpyAsync(omega_n6, d_on, sizeof(float) * 6 * n, cudaMemcpyDeviceToHost, st));
  NICP_CUDA(cudaStreamSynchronize(st));
  return NICP_OK;
}

int nicp_last_integral_image(nicp_context *ctx, float *integral10) {
  if (!ctx || !integral10 || ctx->lastRows <= 0) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  size_t px = (size_t)ctx->lastRows * ctx->lastCols;
  std::vector<float> planar(px * kIntegralCh);
  NICP_CUDA(cudaMemcpyAsync(planar.data(), ctx->d_integral, planar.size() * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  for (size_t p = 0; p < px; p++)
    for (int k = 0; k < kIntegralCh; k++) integral10[p * kIntegralCh + k] = planar[k * px + p];
  return NICP_OK;
}

int nicp_last_interval_image(nicp_context *ctx, int *interval) {
  if (!ctx || !interval || ctx->lastRows <= 0) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  size_t px = (size_t)ctx->lastRows * ctx->lastCols;
  NICP_CUDA(cudaMemcpyAsync(interval, ctx->d_interval, px * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  return NICP_OK;
}

// ---- projection --------------------------------------------------------------------------------
int nicp_project(nicp_context *ctx, const nicp_cloud *cloud, const float KRt[16], int rows, int cols, float min_distance,
                 float max_distance, int *index, float *depth) {
  if (!ctx || !cloud || !KRt || rows <= 0 || cols <= 0) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  size_t px = (size_t)rows * cols;
  int rc;
  if ((rc = ensure_align(ctx, 1, px))) return rc;
  if ((rc = ensure_prep(ctx, px))) return rc;
  unsigned long long *z = ctx->d_curZ;
  if ((rc = launch_project_single(ctx, cloud, KRt, rows, cols, min_distance, max_distance, z))) return rc;
  if ((rc = launch_decode_z(ctx, z, (int)px, ctx->d_index, ctx->d_depth))) return rc;
  if (index) NICP_CUDA(cudaMemcpyAsync(index, ctx->d_index, px * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  if (depth) NICP_CUDA(cudaMemcpyAsync(depth, ctx->d_depth, px * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  ctx->lastAlignValid = false;
  return NICP_OK;
}

// ---- stage-level correspondence + linearisation ------------------------------------------------------
static int fetch_stage_result(nicp_context *ctx, float H[36], float b[6], float *error, int *inliers, int *ncorr) {
  PairState st;
  NICP_CUDA(cudaMemcpyAsync(&st, ctx->d_state, sizeof st, cudaMemcpyDeviceToHost, ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  if (H) memcpy(H, st.H, sizeof st.H);
  if (b) memcpy(b, st.b, sizeof st.b);
  if (error) *error = st.error;
  if (inliers) *inliers = st.inliers;
  if (ncorr) *ncorr = st.ncorr;
  return NICP_OK;
}

static int stage_set_T(nicp_context *ctx, const float T[16]) {
  float invT[16];
  for (int i = 0; i < 16; i++) invT[i] = T[i];
  fix_last_row(invT);
  NICP_CUDA(cudaMemcpyAsync(reinterpret_cast<char *>(ctx->d_state) + offsetof(PairState, invT), invT, sizeof invT,
                            cudaMemcpyHostToDevice, ctx->stream));
  return NICP_OK;
}

int nicp_correspond_linearize(nicp_context *ctx, const nicp_cloud *reference, const nicp_cloud *current,
                              const int *reference_index, const int *current_index, int rows, int cols, const float T[16],
                              const nicp_align_params *ap, float H[36], float b[6], float *error, int *inliers,
                              int *num_correspondences, int *corr_image) {
  if (!ctx || !reference || !current || !reference_index || !current_index || !T || !ap || rows <= 0 || cols <= 0)
    return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  size_t px = (size_t)rows * cols;
  int rc;
  if ((rc = ensure_align(ctx, 1, px))) return rc;
  nicp_projector proj;
  memset(&proj, 0, sizeof proj);
  proj.rows = rows;
  proj.cols = cols;
  AlignConsts ac = make_consts(&proj, ap, nullptr);
  fill_desc(ctx, 0, 0, reference, current, nullptr, nullptr, nullptr);
  std::vector<unsigned long long> z(px);
  for (size_t i = 0; i < px; i++) z[i] = reference_index[i] < 0 ? kEmptyZ : ((unsigned long long)kEpochFresh << 60) | (unsigned int)reference_index[i];
  NICP_CUDA(cudaMemcpyAsync(ctx->d_desc, ctx->h_desc, sizeof(PairDesc), cudaMemcpyHostToDevice, ctx->stream));
  NICP_CUDA(cudaMemcpyAsync(ctx->h_desc[0].refZ[0], z.data(), px * sizeof(unsigned long long), cudaMemcpyHostToDevice, ctx->stream));
  NICP_CUDA(cudaMemcpyAsync(ctx->h_desc[0].curIndex, current_index, px * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  if ((rc = stage_set_T(ctx, T))) return rc;
  if ((rc = upload_single_group(ctx))) return rc;
  ctx->zIter = ctx->zCurGen = -1;  // slot 0 was staged by hand
  if ((rc = run_correspond_linearize(ctx, ac, false, (int)px))) return rc;
  if (corr_image)
    NICP_CUDA(cudaMemcpyAsync(corr_image, ctx->h_desc[0].corrImage, px * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  ctx->lastAlignValid = false;
  return fetch_stage_result(ctx, H, b, error, inliers, num_correspondences);
}

int nicp_linearize(nicp_context *ctx, const nicp_cloud *reference, const nicp_cloud *current, const int *correspondences,
                   int n, const float T[16], const nicp_align_params *ap, float H[36], float b[6], float *error,
                   int *inliers) {
  if (!ctx || !reference || !current || (!correspondences && n > 0) || n < 0 || !T || !ap) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  size_t px = n > 0 ? (size_t)n : 1;
  int rc;
  if ((rc = ensure_align(ctx, 1, px))) return rc;
  nicp_projector proj;
  memset(&proj, 0, sizeof proj);
  proj.rows = 1;
  proj.cols = (int)px;
  AlignConsts ac = make_consts(&proj, ap, nullptr);
  fill_desc(ctx, 0, 0, reference, current, nullptr, nullptr, nullptr);
  std::vector<int> ri(px, -1), ci(px, -1);
  for (int i = 0; i < n; i++) {
    ri[i] = correspondences[2 * i];
    ci[i] = correspondences[2 * i + 1];
  }
  NICP_CUDA(cudaMemcpyAsync(ctx->d_desc, ctx->h_desc, sizeof(PairDesc), cudaMemcpyHostToDevice, ctx->stream));
  NICP_CUDA(cudaMemcpyAsync(ctx->h_desc[0].corrImage, ri.data(), px * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  NICP_CUDA(cudaMemcpyAsync(ctx->h_desc[0].curIndex, ci.data(), px * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  if ((rc = stage_set_T(ctx, T))) return rc;
  if ((rc = upload_single_group(ctx))) return rc;
  ctx->zIter = ctx->zCurGen = -1;
  if ((rc = run_correspond_linearize(ctx, ac, true, (int)px))) return rc;
  ctx->lastAlignValid = false;
  return fetch_stage_result(ctx, H, b, error, inliers, nullptr);
}

// ---- alignment -----------------------------------------------------------------------------------
// host mirror of align.cu's DevPrior
struct HostPrior {
  int kind;
  float mean[16];
  float refInv[16];
  float info[36];
};

// everything a captured single-pair graph has baked in
struct GraphKey {
  AlignConsts ac;
  float co[16];
  int outer, inner, numPriors, slots, partialRows;
  float imgThr;
  size_t slotPixels;
  const void *desc, *results, *statHb, *trace, *priors, *refZ;
};
static_assert(sizeof(GraphKey) <= 512, "graph key fits the context buffer");

static int align_common(nicp_context *ctx, int n, const nicp_cloud *const *refs, const nicp_cloud *const *curs,
                        const nicp_projector *proj, const nicp_align_params *ap, const float *refOffset,
                        const float *curOffset, const float *guesses, float imgThr, nicp_align_result *results,
                        bool single, const nicp_prior *priors = nullptr, int numPriors = 0, const CamSet *multiCams = nullptr,
                        const int *priorOffsets = nullptr, int slotCap = INT_MAX) {
  // priorOffsets (batch): pair i owns priors[priorOffsets[i] .. priorOffsets[i + 1]); null: every pair gets all numPriors
  if (priorOffsets) numPriors = priorOffsets[n];
  const size_t P = (size_t)proj->rows * proj->cols;
  int maxSlots = single ? 1 : env_int("NICP_BATCH_SLOTS", 256);
  if (maxSlots > slotCap) maxSlots = slotCap;
  if (maxSlots > n) maxSlots = n;
  int rc;
  if ((rc = ensure_align(ctx, maxSlots, P))) return rc;
  if ((rc = ensure_results(ctx, n))) return rc;
  if (single && (rc = ensure_trace(ctx, ap->outer_iterations > 0 ? ap->outer_iterations : 1))) return rc;
  if (single) ctx->zIter = ctx->zCurGen = -1;  // slot 0 is about to be used with its own epochs (also by a graph replay)
  if (numPriors > 0) {
    // SE3AbsolutePrior keeps the inverse of its reference transform (se3_prior.h setReferenceTransform)
    std::vector<HostPrior> hp(numPriors);
    for (int j = 0; j < numPriors; j++) {
      hp[j].kind = priors[j].kind;
      float m[16], r[16];
      for (int i = 0; i < 16; i++) { m[i] = priors[j].mean[i]; r[i] = priors[j].reference[i]; }
      for (int i = 0; i < 16; i++) hp[j].mean[i] = m[i];
      iso_inverse(r, hp[j].refInv);
      for (int i = 0; i < 36; i++) hp[j].info[i] = priors[j].information[i];
    }
    if (numPriors > ctx->priorCap) {
      invalidate_graphs(ctx);
      if (ctx->d_priors) cudaFree(ctx->d_priors);
      ctx->d_priors = nullptr;
      NICP_CUDA(cudaMalloc(&ctx->d_priors, sizeof(HostPrior) * numPriors));
      ctx->priorCap = numPriors;
    }
    NICP_CUDA(cudaMemcpyAsync(ctx->d_priors, hp.data(), sizeof(HostPrior) * numPriors, cudaMemcpyHostToDevice, ctx->stream));
    NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  AlignConsts ac = make_consts(proj, ap, refOffset);
  const CamSet cams = multiCams ? *multiCams : camset_pinhole(proj);
  if ((rc = upload_cams(ctx, cams))) return rc;
  ac.cams = &ctx->d_cams->set;
  float eye[16], co[16];
  mat4_identity(eye);
  for (int i = 0; i < 16; i++) co[i] = curOffset ? curOffset[i] : eye[i];
  fix_last_row(co);  // aligner.cpp:60: projector->setTransform(_currentSensorOffset)
  const int slots = ctx->slots;
  std::vector<int> owns(slots);
  int chunk = 0, prevBase = 0, prevM = 0;
  for (int base = 0; base < n; base += maxSlots, chunk++) {
    int m = n - base < maxSlots ? n - base : maxSlots;
    // chunk c stages into descriptor set c&1; the event of chunk c-2 (same set) was waited for when the
    // host post-processed that chunk, so the set is free
    select_desc_set(ctx, chunk & 1);
    // descriptor order inside the chunk: pairs that share a current cloud adjacent (stable, by first appearance), so that
    // the grouped kernel can walk them with the current side of a tile held in registers; the result of descriptor i
    // still goes to the record of the pair it came from
    std::map<const nicp_cloud *, int> curRank;
    std::vector<int> order(m), rankOf(m);
    for (int i = 0; i < m; i++) {
      const nicp_cloud *r = refs[base + i], *c = curs[base + i];
      if (!r || !c) {
        set_error("null cloud in pair %d", base + i);
        return NICP_ERR_INVALID;
      }
      if (r->device != ctx->device || c->device != ctx->device) {
        set_error("pair %d: cloud lives on GPU %d / %d, the context on GPU %d", base + i, r->device, c->device, ctx->device);
        return NICP_ERR_INVALID;
      }
      auto it = curRank.find(c);
      if (it == curRank.end()) it = curRank.insert(std::make_pair(c, (int)curRank.size())).first;
      rankOf[i] = it->second;
      order[i] = i;
    }
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return rankOf[a] < rankOf[b]; });
    std::vector<int> curSlotOf(m);
    for (int i = 0; i < m; i++) {
      const int src = base + order[i];
      const nicp_cloud *r = refs[src], *c = curs[src];
      const bool first = i == 0 || rankOf[order[i]] != rankOf[order[i - 1]];
      const int cs = first ? i : curSlotOf[i - 1];
      curSlotOf[i] = cs;
      owns[i] = first ? 1 : 0;
      fill_desc(ctx, i, cs, r, c, guesses ? guesses + 16 * (size_t)src : nullptr, ctx->d_results + src,
                single ? ctx->d_trace : nullptr);
      // big chunks are DRAM bound: the pinhole projection kernel streams the reference points from the packed copy
      // (a lone pair is latency bound and keeps the direct float4 loads)
      if (!cams.multi && m >= 8) {
        if ((rc = ensure_points3(ctx, const_cast<nicp_cloud *>(r)))) return rc;
        ctx->h_desc[i].refPoints3 = r->points3;
      }
      if (m >= 3 || ctx->groupMinAvg == 0) {  // chunks that may take the grouped kernel gather from the interleaved point + normal caches
        if ((rc = ensure_pn(ctx, const_cast<nicp_cloud *>(r))) || (rc = ensure_pn(ctx, const_cast<nicp_cloud *>(c)))) return rc;
        ctx->h_desc[i].refPN = r->pn;
        ctx->h_desc[i].curPN = c->pn;
      }
      if (numPriors > 0) {
        const int p0 = priorOffsets ? priorOffsets[src] : 0, p1 = priorOffsets ? priorOffsets[src + 1] : numPriors;
        ctx->h_desc[i].priors = p1 > p0 ? reinterpret_cast<const HostPrior *>(ctx->d_priors) + p0 : nullptr;
        ctx->h_desc[i].numPriors = p1 - p0;
      }
    }
    const int nGroups = stage_groups(ctx, m, curSlotOf.data());
    const bool useGraph = single && ctx->graphsEnabled && !cams.multi && !ctx->timing;
    bool replayed = false;
    cudaStream_t tail = ctx->stream;  // where this chunk's records are finished and copied out
    if (useGraph) {
      GraphKey key;
      memset(&key, 0, sizeof key);
      key.ac = ac;
      memcpy(key.co, co, sizeof co);
      key.outer = ap->outer_iterations; key.inner = ap->inner_iterations; key.numPriors = numPriors;
      key.slots = ctx->slots;
      key.partialRows = ctx->partialRows; key.imgThr = imgThr; key.slotPixels = ctx->slotPixels;
      key.desc = ctx->d_desc; key.results = ctx->d_results; key.statHb = ctx->d_statHb; key.trace = ctx->d_trace;
      key.priors = ctx->d_priors; key.refZ = ctx->d_refZ;
      int hit = -1, victim = 0;
      for (int g = 0; g < nicp_context::kGraphCache; g++) {
        if (ctx->graphValid[g] && memcmp(&key, ctx->graphKey[g], sizeof key) == 0) hit = g;
        if (!ctx->graphValid[g]) victim = g;
      }
      if (hit < 0) {
        bool anyFree = false;
        for (int g = 0; g < nicp_context::kGraphCache; g++) anyFree = anyFree || !ctx->graphValid[g];
        if (!anyFree) {
          victim = 0;
          for (int g = 1; g < nicp_context::kGraphCache; g++)
            if (ctx->graphUse[g] < ctx->graphUse[victim]) victim = g;  // least recently used
        }
      }
      if (hit >= 0) {
        NICP_CUDA(cudaGraphLaunch(ctx->graphExec[hit], ctx->stream));
        ctx->graphUse[hit] = ++ctx->graphClock;
        ctx->launches += ctx->graphLaunches[hit];  // the kernels the captured chunk launches
        replayed = true;
      } else {
        if (ctx->graphValid[victim]) {
          cudaGraphExecDestroy(ctx->graphExec[victim]);
          ctx->graphValid[victim] = false;
        }
        cudaGraph_t graph = nullptr;
        const long long launchesBefore = ctx->launches;
        NICP_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
        rc = run_align_chunk(ctx, m, ac, cams, co, ap->outer_iterations, ap->inner_iterations, imgThr, nGroups,
                             owns.data(), single, base);
        cudaError_t e1 = cudaMemcpyAsync(ctx->h_results + base, ctx->d_results + base, sizeof(nicp_align_result) * m,
                                         cudaMemcpyDeviceToHost, ctx->stream);
        cudaError_t e2 = cudaMemcpyAsync(ctx->h_statHb + (size_t)base * 42, ctx->d_statHb + (size_t)base * 42,
                                         sizeof(float) * 42 * m, cudaMemcpyDeviceToHost, ctx->stream);
        cudaError_t e3 = cudaStreamEndCapture(ctx->stream, &graph);
        if (rc) return rc;
        if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess || !graph) {
          set_error("CUDA graph capture of nicp_align failed: %s", cudaGetErrorString(e3 != cudaSuccess ? e3 : (e1 != cudaSuccess ? e1 : e2)));
          return NICP_ERR_CUDA;
        }
        NICP_CUDA(cudaGraphInstantiate(&ctx->graphExec[victim], graph, 0));
        cudaGraphDestroy(graph);
        memcpy(ctx->graphKey[victim], &key, sizeof key);
        ctx->graphValid[victim] = true;
        ctx->graphLaunches[victim] = ctx->launches - launchesBefore;
        ctx->graphUse[victim] = ++ctx->graphClock;
        NICP_CUDA(cudaGraphLaunch(ctx->graphExec[victim], ctx->stream));
        replayed = true;
      }
    }
    if (!replayed) {
      if ((rc = run_align_chunk(ctx, m, ac, cams, co, ap->outer_iterations, ap->inner_iterations, imgThr, nGroups,
                                owns.data(), single, base)))
        return rc;
      // a batch finishes its records (Aligner::_computeStatistics tail, one thread per pair: 0.1 ms of a nearly idle GPU)
      // and copies them out on the tail stream, beside the kernels of the next chunk
      if (!single) {
        NICP_CUDA(cudaEventRecord(ctx->evTail[chunk & 1], ctx->stream));
        NICP_CUDA(cudaStreamWaitEvent(ctx->tailStream, ctx->evTail[chunk & 1], 0));
        if ((rc = launch_statistics(ctx, ctx->tailStream, base, m))) return rc;
        tail = ctx->tailStream;
      }
      NICP_CUDA(cudaMemcpyAsync(ctx->h_results + base, ctx->d_results + base, sizeof(nicp_align_result) * m,
                                cudaMemcpyDeviceToHost, tail));
      NICP_CUDA(cudaMemcpyAsync(ctx->h_statHb + (size_t)base * 42, ctx->d_statHb + (size_t)base * 42, sizeof(float) * 42 * m,
                                cudaMemcpyDeviceToHost, tail));
    }
    NICP_CUDA(cudaEventRecord(ctx->evChunk[chunk & 1], tail));
    // while this chunk runs on the GPU, finish the previous one on the host (Aligner::_computeStatistics tail)
    if (chunk > 0) {
      NICP_CUDA(cudaEventSynchronize(ctx->evChunk[(chunk - 1) & 1]));
      finish_results(ctx, prevBase, prevM, results, !single);
    }
    prevBase = base;
    prevM = m;
  }
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->tailStream));
  collect_timing(ctx);
  finish_results(ctx, prevBase, prevM, results, !single);
  ctx->lastAlignRows = proj->rows;
  ctx->lastAlignCols = proj->cols;
  ctx->lastAlignIters = ap->outer_iterations;
  // which reference z-buffer / epoch the last iteration used (set here, not in run_align_chunk: a CUDA-graph replay
  // does not pass through it)
  ctx->lastAlignParity = ap->outer_iterations > 0 ? ((ap->outer_iterations - 1) & 1) : 0;
  ctx->lastAlignEpoch = ap->outer_iterations > 0 ? epoch_of_iteration(ap->outer_iterations - 1) : kEpochFresh;
  ctx->lastAlignValid = single;
  ctx->lastAlignEmptyDepth = cams.multi ? 0.0f : FLT_MAX;
  return NICP_OK;
}

int nicp_align(nicp_context *ctx, const nicp_cloud *reference, const nicp_cloud *current, const nicp_projector *proj,
               const nicp_align_params *ap, const float reference_sensor_offset[16], const float current_sensor_offset[16],
               const float initial_guess[16], const nicp_prior *priors, int num_priors, float frame_inlier_depth_threshold,
               nicp_align_result *result) {
  if (!ctx || !reference || !current || !proj || !ap || !result || proj->rows <= 0 || proj->cols <= 0) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  if (num_priors < 0 || (num_priors > 0 && !priors)) return NICP_ERR_INVALID;
  return align_common(ctx, 1, &reference, &current, proj, ap, reference_sensor_offset, current_sensor_offset, initial_guess,
                      frame_inlier_depth_threshold, result, true, priors, num_priors);
}

int nicp_align_batch(nicp_context *ctx, int n, const nicp_cloud *const *references, const nicp_cloud *const *currents,
                     const nicp_projector *proj, const nicp_align_params *ap, const float reference_sensor_offset[16],
                     const float current_sensor_offset[16], const float *initial_guesses, float frame_inlier_depth_threshold,
                     nicp_align_result *results) {
  if (!ctx || n < 0 || !proj || !ap || proj->rows <= 0 || proj->cols <= 0) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  if (n == 0) return NICP_OK;
  if (!references || !currents || !results) return NICP_ERR_INVALID;
  return align_common(ctx, n, references, currents, proj, ap, reference_sensor_offset, current_sensor_offset, initial_guesses,
                      frame_inlier_depth_threshold, results, false);
}

int nicp_align_batch_priors(nicp_context *ctx, int n, const nicp_cloud *const *references, const nicp_cloud *const *currents,
                            const nicp_projector *proj, const nicp_align_params *ap, const float reference_sensor_offset[16],
                            const float current_sensor_offset[16], const float *initial_guesses, const nicp_prior *priors,
                            const int *prior_offsets, float frame_inlier_depth_threshold, nicp_align_result *results) {
  if (!ctx || n < 0 || !proj || !ap || proj->rows <= 0 || proj->cols <= 0) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  if (n == 0) return NICP_OK;
  if (!references || !currents || !results) return NICP_ERR_INVALID;
  if (!prior_offsets_valid(n, priors, prior_offsets)) return NICP_ERR_INVALID;
  return align_common(ctx, n, references, currents, proj, ap, reference_sensor_offset, current_sensor_offset, initial_guesses,
                      frame_inlier_depth_threshold, results, false, priors, 0, nullptr, prior_offsets);
}

void nicp_multi_image_size(const nicp_multi_projector *mp, int *rows, int *cols) {
  CamSet c;
  int r = 0, cc = 0;
  if (camset_multi(mp, c, r, cc) != NICP_OK) r = cc = 0;
  if (rows) *rows = r;
  if (cols) *cols = cc;
}

int nicp_multi_depth_to_cloud(nicp_context *ctx, const float *depth, const nicp_multi_projector *mp, const nicp_stats_params *sp,
                              const float sensor_offset[16], int keep_stats, nicp_cloud *cloud, int *index) {
  if (!ctx || !depth || !mp || !sp || !cloud) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  CamSet cams;
  int rows, cols, rc;
  if ((rc = camset_multi(mp, cams, rows, cols))) return rc;
  size_t px = (size_t)rows * cols;
  if ((size_t)cloud->capacity < px) {
    set_error("cloud capacity %d smaller than the composite image (%zu pixels)", cloud->capacity, px);
    return NICP_ERR_INVALID;
  }
  if ((rc = ensure_prep(ctx, px))) return rc;
  if ((rc = upload_cams(ctx, cams))) return rc;
  if (keep_stats && (rc = ensure_stats(cloud))) return rc;
  NICP_CUDA(cudaMemcpyAsync(ctx->d_depth, depth, px * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  nicp_projector proj = mp->camera[0];
  proj.rows = rows;
  proj.cols = cols;
  float eye[16];
  mat4_identity(eye);
  if ((rc = launch_frame_prep(ctx, ctx->d_depth, &proj, sp, sensor_offset ? sensor_offset : eye, keep_stats, cloud,
                              ctx->d_index, &cams)))
    return rc;
  if (index) NICP_CUDA(cudaMemcpyAsync(index, ctx->d_index, px * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  return NICP_OK;
}

int nicp_multi_project(nicp_context *ctx, const nicp_cloud *cloud, const nicp_multi_projector *mp, const float T[16],
                       int *index, float *depth) {
  if (!ctx || !cloud || !mp || !T) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  CamSet cams;
  int rows, cols, rc;
  if ((rc = camset_multi(mp, cams, rows, cols))) return rc;
  size_t px = (size_t)rows * cols;
  if ((rc = ensure_align(ctx, 1, px))) return rc;
  if ((rc = ensure_prep(ctx, px))) return rc;
  float Tf[16];
  for (int i = 0; i < 16; i++) Tf[i] = T[i];
  fix_last_row(Tf);
  unsigned long long *z = ctx->d_curZ;
  if ((rc = launch_project_cams(ctx, cloud, cams, Tf, rows, cols, z))) return rc;
  if ((rc = launch_decode_z(ctx, z, (int)px, ctx->d_index, ctx->d_depth, 0.0f))) return rc;
  if (index) NICP_CUDA(cudaMemcpyAsync(index, ctx->d_index, px * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  if (depth) NICP_CUDA(cudaMemcpyAsync(depth, ctx->d_depth, px * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  ctx->lastAlignValid = false;
  return NICP_OK;
}

int nicp_multi_align(nicp_context *ctx, const nicp_cloud *reference, const nicp_cloud *current, const nicp_multi_projector *mp,
                     const nicp_align_params *ap, const float reference_sensor_offset[16], const float current_sensor_offset[16],
                     const float initial_guess[16], const nicp_prior *priors, int num_priors, float frame_inlier_depth_threshold,
                     nicp_align_result *result) {
  if (!ctx || !reference || !current || !mp || !ap || !result) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  if (num_priors < 0 || (num_priors > 0 && !priors)) return NICP_ERR_INVALID;
  CamSet cams;
  int rows, cols, rc;
  if ((rc = camset_multi(mp, cams, rows, cols))) return rc;
  nicp_projector proj = mp->camera[0];
  proj.rows = rows;
  proj.cols = cols;
  return align_common(ctx, 1, &reference, &current, &proj, ap, reference_sensor_offset, current_sensor_offset, initial_guess,
                      frame_inlier_depth_threshold, result, true, priors, num_priors, &cams);
}

int nicp_multi_align_batch(nicp_context *ctx, int n, const nicp_cloud *const *references, const nicp_cloud *const *currents,
                           const nicp_multi_projector *mp, const nicp_align_params *ap, const float reference_sensor_offset[16],
                           const float current_sensor_offset[16], const float *initial_guesses, const nicp_prior *priors,
                           const int *prior_offsets, float frame_inlier_depth_threshold, nicp_align_result *results) {
  if (!ctx || n < 0 || !mp || !ap) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  if (n == 0) return NICP_OK;
  if (!references || !currents || !results) return NICP_ERR_INVALID;
  if (!prior_offsets_valid(n, priors, prior_offsets)) return NICP_ERR_INVALID;
  CamSet cams;
  int rows, cols, rc;
  if ((rc = camset_multi(mp, cams, rows, cols))) return rc;
  nicp_projector proj = mp->camera[0];
  proj.rows = rows;
  proj.cols = cols;
  // a slot holds 32 B per pixel of z-buffers and index images: a chunk gets at most the memory of 256 pinhole 640x480 slots
  // (2.5 GB; 16 slots at 1280x3840)
  const size_t P = (size_t)rows * cols;
  const int slotCap = (int)std::max<size_t>(1, (size_t)256 * 640 * 480 / P);
  return align_common(ctx, n, references, currents, &proj, ap, reference_sensor_offset, current_sensor_offset, initial_guesses,
                      frame_inlier_depth_threshold, results, false, priors, 0, &cams, prior_offsets, slotCap);
}

int nicp_align_get_state(nicp_context *ctx, int *reference_index, float *reference_depth, int *current_index,
                         float *current_depth, int *correspondences, float H[36], float b[6]) {
  if (!ctx || !ctx->lastAlignValid) {
    set_error("no single nicp_align state available on this context");
    return NICP_ERR_INVALID;
  }
  NICP_CUDA(cudaSetDevice(ctx->device));
  const size_t P = (size_t)ctx->lastAlignRows * ctx->lastAlignCols;
  int rc;
  if ((rc = ensure_prep(ctx, P))) return rc;
  const PairDesc &D = ctx->h_desc[0];
  std::vector<int> ci, corrImg;
  if (reference_index || reference_depth) {
    if ((rc = launch_decode_z(ctx, D.refZ[ctx->lastAlignParity], (int)P, ctx->d_index, ctx->d_depth, ctx->lastAlignEmptyDepth,
                              ctx->lastAlignEpoch)))
      return rc;
    if (reference_index) NICP_CUDA(cudaMemcpyAsync(reference_index, ctx->d_index, P * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (reference_depth) NICP_CUDA(cudaMemcpyAsync(reference_depth, ctx->d_depth, P * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  if (current_index || current_depth) {
    if ((rc = launch_decode_z(ctx, D.curZ, (int)P, ctx->d_index, ctx->d_depth, ctx->lastAlignEmptyDepth))) return rc;
    if (current_index) NICP_CUDA(cudaMemcpyAsync(current_index, ctx->d_index, P * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (current_depth) NICP_CUDA(cudaMemcpyAsync(current_depth, ctx->d_depth, P * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  if (correspondences) {
    ci.resize(P);
    corrImg.resize(P);
    NICP_CUDA(cudaMemcpyAsync(ci.data(), D.curIndex, P * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    NICP_CUDA(cudaMemcpyAsync(corrImg.data(), D.corrImage, P * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    NICP_CUDA(cudaStreamSynchronize(ctx->stream));
    size_t k = 0;  // raster-order compaction, the order of correspondencefinder.cpp:108-113
    for (size_t p = 0; p < P; p++)
      if (corrImg[p] >= 0) {
        correspondences[2 * k] = corrImg[p];
        correspondences[2 * k + 1] = ci[p];
        k++;
      }
  }
  if (H) memcpy(H, ctx->h_statHb, sizeof(float) * 36);
  if (b) memcpy(b, ctx->h_statHb + 36, sizeof(float) * 6);
  return NICP_OK;
}

int nicp_align_get_trace(nicp_context *ctx, float *trace61, int max_iterations) {
  if (!ctx || !trace61 || !ctx->lastAlignValid) return NICP_ERR_INVALID;
  NICP_CUDA(cudaSetDevice(ctx->device));
  int it = ctx->lastAlignIters < max_iterations ? ctx->lastAlignIters : max_iterations;
  if (it <= 0) return NICP_OK;
  NICP_CUDA(cudaMemcpyAsync(trace61, ctx->d_trace, sizeof(float) * 61 * it, cudaMemcpyDeviceToHost, ctx->stream));
  NICP_CUDA(cudaStreamSynchronize(ctx->stream));
  return NICP_OK;
}

}  // extern "C"

// shard.cu -- pair-wise sharding of batched alignment over the GPUs of one process (SURVEY.md section 8e).
//
// The caller that owns this loop in the reference is the loop closer: PwnCloser::processPartition walks the candidate
// pairs of a partition one by one, builds (or fetches from its cache) the clouds of both frames and matches them
// (pwn_tracker2/pwn_closer.cpp:83-182 -> PwnMatcherBase::makeCloud / matchClouds, pwn_matcher_base.cpp:46-196).  Pairs are
// independent, so the pair list is cut into contiguous blocks, one per device; every device builds the clouds of the
// frames ITS pairs reference from the raw images (a frame needed on two devices is prepared on both: 50 MB of local
// traffic instead of 25 MB over NVLink) and aligns its block; the only "collective" is the result records landing in the
// caller's array.  No data-path exchange, hence no NCCL here: one process, host memory is shared.  (The one-process-per-
// GPU deployment gathers the same 256-byte records with one all-gather, g2o_frontend_b200/sharding.py.)
//
// One worker thread per device per call; each worker owns a nicp_context (one context per host thread / GPU, like the
// rest of the library) and a cache of device clouds that persists across calls.
//
// MultiPointProjector rigs (nicp_multi_align_frames_sharded) take the same partition with two differences.  A rig cloud at
// BASELINE config 5 (1280 x 3840 composite) is ~550 MB, so a worker does not build every frame of its block at once: it
// walks the block in windows, a window being the longest run of consecutive pairs whose distinct frames fit in the
// worker's frame cap, keeps the clouds of frames the next window still uses and rebuilds only the others into the freed
// slots.  And rigs keep a cloud cache of their own, so that a rig call never grows the pinhole cache to rig size.  A frame
// needed on two devices is still prepared on both: whether shipping its cloud would be cheaper than preparing it again is
// an open question for rigs (tools/rig_sharded_timing.py reports the prep / align split that decides it).
#include <algorithm>
#include <climits>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <thread>
#include <vector>

#include "nicp_internal.cuh"

struct nicp_shard_pool {
  struct Worker {
    int device;
    nicp_context *ctx;
    std::vector<nicp_cloud *> clouds;  // cache, capacity = cloudCapacity each
    int cloudCapacity;
    std::vector<nicp_cloud *> rigClouds;  // rig cache (nicp_multi_align_frames_sharded), capacity = rigCapacity each
    int rigCapacity;
    size_t deviceBytes;   // memory of this worker's GPU
    int workersOnDevice;  // workers of the pool sharing that GPU (this one included)
    int rc;
    std::string error;
  };
  std::vector<Worker> workers;
  int rigFrameCap;  // NICP_SHARD_FRAMES (>= 2), 0 = unset
};

using namespace nicp;

// frames a worker keeps as rig clouds of px composite pixels at once.  A rig cloud costs 112 B per pixel: 80 B of points,
// normals and Omega, and the 32 B interleaved point / normal copy its first alignment adds (ensure_pn).  The clouds of the
// workers sharing a GPU take at most half of its memory, the rest is left to the prep and align scratch and to the
// caller; NICP_SHARD_FRAMES lowers the cap.  At least 2, so that any pair fits.
static int rig_frame_cap(const nicp_shard_pool *pool, const nicp_shard_pool::Worker &w, size_t px) {
  const size_t fit = w.deviceBytes / 2 / (112 * px) / (size_t)w.workersOnDevice;
  int cap = (int)std::min<size_t>(fit, INT_MAX);
  if (pool->rigFrameCap && pool->rigFrameCap < cap) cap = pool->rigFrameCap;
  return std::max(cap, 2);
}

extern "C" {

int nicp_shard_pool_create(const int *devices, int n_devices, nicp_shard_pool **out) {
  if (!out) return NICP_ERR_INVALID;
  *out = nullptr;
  if (!devices || n_devices <= 0) {
    set_error("a shard pool needs at least one device");
    return NICP_ERR_INVALID;
  }
  nicp_shard_pool *pool = new nicp_shard_pool();
  pool->workers.resize(n_devices);
  for (int i = 0; i < n_devices; i++) {
    nicp_shard_pool::Worker &w = pool->workers[i];
    w.device = devices[i];
    w.ctx = nullptr;
    w.cloudCapacity = 0;
    w.rigCapacity = 0;
    w.workersOnDevice = (int)std::count(devices, devices + n_devices, devices[i]);
    w.rc = NICP_OK;
    int rc = nicp_create(devices[i], &w.ctx);  // fails loudly without a usable GPU: there is no CPU fallback
    cudaDeviceProp prop;
    if (rc == NICP_OK && cudaGetDeviceProperties(&prop, devices[i]) != cudaSuccess) {
      set_error("cudaGetDeviceProperties(%d) failed", devices[i]);
      rc = NICP_ERR_CUDA;
    }
    if (rc != NICP_OK) {
      for (int j = 0; j <= i; j++) nicp_destroy(pool->workers[j].ctx);
      delete pool;
      return rc;
    }
    w.deviceBytes = prop.totalGlobalMem;
  }
  const char *v = getenv("NICP_SHARD_FRAMES");
  pool->rigFrameCap = (v && *v) ? std::max(2, atoi(v)) : 0;
  *out = pool;
  return NICP_OK;
}

void nicp_shard_pool_destroy(nicp_shard_pool *pool) {
  if (!pool) return;
  for (nicp_shard_pool::Worker &w : pool->workers) {
    for (nicp_cloud *c : w.clouds) nicp_cloud_destroy(c);
    for (nicp_cloud *c : w.rigClouds) nicp_cloud_destroy(c);
    nicp_destroy(w.ctx);
  }
  delete pool;
}

int nicp_shard_pool_size(const nicp_shard_pool *pool) { return pool ? (int)pool->workers.size() : 0; }

int nicp_align_frames_sharded(nicp_shard_pool *pool, int n_frames, const uint16_t *const *raws, int raw_rows, int raw_cols,
                              float depth_scale, int step, float max_depth_cov, const nicp_projector *proj,
                              const nicp_stats_params *sp, const float sensor_offset[16], int n_pairs,
                              const int *reference_frame, const int *current_frame, const float *initial_guesses,
                              const nicp_align_params *ap, float frame_inlier_depth_threshold, nicp_align_result *results) {
  if (!pool || n_frames < 0 || n_pairs < 0 || !proj || !sp || !ap || raw_rows <= 0 || raw_cols <= 0) return NICP_ERR_INVALID;
  if (n_pairs == 0) return NICP_OK;
  if (!raws || !reference_frame || !current_frame || !results) return NICP_ERR_INVALID;
  for (int i = 0; i < n_pairs; i++)
    if (reference_frame[i] < 0 || reference_frame[i] >= n_frames || current_frame[i] < 0 || current_frame[i] >= n_frames) {
      set_error("pair %d references frame %d / %d outside [0, %d)", i, reference_frame[i], current_frame[i], n_frames);
      return NICP_ERR_INVALID;
    }
  for (int f = 0; f < n_frames; f++)
    if (!raws[f]) {
      set_error("frame %d is null", f);
      return NICP_ERR_INVALID;
    }
  const int G = (int)pool->workers.size();
  const int px = proj->rows * proj->cols;

  auto work = [&](int g) {
    nicp_shard_pool::Worker &w = pool->workers[g];
    w.rc = NICP_OK;
    w.error.clear();
    // static block partition of the pair list (SURVEY.md 8e): device g takes pairs [g n / G, (g + 1) n / G)
    const long long lo = (long long)g * n_pairs / G, hi = (long long)(g + 1) * n_pairs / G;
    const int m = (int)(hi - lo);
    if (m <= 0) return;
    auto fail = [&](int rc) {
      w.rc = rc;
      w.error = nicp_last_error();  // this worker thread's message
    };
    // the frames this block references, in order of first use -> local cloud slots
    std::map<int, int> slotOf;
    std::vector<int> frames;
    for (long long i = lo; i < hi; i++)
      for (int f : {current_frame[i], reference_frame[i]})
        if (slotOf.find(f) == slotOf.end()) {
          slotOf[f] = (int)frames.size();
          frames.push_back(f);
        }
    if (w.cloudCapacity < px) {  // a different image size: the cache starts over
      for (nicp_cloud *c : w.clouds) nicp_cloud_destroy(c);
      w.clouds.clear();
      w.cloudCapacity = px;
    }
    while (w.clouds.size() < frames.size()) {
      nicp_cloud *c = nullptr;
      int rc = nicp_cloud_create(w.ctx, w.cloudCapacity, &c);
      if (rc) return fail(rc);
      w.clouds.push_back(c);
    }
    std::vector<const uint16_t *> r(frames.size());
    for (size_t k = 0; k < frames.size(); k++) r[k] = raws[frames[k]];
    int rc = nicp_raw_depth_to_cloud_batch(w.ctx, (int)frames.size(), r.data(), raw_rows, raw_cols, depth_scale, step,
                                           max_depth_cov, proj, sp, sensor_offset, 0, w.clouds.data());
    if (rc) return fail(rc);
    std::vector<const nicp_cloud *> refs(m), curs(m);
    for (int i = 0; i < m; i++) {
      refs[i] = w.clouds[slotOf[reference_frame[lo + i]]];
      curs[i] = w.clouds[slotOf[current_frame[lo + i]]];
    }
    rc = nicp_align_batch(w.ctx, m, refs.data(), curs.data(), proj, ap, sensor_offset, sensor_offset,
                          initial_guesses ? initial_guesses + 16 * lo : nullptr, frame_inlier_depth_threshold, results + lo);
    if (rc) return fail(rc);
  };

  if (G == 1) {
    work(0);
  } else {
    std::vector<std::thread> threads;
    threads.reserve(G);
    for (int g = 0; g < G; g++) threads.emplace_back(work, g);
    for (std::thread &t : threads) t.join();
  }
  for (int g = 0; g < G; g++)
    if (pool->workers[g].rc != NICP_OK) {
      set_error("device %d (shard %d of %d): %s", pool->workers[g].device, g, G, pool->workers[g].error.c_str());
      return pool->workers[g].rc;
    }
  return NICP_OK;
}

int nicp_multi_align_frames_sharded(nicp_shard_pool *pool, int n_frames, const uint16_t *const *raws, const int *raw_rows,
                                    const int *raw_cols, float depth_scale, int step, float max_depth_cov,
                                    const nicp_multi_projector *mp, const nicp_stats_params *sp,
                                    const float sensor_offset[16], int n_pairs, const int *reference_frame,
                                    const int *current_frame, const float *initial_guesses, const nicp_prior *priors,
                                    const int *prior_offsets, const nicp_align_params *ap,
                                    float frame_inlier_depth_threshold, nicp_align_result *results) {
  if (!pool || n_frames < 0 || n_pairs < 0 || !mp || !sp || !ap) return NICP_ERR_INVALID;
  if (n_pairs == 0) return NICP_OK;
  if (!raws || !raw_rows || !raw_cols || !reference_frame || !current_frame || !results) return NICP_ERR_INVALID;
  // every check the workers' batch calls would make, here in the calling thread: the error is the same whichever worker
  // would have met it first
  int rows = 0, cols = 0;
  nicp_multi_image_size(mp, &rows, &cols);
  if (rows <= 0 || cols <= 0) {
    set_error("multi projector needs 1..%d cameras of positive size", NICP_MAX_CAMERAS);
    return NICP_ERR_INVALID;
  }
  const int nc = mp->num_cameras;
  if (step < 1) step = 1;
  for (int i = 0; i < nc; i++)
    if (raw_rows[i] <= 0 || raw_cols[i] <= 0 || raw_rows[i] / step != mp->camera[i].cols ||
        raw_cols[i] / step != mp->camera[i].rows) {
      set_error("camera %d: raw image %dx%d at step %d does not scale to the projector's %dx%d (rows x cols = height x width)",
                i, raw_rows[i], raw_cols[i], step, mp->camera[i].cols, mp->camera[i].rows);
      return NICP_ERR_INVALID;
    }
  for (int i = 0; i < n_pairs; i++)
    if (reference_frame[i] < 0 || reference_frame[i] >= n_frames || current_frame[i] < 0 || current_frame[i] >= n_frames) {
      set_error("pair %d references frame %d / %d outside [0, %d)", i, reference_frame[i], current_frame[i], n_frames);
      return NICP_ERR_INVALID;
    }
  for (int f = 0; f < n_frames; f++)
    for (int i = 0; i < nc; i++)
      if (!raws[(size_t)f * nc + i]) {
        set_error("null raw image of camera %d in frame %d", i, f);
        return NICP_ERR_INVALID;
      }
  if (!prior_offsets_valid(n_pairs, priors, prior_offsets)) {
    int bad = 0;
    while (bad < n_pairs && prior_offsets[bad + 1] >= prior_offsets[bad]) bad++;
    if (prior_offsets[0] != 0)
      set_error("prior_offsets[0] is %d, not 0", prior_offsets[0]);
    else if (bad < n_pairs)
      set_error("prior_offsets decrease at pair %d (%d -> %d)", bad, prior_offsets[bad], prior_offsets[bad + 1]);
    else
      set_error("prior_offsets name %d priors but priors is null", prior_offsets[n_pairs]);
    return NICP_ERR_INVALID;
  }
  const int G = (int)pool->workers.size();
  const size_t px = (size_t)rows * cols;

  auto work = [&](int g) {
    nicp_shard_pool::Worker &w = pool->workers[g];
    w.rc = NICP_OK;
    w.error.clear();
    // the pinhole partition: worker g takes pairs [g n / G, (g + 1) n / G)
    const long long lo = (long long)g * n_pairs / G, hi = (long long)(g + 1) * n_pairs / G;
    if (hi <= lo) return;
    auto fail = [&](int rc) {
      w.rc = rc;
      w.error = nicp_last_error();
    };
    if ((size_t)w.rigCapacity != px) {  // another composite size: the rig cache starts over, so it never holds more than cap
      for (nicp_cloud *c : w.rigClouds) nicp_cloud_destroy(c);
      w.rigClouds.clear();
      w.rigCapacity = (int)px;
    }
    const size_t cap = (size_t)rig_frame_cap(pool, w, px);
    std::vector<int> slotFrame(w.rigClouds.size(), -1);  // frame held by each cached cloud; none from this call yet
    std::map<int, int> slotOf;                           // frame -> slot, for the frames of the current window
    std::vector<const uint16_t *> buildRaws;
    std::vector<nicp_cloud *> buildClouds;
    std::vector<const nicp_cloud *> refs, curs;
    std::vector<int> offs;
    for (long long i = lo; i < hi;) {
      // the window: the longest run of pairs from i whose distinct frames fit in cap (one pair always does)
      slotOf.clear();
      long long j = i;
      for (; j < hi; j++) {
        const int a = reference_frame[j], b = current_frame[j];
        const size_t grow = (slotOf.count(a) ? 0 : 1) + (a == b || slotOf.count(b) ? 0 : 1);
        if (slotOf.size() + grow > cap) break;
        slotOf.emplace(a, -1);
        slotOf.emplace(b, -1);
      }
      // keep the clouds of the window's frames that are resident; the other frames go to empty slots first, then to new
      // clouds while the cache is below cap, then to the slots of frames this window does not use
      std::vector<char> taken(slotFrame.size(), 0);
      for (size_t s = 0; s < slotFrame.size(); s++) {
        auto it = slotFrame[s] >= 0 ? slotOf.find(slotFrame[s]) : slotOf.end();
        if (it != slotOf.end()) {
          it->second = (int)s;
          taken[s] = 1;
        }
      }
      buildRaws.clear();
      buildClouds.clear();
      for (auto &fs : slotOf) {
        if (fs.second >= 0) continue;
        size_t s = 0;
        while (s < slotFrame.size() && (taken[s] || slotFrame[s] >= 0)) s++;
        if (s == slotFrame.size() && slotFrame.size() < cap) {
          nicp_cloud *c = nullptr;
          int rc = nicp_cloud_create(w.ctx, (int)px, &c);
          if (rc) return fail(rc);
          w.rigClouds.push_back(c);
          slotFrame.push_back(-1);
          taken.push_back(0);
        }
        if (s == slotFrame.size()) s = std::find(taken.begin(), taken.end(), 0) - taken.begin();
        taken[s] = 1;
        slotFrame[s] = fs.first;
        fs.second = (int)s;
        for (int c = 0; c < nc; c++) buildRaws.push_back(raws[(size_t)fs.first * nc + c]);
        buildClouds.push_back(w.rigClouds[s]);
      }
      int rc;
      if (!buildClouds.empty() &&
          (rc = nicp_multi_raw_depth_to_cloud_batch(w.ctx, (int)buildClouds.size(), buildRaws.data(), raw_rows, raw_cols,
                                                    depth_scale, step, max_depth_cov, mp, sp, sensor_offset, 0,
                                                    buildClouds.data())))
        return fail(rc);
      const int m = (int)(j - i);
      refs.resize(m);
      curs.resize(m);
      for (int k = 0; k < m; k++) {
        refs[k] = w.rigClouds[slotOf[reference_frame[i + k]]];
        curs[k] = w.rigClouds[slotOf[current_frame[i + k]]];
      }
      // the window's priors, with prior_offsets rebased to its first pair
      const nicp_prior *wp = nullptr;
      if (prior_offsets) {
        offs.resize(m + 1);
        for (int k = 0; k <= m; k++) offs[k] = prior_offsets[i + k] - prior_offsets[i];
        if (priors) wp = priors + prior_offsets[i];
      }
      if ((rc = nicp_multi_align_batch(w.ctx, m, refs.data(), curs.data(), mp, ap, sensor_offset, sensor_offset,
                                       initial_guesses ? initial_guesses + 16 * i : nullptr, wp,
                                       prior_offsets ? offs.data() : nullptr, frame_inlier_depth_threshold, results + i)))
        return fail(rc);
      i = j;
    }
  };

  if (G == 1) {
    work(0);
  } else {
    std::vector<std::thread> threads;
    threads.reserve(G);
    for (int g = 0; g < G; g++) threads.emplace_back(work, g);
    for (std::thread &t : threads) t.join();
  }
  for (int g = 0; g < G; g++)
    if (pool->workers[g].rc != NICP_OK) {
      set_error("device %d (shard %d of %d): %s", pool->workers[g].device, g, G, pool->workers[g].error.c_str());
      return pool->workers[g].rc;
    }
  return NICP_OK;
}

}  // extern "C"

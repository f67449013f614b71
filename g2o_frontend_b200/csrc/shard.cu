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
// Pinhole frames (nicp_align_frames_sharded) and MultiPointProjector rig frames (nicp_multi_align_frames_sharded) take the
// same path: a pinhole camera is a frame set of one camera (FrameSet, nicp_internal.cuh).  A rig cloud at BASELINE config 5
// (1280 x 3840 composite) is ~550 MB, so a worker does not build every frame of its block at once: it walks the block in
// windows, a window being the longest run of consecutive pairs whose distinct frames fit in the worker's frame cap, keeps
// the clouds of frames the next window still uses and rebuilds only the others into the freed slots.  At 640 x 480 the cap
// is thousands of frames, so a pinhole block is one window.  A frame needed on two devices is still prepared on both:
// whether shipping its cloud would be cheaper than preparing it again is an open question for rigs
// (tools/rig_sharded_timing.py reports the prep / align split that decides it).
//
// A frame store (nicp_frame_store_*) runs the same walker with frames named by caller-chosen ids instead of the index in
// one call's array, and with a slot table per worker that outlives the call: the incremental closer's PwnCloudCache
// (pwn_tracker2/pwn_cloud_cache.cpp:60-102), which rebuilds a node's cloud only after it was evicted.
#include <algorithm>
#include <climits>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <thread>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "nicp_internal.cuh"

// The clouds a worker holds for one key space, slot by slot.  The sharded entries share one per worker whose keys are the
// frame indices of the call in flight (emptied when a call starts); a frame store has one per worker whose keys are frame
// ids and which lasts across calls.
struct Residency {
  size_t px = 0;                         // pixels every cloud holds
  std::vector<nicp_cloud *> clouds;
  std::vector<char> held;                // slot s holds the complete cloud of frame key[s]
  std::vector<long long> key;
  std::vector<unsigned long long> used;  // stamp of the last window that used slot s (least recently used goes first)
  unsigned long long stamp = 0;
  long long built = 0, reused = 0;       // frames a window prepared / found held, since creation

  void release() {
    for (nicp_cloud *c : clouds) nicp_cloud_destroy(c);
    clouds.clear();
    held.clear();
    key.clear();
    used.clear();
  }
  void drop(long long k) {
    for (size_t s = 0; s < clouds.size(); s++)
      if (held[s] && key[s] == k) held[s] = 0;
  }
};

struct nicp_shard_pool {
  struct Worker {
    int device;
    nicp_context *ctx;
    Residency calls;      // cloud cache of nicp_align_frames_sharded / nicp_multi_align_frames_sharded
    size_t deviceBytes;   // memory of this worker's GPU
    int workersOnDevice;  // workers of the pool sharing that GPU (this one included)
    int rc;
    std::string error;
  };
  std::vector<Worker> workers;
  int frameCap;  // NICP_SHARD_FRAMES (>= 2), 0 = unset
  std::vector<nicp_frame_store *> stores;  // released when the pool is destroyed
};

struct nicp_frame_store {
  nicp_shard_pool *pool;  // null once the pool has been destroyed
  nicp::FrameSet fs;
  nicp_stats_params sp;
  float sensorOffset[16];
  bool hasOffset;
  std::unordered_map<long long, std::vector<uint16_t>> raws;  // id -> raw images of its cameras, back to back
  std::vector<Residency> res;                                  // one per worker of the pool
};

using namespace nicp;

// frames a worker keeps as clouds of px pixels at once.  A cloud costs 112 B per pixel: 80 B of points, normals and Omega,
// and the 32 B interleaved point / normal copy its first alignment adds (ensure_pn; a pinhole cloud aligned in chunks of
// 8+ pairs also gets the 12 B packed point copy of ensure_points3).  The clouds of the workers sharing a GPU take about
// half of its memory, the rest is left to the prep and align scratch and to the caller; NICP_SHARD_FRAMES lowers the cap.
// At least 2, so that any pair fits.
static int frame_cap(const nicp_shard_pool *pool, const nicp_shard_pool::Worker &w, size_t px) {
  const size_t fit = w.deviceBytes / 2 / (112 * px) / (size_t)w.workersOnDevice;
  int cap = (int)std::min<size_t>(fit, INT_MAX);
  if (pool->frameCap && pool->frameCap < cap) cap = pool->frameCap;
  return std::max(cap, 2);
}

// The pairs of a sharded call, frames in and records out: every check in the calling thread, so that the error is the same
// whichever worker would have met it first, then worker g takes pairs [g n / G, (g + 1) n / G) (SURVEY.md 8e) and walks
// them in windows.  fs has been validated by frames_pinhole / frames_rig.  Frame f of the call is resident under key
// keys[f] in store's slot tables, or under key f in the workers' per-call caches when store is null.
static int align_frames_sharded(nicp_shard_pool *pool, nicp_frame_store *store, const long long *keys, const FrameSet &fs,
                                int n_frames, const uint16_t *const *raws, const nicp_stats_params *sp,
                                const float sensor_offset[16], int n_pairs, const int *reference_frame,
                                const int *current_frame, const float *initial_guesses, const nicp_prior *priors,
                                const int *prior_offsets, const nicp_align_params *ap, float frame_inlier_depth_threshold,
                                nicp_align_result *results) {
  if (!raws || !reference_frame || !current_frame || !results) return NICP_ERR_INVALID;
  for (int i = 0; i < n_pairs; i++)
    if (reference_frame[i] < 0 || reference_frame[i] >= n_frames || current_frame[i] < 0 || current_frame[i] >= n_frames) {
      set_error("pair %d references frame %d / %d outside [0, %d)", i, reference_frame[i], current_frame[i], n_frames);
      return NICP_ERR_INVALID;
    }
  const int nc = fs.cams.n;
  for (int f = 0; f < n_frames; f++)
    for (int i = 0; i < nc; i++)
      if (!raws[(size_t)f * nc + i]) {
        set_error("null raw image of camera %d in frame %d", i, f);
        return NICP_ERR_INVALID;
      }
  int rc;
  if ((rc = check_prior_offsets(n_pairs, priors, prior_offsets))) return rc;
  const size_t px = (size_t)fs.proj.rows * fs.proj.cols;

  // pairs [lo, hi) on worker w, with the clouds of res
  auto align_block = [&](nicp_shard_pool::Worker &w, Residency &res, long long lo, long long hi) -> int {
    NICP_CUDA(cudaSetDevice(w.device));
    const size_t cap = (size_t)frame_cap(pool, w, px);
    struct Use {
      int frame, slot;
    };
    std::map<long long, Use> win;                     // key -> frame of this call and slot, for the frames of the window
    std::vector<std::pair<int, long long>> fresh;     // slots the window builds and the keys they will hold
    std::vector<const uint16_t *> buildRaws;
    std::vector<nicp_cloud *> buildClouds;
    std::vector<const nicp_cloud *> refs, curs;
    std::vector<int> offs;
    auto keyOf = [&](int f) { return keys ? keys[f] : (long long)f; };
    for (long long i = lo; i < hi;) {
      // the window: the longest run of pairs from i whose distinct frames fit in cap (one pair always does)
      win.clear();
      long long j = i;
      for (; j < hi; j++) {
        const int a = reference_frame[j], b = current_frame[j];
        const long long ka = keyOf(a), kb = keyOf(b);
        const size_t grow = (win.count(ka) ? 0 : 1) + (ka == kb || win.count(kb) ? 0 : 1);
        if (win.size() + grow > cap) break;
        win.emplace(ka, Use{a, -1});
        win.emplace(kb, Use{b, -1});
      }
      // keep the clouds of the window's frames that are held; the other frames go to empty slots first, then to new
      // clouds while the worker is below cap, then to the least recently used slots this window does not use
      res.stamp++;
      std::vector<char> taken(res.clouds.size(), 0);
      long long found = 0;
      for (size_t s = 0; s < res.clouds.size(); s++) {
        auto it = res.held[s] ? win.find(res.key[s]) : win.end();
        if (it != win.end()) {
          it->second.slot = (int)s;
          taken[s] = 1;
          res.used[s] = res.stamp;
          found++;
        }
      }
      buildRaws.clear();
      buildClouds.clear();
      fresh.clear();
      for (auto &fr : win) {
        if (fr.second.slot >= 0) continue;
        size_t s = 0;
        while (s < res.clouds.size() && (taken[s] || res.held[s])) s++;
        if (s == res.clouds.size() && res.clouds.size() < cap) {
          nicp_cloud *c = nullptr;
          int rc = nicp_cloud_create(w.ctx, (int)px, &c);
          if (rc) return rc;
          res.clouds.push_back(c);
          res.held.push_back(0);
          res.key.push_back(0);
          res.used.push_back(0);
          taken.push_back(0);
        }
        if (s == res.clouds.size()) {
          s = SIZE_MAX;
          for (size_t t = 0; t < res.clouds.size(); t++)
            if (!taken[t] && (s == SIZE_MAX || res.used[t] < res.used[s])) s = t;
        }
        // the slot claims its new frame only once the window that builds it has been aligned
        taken[s] = 1;
        res.held[s] = 0;
        fr.second.slot = (int)s;
        fresh.emplace_back((int)s, fr.first);
        for (int c = 0; c < nc; c++) buildRaws.push_back(raws[(size_t)fr.second.frame * nc + c]);
        buildClouds.push_back(res.clouds[s]);
      }
      int rc;
      if (!buildClouds.empty() &&
          (rc = prep_frames(w.ctx, fs, (int)buildClouds.size(), buildRaws.data(), sp, sensor_offset, 0, buildClouds.data())))
        return rc;
      const int m = (int)(j - i);
      refs.resize(m);
      curs.resize(m);
      for (int k = 0; k < m; k++) {
        refs[k] = res.clouds[win[keyOf(reference_frame[i + k])].slot];
        curs[k] = res.clouds[win[keyOf(current_frame[i + k])].slot];
      }
      // the window's priors, with prior_offsets rebased to its first pair
      const nicp_prior *wp = nullptr;
      if (prior_offsets) {
        offs.resize(m + 1);
        for (int k = 0; k <= m; k++) offs[k] = prior_offsets[i + k] - prior_offsets[i];
        if (priors) wp = priors + prior_offsets[i];
      }
      if ((rc = align_frame_pairs(w.ctx, fs, m, refs.data(), curs.data(), ap, sensor_offset, sensor_offset,
                                  initial_guesses ? initial_guesses + 16 * i : nullptr, wp,
                                  prior_offsets ? offs.data() : nullptr, frame_inlier_depth_threshold, results + i)))
        return rc;
      for (auto &sk : fresh) {
        res.held[sk.first] = 1;
        res.key[sk.first] = sk.second;
        res.used[sk.first] = res.stamp;
      }
      res.built += (long long)fresh.size();
      res.reused += found;
      i = j;
    }
    return NICP_OK;
  };

  const int G = (int)pool->workers.size();
  auto work = [&](int g) {
    nicp_shard_pool::Worker &w = pool->workers[g];
    const long long lo = (long long)g * n_pairs / G, hi = (long long)(g + 1) * n_pairs / G;
    Residency &res = store ? store->res[g] : w.calls;
    if (!store) {  // the frame indices name other frames in every call
      if (res.px != px) {  // another image size: the cache starts over, so it never holds more than cap
        res.release();
        res.px = px;
      }
      std::fill(res.held.begin(), res.held.end(), 0);
    }
    w.rc = hi > lo ? align_block(w, res, lo, hi) : NICP_OK;
    w.error = w.rc ? nicp_last_error() : "";  // this worker thread's message
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

static int store_create(nicp_shard_pool *pool, const FrameSet &fs, const nicp_stats_params *sp,
                        const float sensor_offset[16], nicp_frame_store **out) {
  nicp_frame_store *st = new nicp_frame_store();
  st->pool = pool;
  st->fs = fs;
  st->sp = *sp;
  st->hasOffset = sensor_offset != nullptr;
  if (sensor_offset) memcpy(st->sensorOffset, sensor_offset, sizeof st->sensorOffset);
  st->res.resize(pool->workers.size());
  for (Residency &r : st->res) r.px = (size_t)fs.proj.rows * fs.proj.cols;
  pool->stores.push_back(st);
  *out = st;
  return NICP_OK;
}

// NICP_ERR_INVALID (with a message) for a null store or one whose pool is gone
static int store_usable(const nicp_frame_store *st) {
  if (!st) return NICP_ERR_INVALID;
  if (!st->pool) {
    set_error("the frame store's shard pool has been destroyed: only nicp_frame_store_destroy may be called");
    return NICP_ERR_INVALID;
  }
  return NICP_OK;
}

static void store_release(nicp_frame_store *st) {
  for (Residency &r : st->res) r.release();
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
  pool->frameCap = (v && *v) ? std::max(2, atoi(v)) : 0;
  *out = pool;
  return NICP_OK;
}

void nicp_shard_pool_destroy(nicp_shard_pool *pool) {
  if (!pool) return;
  for (nicp_frame_store *st : pool->stores) {
    store_release(st);
    st->pool = nullptr;
  }
  for (nicp_shard_pool::Worker &w : pool->workers) {
    w.calls.release();
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
  FrameSet fs;
  int rc = frames_pinhole(proj, raw_rows, raw_cols, depth_scale, step, max_depth_cov, fs);
  return rc ? rc
            : align_frames_sharded(pool, nullptr, nullptr, fs, n_frames, raws, sp, sensor_offset, n_pairs, reference_frame,
                                   current_frame, initial_guesses, nullptr, nullptr, ap, frame_inlier_depth_threshold,
                                   results);
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
  FrameSet fs;
  int rc = frames_rig(mp, raw_rows, raw_cols, depth_scale, step, max_depth_cov, fs);
  return rc ? rc
            : align_frames_sharded(pool, nullptr, nullptr, fs, n_frames, raws, sp, sensor_offset, n_pairs, reference_frame,
                                   current_frame, initial_guesses, priors, prior_offsets, ap, frame_inlier_depth_threshold,
                                   results);
}

int nicp_frame_store_create(nicp_shard_pool *pool, int raw_rows, int raw_cols, float depth_scale, int step,
                            float max_depth_cov, const nicp_projector *proj, const nicp_stats_params *sp,
                            const float sensor_offset[16], nicp_frame_store **store) {
  if (!store) return NICP_ERR_INVALID;
  *store = nullptr;
  if (!pool || !proj || !sp || raw_rows <= 0 || raw_cols <= 0) return NICP_ERR_INVALID;
  FrameSet fs;
  int rc = frames_pinhole(proj, raw_rows, raw_cols, depth_scale, step, max_depth_cov, fs);
  return rc ? rc : store_create(pool, fs, sp, sensor_offset, store);
}

int nicp_multi_frame_store_create(nicp_shard_pool *pool, const int *raw_rows, const int *raw_cols, float depth_scale,
                                  int step, float max_depth_cov, const nicp_multi_projector *mp,
                                  const nicp_stats_params *sp, const float sensor_offset[16], nicp_frame_store **store) {
  if (!store) return NICP_ERR_INVALID;
  *store = nullptr;
  if (!pool || !mp || !sp) return NICP_ERR_INVALID;
  FrameSet fs;
  int rc = frames_rig(mp, raw_rows, raw_cols, depth_scale, step, max_depth_cov, fs);
  return rc ? rc : store_create(pool, fs, sp, sensor_offset, store);
}

void nicp_frame_store_destroy(nicp_frame_store *store) {
  if (!store) return;
  if (store->pool) {
    std::vector<nicp_frame_store *> &v = store->pool->stores;
    v.erase(std::remove(v.begin(), v.end(), store), v.end());
    store_release(store);
  }
  delete store;
}

int nicp_frame_store_add(nicp_frame_store *store, int n, const long long *ids, const uint16_t *const *raws) {
  int rc;
  if ((rc = store_usable(store))) return rc;
  if (n < 0) return NICP_ERR_INVALID;
  if (n == 0) return NICP_OK;
  if (!ids || !raws) return NICP_ERR_INVALID;
  const FrameSet &fs = store->fs;
  const int nc = fs.cams.n;
  std::unordered_set<long long> seen;
  for (int f = 0; f < n; f++) {
    if (store->raws.count(ids[f]) || !seen.insert(ids[f]).second) {
      set_error(store->raws.count(ids[f]) ? "frame id %lld is already in the store" : "frame id %lld is added twice",
                ids[f]);
      return NICP_ERR_INVALID;
    }
    for (int i = 0; i < nc; i++)
      if (!raws[(size_t)f * nc + i]) {
        set_error("null raw image of camera %d in frame %d", i, f);
        return NICP_ERR_INVALID;
      }
  }
  for (int f = 0; f < n; f++) {
    std::vector<uint16_t> &copy = store->raws[ids[f]];
    copy.resize(fs.rawPixels);
    uint16_t *dst = copy.data();
    for (int i = 0; i < nc; i++) {
      const size_t cpx = (size_t)fs.rawRows[i] * fs.rawCols[i];
      memcpy(dst, raws[(size_t)f * nc + i], cpx * sizeof(uint16_t));
      dst += cpx;
    }
  }
  return NICP_OK;
}

int nicp_frame_store_remove(nicp_frame_store *store, int n, const long long *ids) {
  int rc;
  if ((rc = store_usable(store))) return rc;
  if (n < 0) return NICP_ERR_INVALID;
  if (n == 0) return NICP_OK;
  if (!ids) return NICP_ERR_INVALID;
  std::unordered_set<long long> seen;
  for (int f = 0; f < n; f++)
    if (!store->raws.count(ids[f]) || !seen.insert(ids[f]).second) {
      set_error(store->raws.count(ids[f]) ? "frame id %lld is removed twice" : "frame id %lld is not in the store", ids[f]);
      return NICP_ERR_INVALID;
    }
  for (int f = 0; f < n; f++) {
    store->raws.erase(ids[f]);
    for (Residency &r : store->res) r.drop(ids[f]);
  }
  return NICP_OK;
}

int nicp_frame_store_size(const nicp_frame_store *store) {
  return store_usable(store) ? -1 : (int)store->raws.size();
}

int nicp_frame_store_align(nicp_frame_store *store, int n_pairs, const long long *reference_ids,
                           const long long *current_ids, const float *initial_guesses, const nicp_prior *priors,
                           const int *prior_offsets, const nicp_align_params *ap, float frame_inlier_depth_threshold,
                           nicp_align_result *results) {
  int rc;
  if ((rc = store_usable(store))) return rc;
  if (n_pairs < 0 || !ap) return NICP_ERR_INVALID;
  if (n_pairs == 0) return NICP_OK;
  if (!reference_ids || !current_ids || !results) return NICP_ERR_INVALID;
  // the call's frames: the distinct ids in order of first use, named by their index as in the sharded entries
  const int nc = store->fs.cams.n;
  std::unordered_map<long long, int> frameOf;
  std::vector<long long> keys;
  std::vector<const uint16_t *> raws;
  std::vector<int> refFrame(n_pairs), curFrame(n_pairs);
  for (int i = 0; i < n_pairs; i++)
    for (int side = 0; side < 2; side++) {
      const long long id = side ? current_ids[i] : reference_ids[i];
      auto it = frameOf.find(id);
      if (it == frameOf.end()) {
        auto fr = store->raws.find(id);
        if (fr == store->raws.end()) {
          set_error("pair %d references frame id %lld, which is not in the store", i, id);
          return NICP_ERR_INVALID;
        }
        it = frameOf.emplace(id, (int)keys.size()).first;
        keys.push_back(id);
        const uint16_t *p = fr->second.data();
        for (int c = 0; c < nc; c++) {
          raws.push_back(p);
          p += (size_t)store->fs.rawRows[c] * store->fs.rawCols[c];
        }
      }
      (side ? curFrame : refFrame)[i] = it->second;
    }
  return align_frames_sharded(store->pool, store, keys.data(), store->fs, (int)keys.size(), raws.data(), &store->sp,
                              store->hasOffset ? store->sensorOffset : nullptr, n_pairs, refFrame.data(), curFrame.data(),
                              initial_guesses, priors, prior_offsets, ap, frame_inlier_depth_threshold, results);
}

int nicp_frame_store_counters(const nicp_frame_store *store, long long *frames_built, long long *frames_reused) {
  int rc;
  if ((rc = store_usable(store))) return rc;
  long long b = 0, r = 0;
  for (const Residency &res : store->res) {
    b += res.built;
    r += res.reused;
  }
  if (frames_built) *frames_built = b;
  if (frames_reused) *frames_reused = r;
  return NICP_OK;
}

}  // extern "C"

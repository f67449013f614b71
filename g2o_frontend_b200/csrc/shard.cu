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
//
// A tracker (nicp_tracker_*) runs SequentialTracker::processFrame (include/pwn/tracker.h) for many independent sequences:
// each sequence stays on one worker with its keyframe and current cloud, and a step is one batched prep and one batched
// alignment per worker, the pose bookkeeping being done in the calling thread once every worker has succeeded.
#include <algorithm>
#include <chrono>
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
  std::vector<nicp_tracker *> trackers;    // likewise
  std::vector<nicp_scene_tracker *> sceneTrackers;  // likewise
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

// The state of one sequence of a tracker: SequentialTracker's members (include/pwn/tracker.h), with the keyframe cloud and
// the cloud the next frame is prepared into living on the sequence's worker.
struct TrackSeq {
  int worker;
  nicp_cloud *key, *cur;
  bool hasKey;                  // SequentialTracker::_previousCloud != 0
  float globalT[16], keyT[16];  // _globalT, _previousCloudTransform (column-major)
  int counter, numKeyframes;
};

struct nicp_tracker {
  nicp_shard_pool *pool;  // null once the pool has been destroyed
  nicp::FrameSet fs;
  nicp_stats_params sp;
  nicp_align_params ap;
  float imgThr, newFrameInliersFraction;
  float sensorOffset[16];
  bool hasOffset;
  std::vector<TrackSeq> seqs;
};

// The state of one sequence of a scene tracker: the loop variables of pwn_aligner.cpp:129-222 (the localmap mode of
// host/pwn_simple_aligner.cpp), with the local map, the cloud the next frame is prepared into and the subscene rendered
// from the map living on the sequence's worker.
struct SceneSeq {
  int worker;
  nicp_cloud *map, *frame, *sub;
  float globalT[16], sceneT[16];  // column-major
  int frames;                     // frames processed since create / reset (0: the next one is the driver's firstDepth)
  int counter;                    // the driver's chunk counter
  int mapPoints;                  // host mirror of the map's count
  bool broken;                    // a step failed on the device after it had started changing this map: reset first
};

struct nicp_scene_tracker {
  nicp_shard_pool *pool;  // null once the pool has been destroyed
  nicp::FrameSet fs;
  nicp_stats_params sp;
  nicp_align_params ap;
  nicp_merge_params mp;
  float imgThr, baseline, alpha;
  float sensorOffset[16];
  int chunkStep, mapCapacity;
  std::vector<SceneSeq> seqs;
  double phaseMs[2];  // host time of phase 1 (prep, render, align) and phase 2 (append, merge), summed over steps
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

// Runs work(g) for every worker of the pool, on one thread per worker when there are several; work sets the worker's rc
// and error.  Returns the first failing worker's status, with its message, or NICP_OK.
template <typename Work>
static int run_workers(nicp_shard_pool *pool, Work &&work) {
  const int G = (int)pool->workers.size();
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

// body() on worker w's device, then a synchronisation of its context (no upload of the step may still be reading the
// caller's raw images when the call returns): the worker's rc and error
template <typename Body>
static void worker_step(nicp_shard_pool::Worker &w, Body &&body) {
  w.rc = body();
  if (w.rc) w.error = nicp_last_error();  // this worker thread's message
  const int sync = nicp_synchronize(w.ctx);
  if (!w.rc && sync) {
    w.rc = sync;
    w.error = nicp_last_error();
  }
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
  return run_workers(pool, work);
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

// ---- trackers -------------------------------------------------------------------------------------------------------------

// The pose bookkeeping of SequentialTracker::processFrame (include/pwn/tracker.h:64-91) after an alignment with relative
// transform T and `inliers` inliers, in float32 and in the operation order of include/pwn/compat.h: iso_mul / iso_inverse
// are Isometry3f::operator* / inverse(), the re-orthogonalisation is written with Matrix3f's product (a sum from 0.0f,
// column index ascending), operator*(float) and operator-.  Returns whether the new cloud becomes the keyframe.
static bool track_bookkeeping(TrackSeq &s, const float guess[16], const float T[16], int inliers, int pixels,
                              float newFrameInliersFraction) {
  if (inliers > 0)
    iso_mul(s.keyT, T, s.globalT);
  else
    iso_mul(s.globalT, guess, s.globalT);
  if (!(s.counter % 50)) {  // pwn_tracker.cpp:153-158: R -= 0.5 R (R^T R - I)
    float R[9], E[9], corr[9];
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) R[c * 3 + r] = NM4(s.globalT, r, c);
    for (int r = 0; r < 3; r++)
      for (int k = 0; k < 3; k++) {
        float acc = 0.0f;
        for (int c = 0; c < 3; c++) acc += R[r * 3 + c] * R[k * 3 + c];  // R^T(r, c) * R(c, k)
        E[k * 3 + r] = acc;
      }
    for (int i = 0; i < 3; i++) E[i * 3 + i] -= 1.0f;
    for (int r = 0; r < 3; r++)
      for (int k = 0; k < 3; k++) {
        float acc = 0.0f;
        for (int c = 0; c < 3; c++) acc += R[c * 3 + r] * E[k * 3 + c];
        corr[k * 3 + r] = acc;
      }
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) NM4(s.globalT, r, c) = R[c * 3 + r] - corr[c * 3 + r] * 0.5f;
  }
  fix_last_row(s.globalT);
  return (float)inliers / (float)pixels < newFrameInliersFraction;
}

static void track_restart(TrackSeq &s) {
  s.hasKey = false;
  mat4_identity(s.globalT);
  mat4_identity(s.keyT);
  s.counter = s.numKeyframes = 0;
}

static void tracker_release(nicp_tracker *t) {
  for (TrackSeq &s : t->seqs) {
    nicp_cloud_destroy(s.key);
    nicp_cloud_destroy(s.cur);
    s.key = s.cur = nullptr;
  }
}

// NICP_ERR_INVALID (with a message) for a null tracker or one whose pool is gone
static int tracker_usable(const nicp_tracker *t) {
  if (!t) return NICP_ERR_INVALID;
  if (!t->pool) {
    set_error("the tracker's shard pool has been destroyed: only nicp_tracker_destroy may be called");
    return NICP_ERR_INVALID;
  }
  return NICP_OK;
}

// The placement of a tracker's S sequences: sequence s on worker floor(s G / S), for the tracker's lifetime.  Each sequence
// needs `units` clouds of px pixels on its worker (each named `each` in the message); NICP_ERR_INVALID when a worker's
// sequences need more than its frame cap.
static int place_sequences(const nicp_shard_pool *pool, int S, size_t px, long long units, const char *each,
                           std::vector<int> &worker) {
  const int G = (int)pool->workers.size();
  std::vector<int> onWorker(G, 0);
  worker.resize(S);
  for (int s = 0; s < S; s++) onWorker[worker[s] = (int)((long long)s * G / S)]++;
  for (int g = 0; g < G; g++) {
    const int cap = frame_cap(pool, pool->workers[g], px);
    if (units * onWorker[g] > cap) {
      set_error("worker %d (GPU %d) would hold %d sequences at %s each, more than its frame cap of %d clouds of "
                "%zu pixels (NICP_SHARD_FRAMES lowers the cap): use more workers or fewer sequences",
                g, pool->workers[g].device, onWorker[g], each, cap, px);
      return NICP_ERR_INVALID;
    }
  }
  return NICP_OK;
}

static int tracker_create(nicp_shard_pool *pool, int S, const FrameSet &fs, const nicp_stats_params *sp,
                          const float sensor_offset[16], const nicp_align_params *ap, float imgThr, float newFraction,
                          nicp_tracker **out) {
  const size_t px = (size_t)fs.proj.rows * fs.proj.cols;
  std::vector<int> worker;
  int rc;
  if ((rc = place_sequences(pool, S, px, 2, "two clouds", worker))) return rc;
  nicp_tracker *t = new nicp_tracker();
  t->pool = pool;
  t->fs = fs;
  t->sp = *sp;
  t->ap = *ap;
  t->imgThr = imgThr;
  t->newFrameInliersFraction = newFraction;
  t->hasOffset = sensor_offset != nullptr;
  if (sensor_offset) memcpy(t->sensorOffset, sensor_offset, sizeof t->sensorOffset);
  t->seqs.resize(S);
  for (int s = 0; s < S; s++) {
    TrackSeq &q = t->seqs[s];
    q.worker = worker[s];
    q.key = q.cur = nullptr;
    track_restart(q);
    nicp_context *ctx = pool->workers[q.worker].ctx;
    if ((rc = nicp_cloud_create(ctx, (int)px, &q.key)) || (rc = nicp_cloud_create(ctx, (int)px, &q.cur))) {
      tracker_release(t);
      delete t;
      return rc;
    }
  }
  pool->trackers.push_back(t);
  *out = t;
  return NICP_OK;
}

// n distinct sequences in [0, S)
static int check_sequences(int S, int n, const int *sequences) {
  std::vector<char> seen(S, 0);
  for (int k = 0; k < n; k++) {
    const int s = sequences[k];
    if (s < 0 || s >= S) {
      set_error("entry %d names sequence %d outside [0, %d)", k, s, S);
      return NICP_ERR_INVALID;
    }
    if (seen[s]) {
      set_error("sequence %d is listed twice", s);
      return NICP_ERR_INVALID;
    }
    seen[s] = 1;
  }
  return NICP_OK;
}

// ---- scene trackers -------------------------------------------------------------------------------------------------------

static void scene_restart(SceneSeq &s, const float *pose) {
  if (pose) {
    memcpy(s.globalT, pose, sizeof s.globalT);
    fix_last_row(s.globalT);
  } else {
    mat4_identity(s.globalT);
  }
  memcpy(s.sceneT, s.globalT, sizeof s.sceneT);
  s.frames = s.counter = s.mapPoints = 0;
  s.broken = false;
}

static void scene_release(nicp_scene_tracker *t) {
  for (SceneSeq &s : t->seqs) {
    nicp_cloud_destroy(s.map);
    nicp_cloud_destroy(s.frame);
    nicp_cloud_destroy(s.sub);
    s.map = s.frame = s.sub = nullptr;
  }
}

// NICP_ERR_INVALID (with a message) for a null scene tracker or one whose pool is gone
static int scene_usable(const nicp_scene_tracker *t) {
  if (!t) return NICP_ERR_INVALID;
  if (!t->pool) {
    set_error("the scene tracker's shard pool has been destroyed: only nicp_scene_tracker_destroy may be called");
    return NICP_ERR_INVALID;
  }
  return NICP_OK;
}

// the frame caps count a sequence's map as its bytes in units of a frame cloud: 112 B per pixel (frame_cap), and 100 B of
// gaussian and flag per point on top for the frame cloud and the map.  A map costs 80 B per point for its record, not
// frame_cap's 112: it is never aligned, so it gets no interleaved point / normal copy (ensure_pn), and the merge and the
// render project it with k_project_single / k_render_maps_z, which read the float4 points, not the packed copy
// (ensure_points3).  The frame cloud and the subscene are aligned and get the copies.
static long long scene_units(size_t px, int mapCapacity) {
  const size_t unit = 112 * px;
  const size_t bytes = (112 + 100) * px + 112 * px + (size_t)(80 + 100) * (size_t)mapCapacity;
  return (long long)((bytes + unit - 1) / unit);
}

// a * b as Isometry3f * Isometry3f (include/pwn/compat.h), last row rewritten
static void scene_mul(const float *a, const float *b, float *out) {
  iso_mul(a, b, out);
  fix_last_row(out);
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
  for (nicp_tracker *t : pool->trackers) {
    tracker_release(t);
    t->pool = nullptr;
  }
  for (nicp_scene_tracker *t : pool->sceneTrackers) {
    scene_release(t);
    t->pool = nullptr;
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

int nicp_tracker_create(nicp_shard_pool *pool, int n_sequences, int raw_rows, int raw_cols, float depth_scale, int step,
                        float max_depth_cov, const nicp_projector *proj, const nicp_stats_params *sp,
                        const float sensor_offset[16], const nicp_align_params *ap, float frame_inlier_depth_threshold,
                        float new_frame_inliers_fraction, nicp_tracker **tracker) {
  if (!tracker) return NICP_ERR_INVALID;
  *tracker = nullptr;
  if (!pool || !proj || !sp || !ap || raw_rows <= 0 || raw_cols <= 0 || n_sequences <= 0) return NICP_ERR_INVALID;
  FrameSet fs;
  int rc = frames_pinhole(proj, raw_rows, raw_cols, depth_scale, step, max_depth_cov, fs);
  return rc ? rc
            : tracker_create(pool, n_sequences, fs, sp, sensor_offset, ap, frame_inlier_depth_threshold,
                             new_frame_inliers_fraction, tracker);
}

int nicp_multi_tracker_create(nicp_shard_pool *pool, int n_sequences, const int *raw_rows, const int *raw_cols,
                              float depth_scale, int step, float max_depth_cov, const nicp_multi_projector *mp,
                              const nicp_stats_params *sp, const float sensor_offset[16], const nicp_align_params *ap,
                              float frame_inlier_depth_threshold, float new_frame_inliers_fraction, nicp_tracker **tracker) {
  if (!tracker) return NICP_ERR_INVALID;
  *tracker = nullptr;
  if (!pool || !mp || !sp || !ap || n_sequences <= 0) return NICP_ERR_INVALID;
  FrameSet fs;
  int rc = frames_rig(mp, raw_rows, raw_cols, depth_scale, step, max_depth_cov, fs);
  return rc ? rc
            : tracker_create(pool, n_sequences, fs, sp, sensor_offset, ap, frame_inlier_depth_threshold,
                             new_frame_inliers_fraction, tracker);
}

void nicp_tracker_destroy(nicp_tracker *tracker) {
  if (!tracker) return;
  if (tracker->pool) {
    std::vector<nicp_tracker *> &v = tracker->pool->trackers;
    v.erase(std::remove(v.begin(), v.end(), tracker), v.end());
    tracker_release(tracker);
  }
  delete tracker;
}

int nicp_tracker_size(const nicp_tracker *tracker) {
  return tracker_usable(tracker) ? -1 : (int)tracker->seqs.size();
}

int nicp_tracker_reset(nicp_tracker *tracker, int n, const int *sequences) {
  int rc;
  if ((rc = tracker_usable(tracker))) return rc;
  if (n < 0) return NICP_ERR_INVALID;
  if (n == 0) return NICP_OK;
  if (!sequences) return NICP_ERR_INVALID;
  if ((rc = check_sequences((int)tracker->seqs.size(), n, sequences))) return rc;
  for (int k = 0; k < n; k++) track_restart(tracker->seqs[sequences[k]]);
  return NICP_OK;
}

int nicp_tracker_step(nicp_tracker *tracker, int n, const int *sequences, const uint16_t *const *raws,
                      const float *odometry, nicp_track_result *results) {
  int rc;
  if ((rc = tracker_usable(tracker))) return rc;
  if (n < 0) return NICP_ERR_INVALID;
  if (n == 0) return NICP_OK;
  if (!sequences || !raws || !results) return NICP_ERR_INVALID;
  if ((rc = check_sequences((int)tracker->seqs.size(), n, sequences))) return rc;
  const FrameSet &fs = tracker->fs;
  const int nc = fs.cams.n;
  for (int k = 0; k < n; k++)
    for (int i = 0; i < nc; i++)
      if (!raws[(size_t)k * nc + i]) {
        set_error("null raw image of camera %d in entry %d (sequence %d)", i, k, sequences[k]);
        return NICP_ERR_INVALID;
      }
  nicp_shard_pool *pool = tracker->pool;
  const float *so = tracker->hasOffset ? tracker->sensorOffset : nullptr;

  // guess = keyT^-1 * globalT * odometry, from the committed state (SequentialTracker::processFrame, tracker.h:64-65)
  std::vector<float> guesses((size_t)16 * n);
  float eye[16];
  mat4_identity(eye);
  const int G = (int)pool->workers.size();
  std::vector<std::vector<int>> entries(G);  // entries of the step on worker g, in listed order
  for (int k = 0; k < n; k++) {
    const TrackSeq &s = tracker->seqs[sequences[k]];
    entries[s.worker].push_back(k);
    float *g = &guesses[(size_t)16 * k];
    if (!s.hasKey) {
      mat4_identity(g);
      continue;
    }
    iso_inverse(s.keyT, g);
    iso_mul(g, s.globalT, g);
    iso_mul(g, odometry ? odometry + (size_t)16 * k : eye, g);
    fix_last_row(g);  // Aligner::setInitialGuess
  }

  // every worker: one batched prep of its entries' frames, one batched alignment of those that have a keyframe
  std::vector<nicp_align_result> recs(n);
  auto work = [&](int g) {
    nicp_shard_pool::Worker &w = pool->workers[g];
    const std::vector<int> &mine = entries[g];
    w.rc = NICP_OK;
    w.error.clear();
    if (mine.empty()) return;
    auto body = [&]() -> int {
      NICP_CUDA(cudaSetDevice(w.device));
      std::vector<const uint16_t *> frameRaws;
      std::vector<nicp_cloud *> clouds;
      std::vector<const nicp_cloud *> refs, curs;
      std::vector<float> gs;
      std::vector<int> aligned;
      for (int k : mine) {
        const TrackSeq &s = tracker->seqs[sequences[k]];
        for (int i = 0; i < nc; i++) frameRaws.push_back(raws[(size_t)k * nc + i]);
        clouds.push_back(s.hasKey ? s.cur : s.key);
        if (s.hasKey) {
          refs.push_back(s.key);
          curs.push_back(s.cur);
          gs.insert(gs.end(), &guesses[(size_t)16 * k], &guesses[(size_t)16 * k] + 16);
          aligned.push_back(k);
        }
      }
      int rc;
      if ((rc = prep_frames(w.ctx, fs, (int)clouds.size(), frameRaws.data(), &tracker->sp, so, 0, clouds.data())))
        return rc;
      if (refs.empty()) return NICP_OK;
      std::vector<nicp_align_result> out(refs.size());
      if ((rc = align_frame_pairs(w.ctx, fs, (int)refs.size(), refs.data(), curs.data(), &tracker->ap, so, so, gs.data(),
                                  nullptr, nullptr, tracker->imgThr, out.data())))
        return rc;
      for (size_t i = 0; i < aligned.size(); i++) recs[aligned[i]] = out[i];
      return NICP_OK;
    };
    worker_step(w, body);
  };
  if ((rc = run_workers(pool, work))) return rc;
  for (int k = 0; k < n; k++)
    if (tracker->seqs[sequences[k]].hasKey && recs[k].status != NICP_OK) {
      set_error("entry %d (sequence %d): the alignment's record has status %d", k, sequences[k], recs[k].status);
      return recs[k].status;
    }

  // commit, in the calling thread
  const int pixels = fs.proj.rows * fs.proj.cols;
  for (int k = 0; k < n; k++) {
    TrackSeq &s = tracker->seqs[sequences[k]];
    nicp_track_result &r = results[k];
    memset(&r, 0, sizeof r);
    r.frame = s.counter;
    r.record.status = NICP_OK;
    if (!s.hasKey) {  // the first frame: its cloud is the keyframe
      s.hasKey = true;
      memcpy(s.keyT, s.globalT, sizeof s.keyT);
      s.numKeyframes++;
      r.keyframe = 1;
      mat4_identity(r.relative_T);
      mat4_identity(r.guess);
    } else {
      const float *guess = &guesses[(size_t)16 * k];
      r.aligned = 1;
      r.record = recs[k];
      memcpy(r.relative_T, recs[k].T, sizeof r.relative_T);
      memcpy(r.guess, guess, sizeof r.guess);
      if (track_bookkeeping(s, guess, recs[k].T, recs[k].inliers, pixels, tracker->newFrameInliersFraction)) {
        std::swap(s.key, s.cur);
        memcpy(s.keyT, s.globalT, sizeof s.keyT);
        s.numKeyframes++;
        r.keyframe = 1;
      }
    }
    s.counter++;
    memcpy(r.global_T, s.globalT, sizeof r.global_T);
    r.num_keyframes = s.numKeyframes;
  }
  return NICP_OK;
}

int nicp_scene_tracker_create(nicp_shard_pool *pool, int n_sequences, int raw_rows, int raw_cols, float depth_scale, int step,
                              float max_depth_cov, const nicp_projector *proj, const nicp_stats_params *sp,
                              const float sensor_offset[16], float baseline, float alpha, const nicp_align_params *ap,
                              float frame_inlier_depth_threshold, const nicp_merge_params *mp, int chunk_step,
                              int map_capacity, nicp_scene_tracker **tracker) {
  if (!tracker) return NICP_ERR_INVALID;
  *tracker = nullptr;
  if (!pool || !proj || !sp || !ap || !mp || raw_rows <= 0 || raw_cols <= 0 || n_sequences <= 0) return NICP_ERR_INVALID;
  if (chunk_step < 0 || map_capacity <= 0) {
    set_error("chunk_step %d must be >= 0 and map_capacity %d > 0", chunk_step, map_capacity);
    return NICP_ERR_INVALID;
  }
  FrameSet fs;
  int rc;
  if ((rc = frames_pinhole(proj, raw_rows, raw_cols, depth_scale, step, max_depth_cov, fs))) return rc;
  const size_t px = (size_t)fs.proj.rows * fs.proj.cols;
  const long long units = scene_units(px, map_capacity);
  char each[128];
  snprintf(each, sizeof each, "%lld clouds (frame, subscene and a map of %d points)", units, map_capacity);
  std::vector<int> worker;
  if ((rc = place_sequences(pool, n_sequences, px, units, each, worker))) return rc;
  nicp_scene_tracker *t = new nicp_scene_tracker();
  t->pool = pool;
  t->fs = fs;
  t->sp = *sp;
  t->ap = *ap;
  t->mp = *mp;
  t->imgThr = frame_inlier_depth_threshold;
  t->baseline = baseline;
  t->alpha = alpha;
  if (sensor_offset)
    memcpy(t->sensorOffset, sensor_offset, sizeof t->sensorOffset);
  else
    mat4_identity(t->sensorOffset);
  t->chunkStep = chunk_step;
  t->mapCapacity = map_capacity;
  t->phaseMs[0] = t->phaseMs[1] = 0.0;
  t->seqs.resize(n_sequences);
  for (int s = 0; s < n_sequences; s++) {
    SceneSeq &q = t->seqs[s];
    q.worker = worker[s];
    q.map = q.frame = q.sub = nullptr;
    scene_restart(q, nullptr);
    nicp_context *ctx = pool->workers[q.worker].ctx;
    if ((rc = nicp_cloud_create(ctx, map_capacity, &q.map)) || (rc = cloud_ensure_gaussians(ctx, q.map)) ||
        (rc = nicp_cloud_create(ctx, (int)px, &q.frame)) || (rc = cloud_ensure_gaussians(ctx, q.frame)) ||
        (rc = nicp_cloud_create(ctx, (int)px, &q.sub))) {
      scene_release(t);
      delete t;
      return rc;
    }
    q.map->has_gauss = true;  // an empty map with gaussians, as Cloud::add leaves it
  }
  pool->sceneTrackers.push_back(t);
  *tracker = t;
  return NICP_OK;
}

void nicp_scene_tracker_destroy(nicp_scene_tracker *tracker) {
  if (!tracker) return;
  if (tracker->pool) {
    std::vector<nicp_scene_tracker *> &v = tracker->pool->sceneTrackers;
    v.erase(std::remove(v.begin(), v.end(), tracker), v.end());
    scene_release(tracker);
  }
  delete tracker;
}

int nicp_scene_tracker_size(const nicp_scene_tracker *tracker) {
  return scene_usable(tracker) ? -1 : (int)tracker->seqs.size();
}

int nicp_scene_tracker_reset(nicp_scene_tracker *tracker, int n, const int *sequences, const float *initial_poses) {
  int rc;
  if ((rc = scene_usable(tracker))) return rc;
  if (n < 0) return NICP_ERR_INVALID;
  if (n == 0) return NICP_OK;
  if (!sequences) return NICP_ERR_INVALID;
  if ((rc = check_sequences((int)tracker->seqs.size(), n, sequences))) return rc;
  // the map's device count is reset by the sequence's next step (it restarts the map)
  for (int k = 0; k < n; k++) scene_restart(tracker->seqs[sequences[k]], initial_poses ? initial_poses + 16 * (size_t)k : nullptr);
  return NICP_OK;
}

int nicp_scene_tracker_step(nicp_scene_tracker *tracker, int n, const int *sequences, const uint16_t *const *raws,
                            nicp_scene_track_result *results) {
  int rc;
  if ((rc = scene_usable(tracker))) return rc;
  if (n < 0) return NICP_ERR_INVALID;
  if (n == 0) return NICP_OK;
  if (!sequences || !raws || !results) return NICP_ERR_INVALID;
  if ((rc = check_sequences((int)tracker->seqs.size(), n, sequences))) return rc;
  for (int k = 0; k < n; k++) {
    if (!raws[k]) {
      set_error("null raw image in entry %d (sequence %d)", k, sequences[k]);
      return NICP_ERR_INVALID;
    }
    if (tracker->seqs[sequences[k]].broken) {
      set_error("sequence %d failed on the device in an earlier step: nicp_scene_tracker_reset it first", sequences[k]);
      return NICP_ERR_INVALID;
    }
  }
  nicp_shard_pool *pool = tracker->pool;
  const FrameSet &fs = tracker->fs;
  const float *so = tracker->sensorOffset;
  const int G = (int)pool->workers.size();
  std::vector<std::vector<int>> entries(G);  // entries of the step on worker g, in listed order
  std::vector<float> views((size_t)16 * n);  // KRt of the render view sceneT * sensorOffset (pwn_aligner.cpp:160)
  for (int k = 0; k < n; k++) {
    const SceneSeq &s = tracker->seqs[sequences[k]];
    entries[s.worker].push_back(k);
    float T[16];
    scene_mul(s.sceneT, so, T);
    compute_KRt(fs.proj.K, T, &views[(size_t)16 * k]);
  }
  using Clock = std::chrono::steady_clock;
  const Clock::time_point t0 = Clock::now();

  // phase 1, every worker: frames, gaussians, renders and subscenes in one batched prep, one batched alignment of the
  // sequences that have a map, the frames' point counts
  std::vector<nicp_align_result> recs(n);
  std::vector<int> framePoints(n, 0);
  auto phase1 = [&](int g) {
    nicp_shard_pool::Worker &w = pool->workers[g];
    const std::vector<int> &mine = entries[g];
    w.rc = NICP_OK;
    w.error.clear();
    if (mine.empty()) return;
    std::vector<int> counts(mine.size(), 0);  // written by the device before worker_step's synchronisation
    auto body = [&]() -> int {
      NICP_CUDA(cudaSetDevice(w.device));
      const size_t m = mine.size();
      std::vector<const uint16_t *> frameRaws(m);
      std::vector<nicp_cloud *> frames(m), subs(m);
      std::vector<const nicp_cloud *> maps(m), refs, curs;
      std::vector<int> mapPoints(m);
      std::vector<float> mv((size_t)16 * m);
      std::vector<int> aligned;
      for (size_t i = 0; i < m; i++) {
        const int k = mine[i];
        const SceneSeq &s = tracker->seqs[sequences[k]];
        frameRaws[i] = raws[k];
        frames[i] = s.frame;
        subs[i] = s.sub;
        maps[i] = s.frames > 0 ? s.map : nullptr;
        mapPoints[i] = s.mapPoints;
        memcpy(&mv[16 * i], &views[(size_t)16 * k], 16 * sizeof(float));
        if (s.frames > 0) {
          refs.push_back(s.sub);
          curs.push_back(s.frame);
          aligned.push_back(k);
        }
      }
      int rc;
      if ((rc = prep_scene_frames(w.ctx, fs, (int)m, frameRaws.data(), &tracker->sp, so, tracker->baseline, tracker->alpha,
                                  frames.data(), maps.data(), mapPoints.data(), mv.data(), subs.data())))
        return rc;
      if (!refs.empty()) {
        std::vector<nicp_align_result> out(refs.size());
        if ((rc = align_frame_pairs(w.ctx, fs, (int)refs.size(), refs.data(), curs.data(), &tracker->ap, so, so, nullptr,
                                    nullptr, nullptr, tracker->imgThr, out.data())))
          return rc;
        for (size_t i = 0; i < aligned.size(); i++) recs[aligned[i]] = out[i];
      }
      for (size_t i = 0; i < m; i++)
        NICP_CUDA(cudaMemcpyAsync(&counts[i], frames[i]->d_n, sizeof(int), cudaMemcpyDeviceToHost, w.ctx->stream));
      return NICP_OK;
    };
    worker_step(w, body);
    if (!w.rc)
      for (size_t i = 0; i < mine.size(); i++) framePoints[mine[i]] = counts[i];
  };
  if ((rc = run_workers(pool, phase1))) return rc;
  const Clock::time_point t1 = Clock::now();

  // between the phases, in the calling thread: tentative poses, chunk decisions (pwn_aligner.cpp:194-205) and capacities
  struct Next {
    float globalT[16], sceneT[16];
    int counter, newMap, base;  // base: the map's size before the append (0 when it restarts)
  };
  std::vector<Next> next(n);
  for (int k = 0; k < n; k++) {
    const SceneSeq &s = tracker->seqs[sequences[k]];
    Next &x = next[k];
    memcpy(x.globalT, s.globalT, sizeof x.globalT);
    memcpy(x.sceneT, s.sceneT, sizeof x.sceneT);
    x.counter = s.counter;
    x.newMap = 0;
    if (s.frames > 0) {
      if (recs[k].status != NICP_OK) {
        set_error("entry %d (sequence %d): the alignment's record has status %d", k, sequences[k], recs[k].status);
        return recs[k].status;
      }
      scene_mul(x.globalT, recs[k].T, x.globalT);
      scene_mul(x.sceneT, recs[k].T, x.sceneT);
      if (tracker->chunkStep > 0 && x.counter++ % tracker->chunkStep == 0) {
        mat4_identity(x.sceneT);
        x.newMap = 1;
      }
    }
    x.base = (x.newMap || s.frames == 0) ? 0 : s.mapPoints;
    if ((long long)x.base + framePoints[k] > tracker->mapCapacity) {
      set_error("entry %d (sequence %d): %d map points + %d frame points exceed the map capacity %d", k, sequences[k], x.base,
                framePoints[k], tracker->mapCapacity);
      return NICP_ERR_INVALID;
    }
  }

  // phase 2, every worker: restarting maps emptied, one append launch, the merges
  std::vector<int> merged(n, 0);
  auto phase2 = [&](int g) {
    nicp_shard_pool::Worker &w = pool->workers[g];
    const std::vector<int> &mine = entries[g];
    w.rc = NICP_OK;
    w.error.clear();
    if (mine.empty()) return;
    auto body = [&]() -> int {
      NICP_CUDA(cudaSetDevice(w.device));
      const size_t m = mine.size();
      std::vector<nicp_cloud *> frames(m), maps(m);
      std::vector<float> poses((size_t)16 * m);
      std::vector<int> fp(m), base(m);
      for (size_t i = 0; i < m; i++) {
        const int k = mine[i];
        const SceneSeq &s = tracker->seqs[sequences[k]];
        frames[i] = s.frame;
        maps[i] = s.map;
        memcpy(&poses[16 * i], next[k].sceneT, sizeof next[k].sceneT);
        fp[i] = framePoints[k];
        base[i] = next[k].base;
        if (!base[i]) NICP_CUDA(cudaMemsetAsync(s.map->d_n, 0, sizeof(int), w.ctx->stream));
      }
      int rc;
      if ((rc = launch_scene_append(w.ctx, (int)m, frames.data(), maps.data(), poses.data(), fp.data(), base.data())))
        return rc;
      for (size_t i = 0; i < m; i++) {
        const int k = mine[i];
        const int size = base[i] + fp[i];
        if (!size) continue;  // nicp_merge leaves an empty map as it is
        float T[16];
        scene_mul(next[k].sceneT, so, T);  // Merger::merge(map, sceneT * sensorOffset), pwn_aligner.cpp:207
        if ((rc = run_merge(w.ctx, maps[i], &fs.proj, T, &tracker->mp, size, nullptr, &merged[k]))) return rc;
      }
      return NICP_OK;
    };
    worker_step(w, body);
  };
  rc = run_workers(pool, phase2);
  const Clock::time_point t2 = Clock::now();
  tracker->phaseMs[0] += std::chrono::duration<double, std::milli>(t1 - t0).count();
  tracker->phaseMs[1] += std::chrono::duration<double, std::milli>(t2 - t1).count();
  if (rc) {
    for (int k = 0; k < n; k++) tracker->seqs[sequences[k]].broken = true;
    return rc;
  }

  // commit, in the calling thread
  for (int k = 0; k < n; k++) {
    SceneSeq &s = tracker->seqs[sequences[k]];
    const Next &x = next[k];
    nicp_scene_track_result &r = results[k];
    memset(&r, 0, sizeof r);
    r.frame = s.frames;
    r.record.status = NICP_OK;
    if (s.frames > 0) {
      r.aligned = 1;
      r.record = recs[k];
    }
    memcpy(s.globalT, x.globalT, sizeof s.globalT);
    memcpy(s.sceneT, x.sceneT, sizeof s.sceneT);
    s.counter = x.counter;
    s.mapPoints = merged[k];
    s.frames++;
    memcpy(r.global_T, s.globalT, sizeof r.global_T);
    memcpy(r.scene_T, s.sceneT, sizeof r.scene_T);
    r.new_map = x.newMap;
    r.added = x.base + framePoints[k];
    r.map_points = s.mapPoints;
  }
  return NICP_OK;
}

int nicp_scene_tracker_download_map(nicp_scene_tracker *tracker, int sequence, int capacity, float *points4, float *normals4,
                                    float *curvature, float *omega_p6, float *omega_n6, float *gauss24, int *gflags, int *n) {
  int rc;
  if ((rc = scene_usable(tracker))) return rc;
  if (sequence < 0 || sequence >= (int)tracker->seqs.size()) {
    set_error("sequence %d outside [0, %d)", sequence, (int)tracker->seqs.size());
    return NICP_ERR_INVALID;
  }
  const SceneSeq &s = tracker->seqs[sequence];
  if (s.broken) {
    set_error("sequence %d failed on the device in an earlier step: its map is undefined until nicp_scene_tracker_reset",
              sequence);
    return NICP_ERR_INVALID;
  }
  if (n) *n = s.mapPoints;
  if (capacity < s.mapPoints) {
    set_error("the map of sequence %d holds %d points, more than the capacity %d", sequence, s.mapPoints, capacity);
    return NICP_ERR_INVALID;
  }
  if (!s.mapPoints) return NICP_OK;
  nicp_context *ctx = tracker->pool->workers[s.worker].ctx;
  if ((rc = nicp_cloud_download(ctx, s.map, points4, normals4, curvature, omega_p6, omega_n6))) return rc;
  if ((gauss24 || gflags) && (rc = nicp_cloud_download_gaussians(ctx, s.map, gauss24, gflags))) return rc;
  return NICP_OK;
}

int nicp_scene_tracker_phase_ms(const nicp_scene_tracker *tracker, double *phase1_ms, double *phase2_ms) {
  int rc;
  if ((rc = scene_usable(tracker))) return rc;
  if (phase1_ms) *phase1_ms = tracker->phaseMs[0];
  if (phase2_ms) *phase2_ms = tracker->phaseMs[1];
  return NICP_OK;
}

}  // extern "C"

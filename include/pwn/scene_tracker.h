// pwn/scene_tracker.h -- scene-based odometry of many independent depth sequences at once, over the C-ABI scene tracker
// (nicp_scene_tracker_*, include/nicp_b200.h).
//
// pwn::BatchSceneTracker runs the mapping loop of pwn_core/pwn_aligner.cpp:129-222 (the localmap mode of
// host/pwn_simple_aligner.cpp) for S sequences: processFrames takes one frame of each listed sequence, aligns it against
// the sequence's local map re-rendered at sceneT * sensorOffset, adds it to the map (Cloud::add) and merges it
// (Merger::merge); after the first alignment and then every chunkStep frames the map is closed and a new one starts
// (chunkStep 0: one map).  Each sequence's globalT, sceneT, inliers, added and map size are those of the driver's loop.  The
// sequences are spread over the GPUs of a device list (a shard pool), each keeping its map on its GPU.  Pinhole cameras
// only: the converter's projector must be a PinholePointProjector.
//
// The C-ABI tracker is created on the first processFrames call from the converter's statistics parameters and sensor model
// (its projector's baseline and alpha), the aligner's parameters (including its frame inlier depth threshold), the
// Merger's thresholds, the scale, the chunk step, the map capacity, the camera matrix, the sensor offset, the raw image size
// and the depth scale.  The camera is built as the driver builds it: setCameraMatrix(K), setImageSize(raw size),
// scale(1 / scale).  A later call whose camera matrix, sensor offset, raw size or depth scale differ, or after setScale /
// setChunkStep changed the values it was created with, throws.
#pragma once
#include <cstring>
#include <stdexcept>
#include <vector>

#include "pwn.h"

namespace pwn {

class BatchSceneTracker {
 public:
  // mapCapacity: points each sequence's map can hold (a frame that would overflow it makes processFrames throw before any
  // sequence changes)
  BatchSceneTracker(DepthImageConverterIntegralImage *converter, Aligner *aligner, Merger *merger,
                    const std::vector<int> &devices, int numSequences, int mapCapacity)
      : _converter(converter), _aligner(aligner), _merger(merger), _scale(1), _chunkStep(10), _mapCapacity(mapCapacity),
        _pool(0), _tracker(0), _seqs(numSequences > 0 ? numSequences : 0) {
    if (numSequences <= 0) throw std::runtime_error("BatchSceneTracker: needs at least one sequence");
    nicpCheck(nicp_shard_pool_create(devices.data(), (int)devices.size(), &_pool), "BatchSceneTracker: nicp_shard_pool_create");
  }
  ~BatchSceneTracker() {
    nicp_scene_tracker_destroy(_tracker);
    nicp_shard_pool_destroy(_pool);
  }
  void setScale(int scale_) { _scale = scale_; }              // the driver's imageScale
  void setChunkStep(int chunkStep_) { _chunkStep = chunkStep_; }  // the driver's chunkStep
  int numSequences() const { return (int)_seqs.size(); }
  const Isometry3f &globalT(int s) const { return _seqs.at(s).globalT; }
  const Isometry3f &sceneT(int s) const { return _seqs.at(s).sceneT; }
  int lastInliers(int s) const { return _seqs.at(s).last.record.inliers; }
  int lastAdded(int s) const { return _seqs.at(s).last.added; }       // map points after Cloud::add, before the merge
  int mapSize(int s) const { return _seqs.at(s).last.map_points; }   // map points after Merger::merge
  bool lastNewMap(int s) const { return _seqs.at(s).last.new_map != 0; }
  // the full result of sequence s's last frame (poses, counters, alignment record)
  const nicp_scene_track_result &lastResult(int s) const { return _seqs.at(s).last; }
  // the C-ABI tracker (null before the first processFrames): nicp_scene_tracker_download_map reads a sequence's map
  nicp_scene_tracker *handle() const { return _tracker; }

  // sequence s starts over with an empty map and globalT = sceneT = initialT (the driver's initialT)
  void reset(int s, const Isometry3f &initialT = Isometry3f::Identity()) {
    Seq &q = _seqs.at(s);
    q.globalT = q.sceneT = initialT;
    std::memset(&q.last, 0, sizeof q.last);
    if (_tracker) nicpCheck(nicp_scene_tracker_reset(_tracker, 1, &s, initialT.data()), "BatchSceneTracker::reset");
  }

  // one iteration of the driver's loop for raws[k] of sequence sequences[k], every k (distinct sequences)
  void processFrames(const std::vector<int> &sequences, const std::vector<const RawDepthImage *> &raws,
                     const Isometry3f &sensorOffset, const Matrix3f &cameraMatrix, float depthScale = 0.001f) {
    const size_t n = sequences.size();
    if (raws.size() != n) throw std::runtime_error("BatchSceneTracker::processFrames: one raw image per sequence");
    if (n == 0) return;
    for (size_t k = 0; k < n; k++)
      if (!raws[k] || raws[k]->rows != raws[0]->rows || raws[k]->cols != raws[0]->cols)
        throw std::runtime_error("BatchSceneTracker::processFrames: every raw image must have the same size");
    ensureTracker(*raws[0], sensorOffset, cameraMatrix, depthScale);
    std::vector<const uint16_t *> ptrs(n);
    for (size_t k = 0; k < n; k++) ptrs[k] = raws[k]->data();
    std::vector<nicp_scene_track_result> results(n);
    nicpCheck(nicp_scene_tracker_step(_tracker, (int)n, sequences.data(), ptrs.data(), results.data()),
              "BatchSceneTracker::processFrames");
    for (size_t k = 0; k < n; k++) {
      Seq &s = _seqs[sequences[k]];
      const nicp_scene_track_result &r = results[k];
      std::memcpy(s.globalT.data(), r.global_T, sizeof r.global_T);
      std::memcpy(s.sceneT.data(), r.scene_T, sizeof r.scene_T);
      s.last = r;
    }
  }

 protected:
  struct Seq {
    Isometry3f globalT, sceneT;
    nicp_scene_track_result last;
    Seq() { std::memset(&last, 0, sizeof last); }
  };
  // Aligner keeps PwnMatcherBase's frame inlier depth threshold protected: read it through a derived class's member pointer
  struct AlignerThreshold : Aligner {
    static float of(const Aligner &a) { return a.*(&AlignerThreshold::_frameInlierDepthThreshold); }
  };

  // the driver's scaled camera and Merger image size (pwn_simple_aligner.cpp localmap: setCameraMatrix, setImageSize,
  // scale(1 / imageScale)); the C-ABI tracker on the first call, then the sequences' pending initial poses
  void ensureTracker(const RawDepthImage &raw, const Isometry3f &sensorOffset, const Matrix3f &cameraMatrix, float depthScale) {
    PinholePointProjector *projector = dynamic_cast<PinholePointProjector *>(_converter->projector());
    PinholePointProjector *alprojector = dynamic_cast<PinholePointProjector *>(_aligner->projector());
    if (!projector || !alprojector)
      throw std::runtime_error("BatchSceneTracker: the converter and the aligner need PinholePointProjectors");
    projector->setCameraMatrix(cameraMatrix);
    projector->setImageSize(raw.rows, raw.cols);
    projector->scale(1.0f / _scale);
    nicp_projector p = projector->abiProjector();
    if (alprojector->minDistance() != p.min_distance || alprojector->maxDistance() != p.max_distance)
      throw std::runtime_error("BatchSceneTracker: the aligner's projector needs the converter's distance range");
    _merger->setImageSize(p.rows, p.cols);
    Key key;
    std::memset(&key, 0, sizeof key);
    key.proj = p;
    key.rawRows = raw.rows;
    key.rawCols = raw.cols;
    key.scale = _scale;
    key.chunkStep = _chunkStep;
    key.depthScale = depthScale;
    std::memcpy(key.sensorOffset, sensorOffset.data(), sizeof key.sensorOffset);
    if (_tracker) {
      if (std::memcmp(&key, &_key, sizeof key))
        throw std::runtime_error("BatchSceneTracker: camera matrix, sensor offset, raw size, depth scale, scale and chunk "
                                 "step are fixed by the first processFrames call");
      return;
    }
    nicp_stats_params sp = _converter->abiStatsParams();
    nicp_align_params ap = _aligner->abiAlignParams();
    nicp_merge_params mp = {_merger->distanceThreshold(), _merger->normalThreshold(), _merger->maxPointDepth()};
    nicpCheck(nicp_scene_tracker_create(_pool, (int)_seqs.size(), raw.rows, raw.cols, depthScale, _scale, 0.01f, &p, &sp,
                                        sensorOffset.data(), projector->baseline(), projector->alpha(), &ap,
                                        AlignerThreshold::of(*_aligner), &mp, _chunkStep, _mapCapacity, &_tracker),
              "BatchSceneTracker: nicp_scene_tracker_create");
    _key = key;
    for (int s = 0; s < (int)_seqs.size(); s++)
      nicpCheck(nicp_scene_tracker_reset(_tracker, 1, &s, _seqs[s].globalT.data()), "BatchSceneTracker: initial pose");
  }

  struct Key {
    nicp_projector proj;
    int rawRows, rawCols, scale, chunkStep;
    float depthScale;
    float sensorOffset[16];
  };
  DepthImageConverterIntegralImage *_converter;
  Aligner *_aligner;
  Merger *_merger;
  int _scale, _chunkStep, _mapCapacity;
  nicp_shard_pool *_pool;
  nicp_scene_tracker *_tracker;
  Key _key;
  std::vector<Seq> _seqs;

 private:
  BatchSceneTracker(const BatchSceneTracker &);
  BatchSceneTracker &operator=(const BatchSceneTracker &);
};

}  // namespace pwn

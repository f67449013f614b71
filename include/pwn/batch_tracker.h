// pwn/batch_tracker.h -- keyframe tracking of many independent depth sequences at once, over the C-ABI tracker
// (nicp_tracker_*, include/nicp_b200.h).
//
// pwn::BatchTracker mirrors pwn::SequentialTracker (tracker.h) for S sequences: processFrames takes one frame of each
// listed sequence and leaves every sequence in the state SequentialTracker::processFrame would leave it in, bit for bit
// (globalT, lastRelative, lastInliers, numKeyframes, lastWasKeyframe).  The sequences are spread over the GPUs of a device
// list (a shard pool), each keeping its keyframe cloud on its GPU; a call is one batched prep and one batched alignment per
// GPU.  Like SequentialTracker, only pinhole cameras: the converter's projector must be a PinholePointProjector.
//
// The C-ABI tracker is created on the first processFrames call from the converter's statistics parameters, the aligner's
// parameters (including its frame inlier depth threshold), the scale, the keyframe fraction, the scaled camera matrix, the
// sensor offset, the raw image size and the depth scale.  A later call whose camera matrix, sensor offset, raw size or depth
// scale differ, or after setScale / setNewFrameInliersFraction changed the values it was created with, throws.
#pragma once
#include <cstring>
#include <stdexcept>
#include <vector>

#include "pwn.h"

namespace pwn {

class BatchTracker {
 public:
  BatchTracker(DepthImageConverterIntegralImage *converter, Aligner *aligner, const std::vector<int> &devices, int numSequences)
      : _converter(converter), _aligner(aligner), _scale(2), _newFrameInliersFraction(0.4f), _pool(0), _tracker(0),
        _seqs(numSequences > 0 ? numSequences : 0) {
    if (numSequences <= 0) throw std::runtime_error("BatchTracker: needs at least one sequence");
    nicpCheck(nicp_shard_pool_create(devices.data(), (int)devices.size(), &_pool), "BatchTracker: nicp_shard_pool_create");
  }
  ~BatchTracker() {
    nicp_tracker_destroy(_tracker);
    nicp_shard_pool_destroy(_pool);
  }
  void setScale(int scale_) { _scale = scale_; }                              // SequentialTracker::setScale
  void setNewFrameInliersFraction(float v) { _newFrameInliersFraction = v; }  // SequentialTracker::setNewFrameInliersFraction
  int numSequences() const { return (int)_seqs.size(); }
  const Isometry3f &globalT(int s) const { return _seqs.at(s).globalT; }
  int numKeyframes(int s) const { return _seqs.at(s).numKeyframes; }
  int lastInliers(int s) const { return _seqs.at(s).lastInliers; }
  bool lastWasKeyframe(int s) const { return _seqs.at(s).lastWasKeyframe; }
  const Isometry3f &lastRelative(int s) const { return _seqs.at(s).lastRelative; }
  // the full result of sequence s's last frame (pose, guess, alignment record)
  const nicp_track_result &lastResult(int s) const { return _seqs.at(s).last; }

  // SequentialTracker::processFrame for raws[k] of sequence sequences[k], every k (distinct sequences); initialGuesses is
  // empty (identity) or holds one guess per frame
  void processFrames(const std::vector<int> &sequences, const std::vector<const RawDepthImage *> &raws,
                     const Isometry3f &sensorOffset, const Matrix3f &cameraMatrix,
                     const std::vector<Isometry3f> &initialGuesses = std::vector<Isometry3f>(), float depthScale = 0.001f) {
    const size_t n = sequences.size();
    if (raws.size() != n || (!initialGuesses.empty() && initialGuesses.size() != n))
      throw std::runtime_error("BatchTracker::processFrames: one raw image (and one guess, if any) per sequence");
    if (n == 0) return;
    for (size_t k = 0; k < n; k++)
      if (!raws[k] || raws[k]->rows != raws[0]->rows || raws[k]->cols != raws[0]->cols)
        throw std::runtime_error("BatchTracker::processFrames: every raw image must have the same size");
    ensureTracker(*raws[0], sensorOffset, cameraMatrix, depthScale);
    std::vector<const uint16_t *> ptrs(n);
    for (size_t k = 0; k < n; k++) ptrs[k] = raws[k]->data();
    std::vector<float> odometry;
    for (const Isometry3f &g : initialGuesses) odometry.insert(odometry.end(), g.data(), g.data() + 16);
    std::vector<nicp_track_result> results(n);
    nicpCheck(nicp_tracker_step(_tracker, (int)n, sequences.data(), ptrs.data(), odometry.empty() ? 0 : odometry.data(),
                                results.data()),
              "BatchTracker::processFrames");
    for (size_t k = 0; k < n; k++) {
      Seq &s = _seqs[sequences[k]];
      const nicp_track_result &r = results[k];
      std::memcpy(s.globalT.data(), r.global_T, sizeof r.global_T);
      if (r.aligned) {  // a first frame leaves SequentialTracker's _lastInliers and _lastRelative as they were
        s.lastInliers = r.record.inliers;
        std::memcpy(s.lastRelative.data(), r.relative_T, sizeof r.relative_T);
      }
      s.numKeyframes = r.num_keyframes;
      s.lastWasKeyframe = r.keyframe != 0;
      s.last = r;
    }
  }

 protected:
  struct Seq {
    Isometry3f globalT, lastRelative;
    int numKeyframes, lastInliers;
    bool lastWasKeyframe;
    nicp_track_result last;
    Seq() : numKeyframes(0), lastInliers(0), lastWasKeyframe(false) { std::memset(&last, 0, sizeof last); }
  };
  // Aligner keeps PwnMatcherBase's frame inlier depth threshold protected: read it through a derived class's member pointer
  struct AlignerThreshold : Aligner {
    static float of(const Aligner &a) { return a.*(&AlignerThreshold::_frameInlierDepthThreshold); }
  };

  // SequentialTracker::makeCloud's scaled camera and image size; the C-ABI tracker on the first call
  void ensureTracker(const RawDepthImage &raw, const Isometry3f &sensorOffset, const Matrix3f &cameraMatrix, float depthScale) {
    PinholePointProjector *projector = dynamic_cast<PinholePointProjector *>(_converter->projector());
    PinholePointProjector *alprojector = dynamic_cast<PinholePointProjector *>(_aligner->projector());
    if (!projector || !alprojector)
      throw std::runtime_error("BatchTracker: the converter and the aligner need PinholePointProjectors");
    float invScale = 1.0f / _scale;
    Matrix3f scaledCameraMatrix = cameraMatrix * invScale;
    scaledCameraMatrix(2, 2) = 1.0f;
    projector->setCameraMatrix(scaledCameraMatrix);
    projector->setImageSize(raw.rows / _scale, raw.cols / _scale);
    nicp_projector p = projector->abiProjector();
    if (alprojector->minDistance() != p.min_distance || alprojector->maxDistance() != p.max_distance)
      throw std::runtime_error("BatchTracker: the aligner's projector needs the converter's distance range");
    Key key;
    std::memset(&key, 0, sizeof key);
    key.proj = p;
    key.rawRows = raw.rows;
    key.rawCols = raw.cols;
    key.scale = _scale;
    key.depthScale = depthScale;
    key.newFrameInliersFraction = _newFrameInliersFraction;
    std::memcpy(key.sensorOffset, sensorOffset.data(), sizeof key.sensorOffset);
    if (_tracker) {
      if (std::memcmp(&key, &_key, sizeof key))
        throw std::runtime_error("BatchTracker: camera matrix, sensor offset, raw size, depth scale, scale and keyframe "
                                 "fraction are fixed by the first processFrames call");
      return;
    }
    nicp_stats_params sp = _converter->abiStatsParams();
    nicp_align_params ap = _aligner->abiAlignParams();
    nicpCheck(nicp_tracker_create(_pool, (int)_seqs.size(), raw.rows, raw.cols, depthScale, _scale, 0.01f, &p, &sp,
                                  sensorOffset.data(), &ap, AlignerThreshold::of(*_aligner), _newFrameInliersFraction,
                                  &_tracker),
              "BatchTracker: nicp_tracker_create");
    _key = key;
  }

  struct Key {
    nicp_projector proj;
    int rawRows, rawCols, scale;
    float depthScale, newFrameInliersFraction;
    float sensorOffset[16];
  };
  DepthImageConverterIntegralImage *_converter;
  Aligner *_aligner;
  int _scale;
  float _newFrameInliersFraction;
  nicp_shard_pool *_pool;
  nicp_tracker *_tracker;
  Key _key;
  std::vector<Seq> _seqs;

 private:
  BatchTracker(const BatchTracker &);
  BatchTracker &operator=(const BatchTracker &);
};

}  // namespace pwn

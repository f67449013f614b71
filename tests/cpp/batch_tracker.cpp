// batch_tracker.cpp -- pwn::BatchTracker (include/pwn/batch_tracker.h) against one pwn::SequentialTracker per sequence
// (include/pwn/tracker.h): after every frame, globalT, lastRelative, lastInliers, numKeyframes and lastWasKeyframe must be
// bit-identical.  tests/test_tracker.py writes the input and builds this file with -ffp-contract=off.
//   batch_tracker in.bin workers
// in.bin: int32 S, F, rows, cols, scale, with_odometry, minImageRadius, maxImageRadius, minPoints;
//         float32 K (9, column-major), sensor offset (16, column-major), newFrameInliersFraction, inlierDistanceThreshold,
//         minDistance, maxDistance;
//         uint16 raw frames [F][S][rows][cols]; float32 odometry [F][S][16] when with_odometry.
// Sequence s takes a frame at step f unless (f + s) % 4 == 3; each step lists its sequences in reverse order.
// Prints "frame f seq s inliers i keyframes k" per processed frame and "batch_tracker ok" at the end; exits 1 on the first
// difference.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "pwn/batch_tracker.h"
#include "pwn/tracker.h"

using namespace pwn;

template <typename T>
static void readv(FILE *f, T *p, size_t n) {
  if (fread(p, sizeof(T), n, f) != n) throw std::runtime_error("short input");
}

static bool same(const Isometry3f &a, const Isometry3f &b) { return std::memcmp(a.data(), b.data(), 64) == 0; }

int main(int argc, char **argv) {
  if (argc < 3) return 2;
  FILE *in = fopen(argv[1], "rb");
  if (!in) return 2;
  int hdr[9];
  readv(in, hdr, 9);
  const int S = hdr[0], F = hdr[1], rows = hdr[2], cols = hdr[3], scale = hdr[4], withOdometry = hdr[5];
  float v[9 + 16 + 4];
  readv(in, v, 29);
  Matrix3f K;
  for (int i = 0; i < 9; i++) K.m[i] = v[i];
  Isometry3f sensorOffset;
  for (int i = 0; i < 16; i++) sensorOffset.data()[i] = v[9 + i];
  std::vector<std::vector<RawDepthImage>> raws(F, std::vector<RawDepthImage>(S));
  for (int f = 0; f < F; f++)
    for (int s = 0; s < S; s++) {
      raws[f][s].create(rows, cols);
      readv(in, raws[f][s].data(), (size_t)rows * cols);
    }
  std::vector<std::vector<Isometry3f>> odometry(F, std::vector<Isometry3f>(S));
  if (withOdometry)
    for (int f = 0; f < F; f++)
      for (int s = 0; s < S; s++) readv(in, odometry[f][s].data(), 16);
  fclose(in);

  PinholePointProjector projector;
  projector.setMinDistance(v[27]);
  projector.setMaxDistance(v[28]);
  StatsCalculatorIntegralImage statsCalculator;
  statsCalculator.setMinImageRadius(hdr[6]);
  statsCalculator.setMaxImageRadius(hdr[7]);
  statsCalculator.setMinPoints(hdr[8]);
  statsCalculator.setCurvatureThreshold(0.2f);
  PointInformationMatrixCalculator pointInfo;
  NormalInformationMatrixCalculator normalInfo;
  DepthImageConverterIntegralImage converter(&projector, &statsCalculator, &pointInfo, &normalInfo);
  CorrespondenceFinder finder;
  finder.setInlierDistanceThreshold(v[26]);
  finder.setInlierNormalAngularThreshold(0.95f);
  Linearizer linearizer;
  Aligner aligner;
  aligner.setProjector(&projector);
  aligner.setLinearizer(&linearizer);
  aligner.setCorrespondenceFinder(&finder);

  std::vector<SequentialTracker *> single(S);
  for (int s = 0; s < S; s++) {
    single[s] = new SequentialTracker(&converter, &aligner);
    single[s]->setScale(scale);
    single[s]->setNewFrameInliersFraction(v[25]);
  }
  BatchTracker batch(&converter, &aligner, std::vector<int>(std::atoi(argv[2]), 0), S);
  batch.setScale(scale);
  batch.setNewFrameInliersFraction(v[25]);

  for (int f = 0; f < F; f++) {
    std::vector<int> seqs;
    std::vector<const RawDepthImage *> frames;
    std::vector<Isometry3f> guesses;
    for (int s = S - 1; s >= 0; s--) {
      if ((f + s) % 4 == 3) continue;
      seqs.push_back(s);
      frames.push_back(&raws[f][s]);
      guesses.push_back(odometry[f][s]);
    }
    batch.processFrames(seqs, frames, sensorOffset, K, withOdometry ? guesses : std::vector<Isometry3f>(), 0.001f);
    for (size_t k = 0; k < seqs.size(); k++) {
      const int s = seqs[k];
      SequentialTracker &t = *single[s];
      t.processFrame(raws[f][s], sensorOffset, K, odometry[f][s], 0.001f);
      if (!same(t.globalT(), batch.globalT(s)) || !same(t.lastRelative(), batch.lastRelative(s)) ||
          t.lastInliers() != batch.lastInliers(s) || t.numKeyframes() != batch.numKeyframes(s) ||
          t.lastWasKeyframe() != batch.lastWasKeyframe(s)) {
        printf("differ at frame %d seq %d: inliers %d / %d, keyframes %d / %d, keyframe %d / %d, globalT %d, relative %d\n",
               f, s, t.lastInliers(), batch.lastInliers(s), t.numKeyframes(), batch.numKeyframes(s), (int)t.lastWasKeyframe(),
               (int)batch.lastWasKeyframe(s), (int)same(t.globalT(), batch.globalT(s)),
               (int)same(t.lastRelative(), batch.lastRelative(s)));
        return 1;
      }
      printf("frame %d seq %d inliers %d keyframes %d\n", f, s, t.lastInliers(), t.numKeyframes());
    }
  }
  // the fixed frame description: another camera matrix is refused
  bool threw = false;
  try {
    Matrix3f K2 = K * 1.01f;
    K2(2, 2) = 1.0f;
    batch.processFrames(std::vector<int>(1, 0), std::vector<const RawDepthImage *>(1, &raws[0][0]), sensorOffset, K2);
  } catch (const std::runtime_error &) {
    threw = true;
  }
  if (!threw) {
    printf("a changed camera matrix was accepted\n");
    return 1;
  }
  for (SequentialTracker *t : single) delete t;
  printf("batch_tracker ok\n");
  return 0;
}

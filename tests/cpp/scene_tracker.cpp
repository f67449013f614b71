// scene_tracker.cpp -- pwn::BatchSceneTracker (include/pwn/scene_tracker.h) set up from the same `key value` configuration as
// host/pwn_simple_aligner.cpp in localmap mode, on S sequences of F PGM frames each.  tests/test_scene_tracker.py builds this
// file with -ffp-contract=off and compares its lines with the driver's, sequence by sequence.
//   scene_tracker config.conf out.jsonl workers S F seq0_frame0.pgm .. seq0_frame{F-1}.pgm seq1_frame0.pgm ...
// Step f lists every sequence (in reverse order on odd f).  Writes, per processed frame, the driver's line with a "seq" key
// in front, and per sequence at the end {"seq", "map_points", "voxel_points"}: the map downloaded and voxelised with
// nicp_voxelize at the configuration's voxelResolution.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <map>
#include <sstream>
#include <string>
#include <vector>

#include "pwn/scene_tracker.h"

using namespace pwn;

static std::map<std::string, float> readConfig(const char *path) {
  std::map<std::string, float> m;
  std::ifstream is(path);
  std::string line;
  while (std::getline(is, line)) {
    if (line.empty() || line[0] == '#' || line[0] == '/') continue;
    std::istringstream ls(line);
    std::string key;
    float v;
    if (ls >> key >> v) m[key] = v;
  }
  return m;
}

static float get(const std::map<std::string, float> &m, const char *k, float def) {
  std::map<std::string, float>::const_iterator it = m.find(k);
  return it == m.end() ? def : it->second;
}

static void readPgm16(const char *path, RawDepthImage &img) {
  FILE *f = fopen(path, "rb");
  if (!f) throw std::runtime_error(std::string("cannot read ") + path);
  int w = 0, h = 0, maxv = 0;
  if (fscanf(f, "P5 %d %d %d", &w, &h, &maxv) != 3) throw std::runtime_error("bad PGM header");
  fgetc(f);
  img.create(h, w);
  std::vector<unsigned char> buf((size_t)w * h * 2);
  if (fread(buf.data(), 1, buf.size(), f) != buf.size()) throw std::runtime_error("short PGM");
  fclose(f);
  for (size_t i = 0; i < (size_t)w * h; i++) img.data()[i] = (uint16_t)((buf[2 * i] << 8) | buf[2 * i + 1]);
}

int main(int argc, char **argv) {
  if (argc < 6) return 2;
  try {
    std::map<std::string, float> cfg = readConfig(argv[1]);
    FILE *out = fopen(argv[2], "w");
    const int workers = std::atoi(argv[3]), S = std::atoi(argv[4]), F = std::atoi(argv[5]);
    if (argc != 6 + S * F || !out) return 2;
    // the driver's objects (pwn_simple_aligner.cpp main, localmap mode)
    const int imageScale = (int)get(cfg, "imageScale", 1);
    const float depthScale = get(cfg, "depthScale", 0.001f);
    Matrix3f K;
    K.setIdentity();
    K(0, 0) = get(cfg, "fx", 525.0f); K(1, 1) = get(cfg, "fy", 525.0f);
    K(0, 2) = get(cfg, "cx", 319.5f); K(1, 2) = get(cfg, "cy", 239.5f);
    Vector6f v;
    v(0) = get(cfg, "sensorOffsetTx", 0); v(1) = get(cfg, "sensorOffsetTy", 0); v(2) = get(cfg, "sensorOffsetTz", 0);
    v(3) = get(cfg, "sensorOffsetQx", 0); v(4) = get(cfg, "sensorOffsetQy", 0); v(5) = get(cfg, "sensorOffsetQz", 0);
    const Isometry3f sensorOffset = v2t(v);
    PinholePointProjector projector;
    projector.setMinDistance(get(cfg, "minDistance", 0.5f));
    projector.setMaxDistance(get(cfg, "maxDistance", 4.5f));
    projector.setCameraMatrix(K);
    StatsCalculatorIntegralImage statsCalculator;
    statsCalculator.setMinImageRadius((int)get(cfg, "minImageRadius", 10));
    statsCalculator.setMaxImageRadius((int)get(cfg, "maxImageRadius", 30));
    statsCalculator.setMinPoints((int)get(cfg, "minPoints", 50));
    statsCalculator.setCurvatureThreshold(get(cfg, "curvatureThreshold", 0.2f));
    statsCalculator.setWorldRadius(get(cfg, "worldRadius", 0.1f));
    PointInformationMatrixCalculator pointInfo;
    NormalInformationMatrixCalculator normalInfo;
    pointInfo.setCurvatureThreshold(get(cfg, "informationMatrixCurvatureThreshold", 0.02f));
    normalInfo.setCurvatureThreshold(get(cfg, "informationMatrixCurvatureThreshold", 0.02f));
    DepthImageConverterIntegralImage converter(&projector, &statsCalculator, &pointInfo, &normalInfo);
    CorrespondenceFinder finder;
    finder.setInlierDistanceThreshold(get(cfg, "inlierDistanceThreshold", 1.0f));
    finder.setInlierNormalAngularThreshold(get(cfg, "inlierNormalAngularThreshold", 0.95f));
    finder.setInlierCurvatureRatioThreshold(get(cfg, "inlierCurvatureRatioThreshold", 1.3f));
    finder.setFlatCurvatureThreshold(get(cfg, "flatCurvatureThreshold", 0.02f));
    Linearizer linearizer;
    linearizer.setInlierMaxChi2(get(cfg, "inlierMaxChi2", 9e3f));
    linearizer.setRobustKernel(get(cfg, "robustKernel", 1) != 0);
    Aligner aligner;
    aligner.setProjector(&projector);
    aligner.setLinearizer(&linearizer);
    aligner.setCorrespondenceFinder(&finder);
    aligner.setOuterIterations((int)get(cfg, "outerIterations", 10));
    aligner.setInnerIterations((int)get(cfg, "innerIterations", 1));
    aligner.setMinInliers((int)get(cfg, "minInliers", 100));
    aligner.setSensorOffset(sensorOffset);
    Merger merger;
    merger.setDepthImageConverter(&converter);
    merger.setDistanceThreshold(get(cfg, "mergerDistanceThreshold", 0.1f));
    merger.setNormalThreshold(get(cfg, "mergerNormalThreshold", cosf(10 * M_PI / 180.0f)));
    merger.setMaxPointDepth(get(cfg, "mergerMaxPointDepth", 10.0f));

    std::vector<std::vector<RawDepthImage>> raws(S, std::vector<RawDepthImage>(F));
    for (int s = 0; s < S; s++)
      for (int f = 0; f < F; f++) readPgm16(argv[6 + s * F + f], raws[s][f]);
    const int px = (raws[0][0].rows / imageScale) * (raws[0][0].cols / imageScale);
    BatchSceneTracker tracker(&converter, &aligner, &merger, std::vector<int>(workers, 0), S, (F + 1) * px);
    tracker.setScale(imageScale);
    tracker.setChunkStep((int)get(cfg, "chunkStep", 10));
    for (int f = 0; f < F; f++) {
      std::vector<int> seqs;
      std::vector<const RawDepthImage *> frames;
      for (int k = 0; k < S; k++) {
        const int s = f % 2 ? S - 1 - k : k;
        seqs.push_back(s);
        frames.push_back(&raws[s][f]);
      }
      tracker.processFrames(seqs, frames, sensorOffset, K, depthScale);
      for (int s : seqs) {
        fprintf(out, "{\"seq\": %d, \"frame\": %d, \"inliers\": %d, \"added\": %d, \"map_points\": %d, \"new_map\": %d, "
                     "\"globalT\": [",
                s, f, tracker.lastInliers(s), tracker.lastAdded(s), tracker.mapSize(s), tracker.lastNewMap(s) ? 1 : 0);
        for (int i = 0; i < 16; i++) fprintf(out, "%s%.9g", i ? ", " : "", tracker.globalT(s).data()[i]);
        fprintf(out, "]}\n");
      }
    }
    // VoxelCalculator on each final map: downloaded, uploaded to a cloud of this thread's context, nicp_voxelize
    const float resolution = get(cfg, "voxelResolution", 0.01f);
    nicp_context *ctx = Context::current().handle();
    for (int s = 0; s < S; s++) {
      const int cap = tracker.mapSize(s);
      std::vector<float> points((size_t)4 * cap + 4), normals((size_t)4 * cap + 4), curvature((size_t)cap + 1);
      int n = 0;
      nicpCheck(nicp_scene_tracker_download_map(tracker.handle(), s, cap, points.data(), normals.data(), curvature.data(), 0, 0,
                                                0, 0, &n),
                "nicp_scene_tracker_download_map");
      int voxels = 0;
      if (n) {
        nicp_cloud *c = 0;
        nicpCheck(nicp_cloud_create(ctx, n, &c), "nicp_cloud_create");
        nicpCheck(nicp_cloud_upload(ctx, c, n, points.data(), normals.data(), curvature.data(), 0, 0), "nicp_cloud_upload");
        nicpCheck(nicp_voxelize(ctx, c, resolution, 0, &voxels), "nicp_voxelize");
        nicp_cloud_destroy(c);
      }
      fprintf(out, "{\"seq\": %d, \"map_points\": %d, \"voxel_points\": %d}\n", s, n, voxels);
    }
    fclose(out);
  } catch (const std::exception &e) {
    fprintf(stderr, "scene_tracker: %s\n", e.what());
    return 1;
  }
  return 0;
}

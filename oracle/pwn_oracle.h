/*
 * pwn_oracle.h -- CPU restatement of g2o_frontend's pwn_core NICP hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is part of the product: only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load it.
 *
 * PARITY UNPINNED: the reference (/root/reference/g2o_frontend/pwn_core) cannot be built in
 * this image (needs Eigen3, OpenCV, PCL, g2o; none installed, no network) and ships no tests
 * or golden vectors for this path.  This file restates the reference's algorithm from its
 * sources; the Eigen arithmetic it relies on (un-vendored, version only lower-bounded at
 * 3.1.2 by /root/reference/CMakeLists.txt:158) is restated from the published Eigen 3.2.x
 * algorithms with one fixed float32 evaluation order (SURVEY.md Appendix A).
 * PINNED since (DESIGN.md section 2), for everything except Eigen's numerical kernels:
 *  - oracle/_ref/libpwn_core_ref.so = the reference's own pwn_core sources compiled (oracle/build_ref_pwn_core.sh)
 *    against the Eigen / OpenCV stand-ins of oracle/shim/; tests/test_reference_pwn_core.py finds this file
 *    bit-identical to it stage by stage and for whole alignments (all thread counts, priors, sensor offsets);
 *  - oracle/_ref/libpwn_cuda_ref.so = the reference's own CUDA implementation (pwn_cuda, CUDA runtime only), unmodified;
 *    tests/test_reference_pwn_cuda.py checks the SE(3) helpers, the gates and the per-correspondence Linearizer terms.
 * Still UNPINNED: what Eigen computes inside (computeDirect, LDLT, JacobiSVD, Quaternion(R), product summation order) --
 * the stand-in delegates those to the restatements below, so both sides share them.
 *
 * Conventions: all matrices are column-major float (Eigen default): M(r,c) = m[c*R + r].
 * Images are row-major rows x cols (cv::Mat_).  Points/normals are 4 floats (x,y,z,w).
 */
#ifndef PWN_ORACLE_H
#define PWN_ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- pwn_static.cpp ---- */
void orc_depth_u16_to_f32(const uint16_t *src, int n, float scale, float *dst);
void orc_depth_f32_to_u16(const float *src, int n, float scale, uint16_t *dst);
void orc_depth_scale(const float *src, int rows, int cols, int step, float maxDepthCov, float *dst);

/* ---- SE(3) helpers, bm_se3.h ---- */
void orc_v2t(const float v[6], float T[16]);
void orc_t2v(const float T[16], float v[6]);
void orc_iso_inverse(const float T[16], float Ti[16]);
void orc_iso_mul(const float A[16], const float B[16], float C[16]);

/* ---- PinholePointProjector ---- */
void orc_update_matrices(const float K[9], const float T[16], float KRt[16], float iKRt[16]);
int orc_unproject(const float *depth, int rows, int cols, const float iKRt[16], float minD, float maxD,
                  float *points, int *index);
void orc_project_intervals(const float *depth, int rows, int cols, const float K[9], float minD, float maxD,
                           float worldRadius, int *interval);
void orc_project(const float *points, int n, int rows, int cols, const float KRt[16], float minD, float maxD,
                 int *index, float *depth);

/* ---- PointIntegralImage (10 unique channels per pixel: n,x,y,z,xx,xy,xz,yy,yz,zz) ---- */
void orc_integral_image(const int *index, const float *points, int rows, int cols, float *integral);

/* ---- StatsCalculatorIntegralImage + information matrices + Cloud::transformInPlace ---- */
typedef struct {
  float worldRadius;
  int minImageRadius, maxImageRadius, minPoints;
  float curvatureThreshold;       /* stats calculator */
  float omegaCurvatureThreshold;  /* information matrix calculators */
  float flatOmegaP[3], nonFlatOmegaP[3]; /* diag; nonFlatOmegaP is overwritten by 1/eigenvalues */
  float flatOmegaN[3], nonFlatOmegaN[3];
} orc_stats_params;

void orc_eigen3(const float C[9], float evals[3], float evecs[9]);      /* Eigen 3.2.x computeDirect */
void orc_eigen3_v33(const float C[9], float evals[3], float evecs[9]);  /* Eigen >= 3.3 computeDirect (sensitivity study) */
void orc_eigen3_devtrig(const float C[9], float evals[3], float evecs[9]); /* 3.2.x, trig in float64 as the CUDA path */
void orc_set_eigen_variant(int v); /* which orc_stats / orc_depth_to_cloud use: 0 = 3.2 (default), 1 = >= 3.3,
                                      2 = 3.2 with the CUDA path's float64 atan2 / cos / sin (orc_eigen3_devtrig) */

void orc_stats(const float *integral, const int *index, const int *interval, const float *points,
               int rows, int cols, int n, const orc_stats_params *p,
               float *normals, float *statsM, float *eigvals, int *statsN, float *curvature);
void orc_information(const float *normals, const float *statsM, const float *eigvals, const float *curvature,
                     int n, const orc_stats_params *p, float *omegaP, float *omegaN);
void orc_cloud_transform(const float T[16], int n, float *points, float *normals, float *statsM,
                         float *omegaP, float *omegaN);

/* DepthImageConverterIntegralImage::compute in one call; returns the number of points */
int orc_depth_to_cloud(const float *depth, int rows, int cols, const float K[9], float minD, float maxD,
                       const orc_stats_params *p, const float sensorOffset[16],
                       float *points, float *normals, float *statsM, float *eigvals, int *statsN,
                       float *curvature, float *omegaP, float *omegaN, int *index, int *interval,
                       float *integral);

/* ---- MultiPointProjector (multipointprojector.{h,cpp}) ------------------------------------------
 * Composite image layout as the Aligner actually executes it (SURVEY.md section 8a rows 11-12): the
 * base-class z-buffer PointProjector::project (pointprojector.cpp:17-40) over the per-point
 * MultiPointProjector::project (multipointprojector.cpp:157-205): composite rows = max child
 * "width" (the pixel u coordinate), composite cols = sum of child "heights" (v + column offset);
 * first child whose pinhole projection lands inside [0,width) x [0,height) wins; empty depth = 0.
 * unProject is DEFINED as the inverse of that layout (the reference's own cv::Rect slicing is
 * inconsistent with it after the Eigen->cv::Mat port): points ordered by child, raster order inside
 * the child's column block. */
#define ORC_MAX_CAMERAS 8
typedef struct {
  int n;
  int width[ORC_MAX_CAMERAS], height[ORC_MAX_CAMERAS];  /* ChildProjectorInfo: setImageSize(width, height) */
  float minD[ORC_MAX_CAMERAS], maxD[ORC_MAX_CAMERAS];
  float K[ORC_MAX_CAMERAS][9];
  float offset[ORC_MAX_CAMERAS][16];                    /* ChildProjectorInfo::sensorOffset */
} orc_multi;

void orc_multi_image_size(const orc_multi *m, int *rows, int *cols);
int orc_multi_unproject(const orc_multi *m, const float T[16], const float *depth, int rows, int cols,
                        float *points, int *index);
void orc_multi_intervals(const orc_multi *m, const float *depth, int rows, int cols, float worldRadius, int *interval);
void orc_multi_project(const orc_multi *m, const float T[16], const float *points, int n, int rows, int cols,
                       int *index, float *depth);
int orc_multi_depth_to_cloud(const orc_multi *m, const float *depth, int rows, int cols, const orc_stats_params *p,
                             const float sensorOffset[16], float *points, float *normals, float *statsM, float *eigvals,
                             int *statsN, float *curvature, float *omegaP, float *omegaN, int *index, int *interval,
                             float *integral);

/* ---- CorrespondenceFinder ---- */
typedef struct {
  float inlierDistanceThreshold;
  float inlierNormalAngularThreshold;
  float flatCurvatureThreshold;
  float inlierCurvatureRatioThreshold;
} orc_corr_params;

int orc_correspond(const int *refIndex, const int *curIndex, int rows, int cols,
                   const float *refPoints, const float *refNormals, const float *refCurv,
                   const float *curPoints, const float *curNormals, const float *curCurv,
                   const float T[16], const orc_corr_params *p, int numThreads,
                   int *corr /* 2*rows*cols, (ref,cur) compacted, tail -1 */,
                   int *corrImage /* rows*cols: refIdx accepted at that pixel or -1; may be NULL */);

/* ---- Linearizer ---- */
void orc_linearize(const int *corr, int numCorr,
                   const float *refPoints, const float *refNormals,
                   const float *curPoints, const float *curNormals,
                   const float *curOmegaP, const float *curOmegaN,
                   const float T[16], float inlierMaxChi2, int robustKernel, int numThreads,
                   float H[36], float b[6], float *error, int *inliers);
/* same sums accumulated in float64 over ALL correspondences (accuracy yardstick, not the reference) */
void orc_linearize_f64(const int *corr, int numCorr,
                       const float *refPoints, const float *refNormals,
                       const float *curPoints, const float *curNormals,
                       const float *curOmegaP, const float *curOmegaN,
                       const float T[16], float inlierMaxChi2, int robustKernel,
                       double H[36], double b[6], double *error, int *inliers);

void orc_ldlt_solve6(const float H[36], const float b[6], float x[6]);

/* ---- SE3 priors (se3_prior.cpp) ---- */
typedef struct {
  int kind;            /* 0 = relative, 1 = absolute */
  float mean[16];
  float refInv[16];    /* inverse reference transform (absolute prior) */
  float info[36];
} orc_prior;

/* ---- Aligner::align ---- */
typedef struct {
  int outerIterations, innerIterations;
  float K[9];
  int rows, cols;
  float minD, maxD;
  float refSensorOffset[16], curSensorOffset[16], initialGuess[16];
  orc_corr_params corr;
  float inlierMaxChi2;
  int robustKernel;
  int numThreads;
  int numPriors;
  const orc_prior *priors;
  const orc_multi *multi;   /* NULL: PinholePointProjector(K); else MultiPointProjector (K, minD, maxD unused) */
} orc_align_params;

typedef struct {
  float T[16];
  float H[36], b[6];     /* last linearisation (the one of _computeStatistics, at the final T) */
  float error;           /* Aligner::error(): from the LAST LOOP linearisation */
  int inliers;
  int numCorrespondences;
  float omega[36], mean[6];
  float translationalRatio, rotationalRatio;
} orc_align_result;

/* trace (optional, may be NULL): per outer iteration, T at the start of the iteration (16),
   H (36), b (6), error, inliers, numCorr -> 61 floats per iteration */
#define ORC_TRACE_STRIDE 61
void orc_align(int nRef, const float *refPoints, const float *refNormals, const float *refCurv,
               int nCur, const float *curPoints, const float *curNormals, const float *curCurv,
               const float *curOmegaP, const float *curOmegaN,
               const orc_align_params *p, orc_align_result *res,
               int *refIndex, float *refDepth, int *curIndex, float *curDepth, int *corr,
               float *trace);
/* the two dense pieces of orc_align on their own (the same static functions, no behaviour of their own):
 * orc_compute_statistics is the _computeStatistics tail (aligner.cpp:172-198) on the linearisation H at T;
 * orc_gn_step is one outer iteration with innerIterations = 1 after its linearisation (aligner.cpp:84-118): invT = T^-1
 * (fixLastRow), H + I + 1000 I and -b with the priors added at invT, LDLT, invT = v2t(dx) invT, T = v2t(t2v(invT^-1)),
 * fixLastRow -> Tnext.  Matrices column-major. */
void orc_compute_statistics(const float H[36], const float T[16], float mean[6], float Omega[36], float *tr, float *rr);
void orc_gn_step(const float H[36], const float b[6], const float T[16], const orc_prior *priors, int numPriors,
                 float Tnext[16]);

/* test knob: float64 accumulation of the Linearizer sums inside orc_align (0 = reference behaviour) */
void orc_set_accumulate_f64(int on);
int orc_set_threads(int n); /* omp_set_num_threads(n) if n > 0; returns omp_get_max_threads() */

/* PwnMatcherBase::matchClouds image statistics (pwn_tracker2/pwn_matcher_base.cpp:156-196) */
void orc_image_stats(const float *curDepth, const float *refDepth, int n, float inlierDepthThreshold,
                     int *nonZeros, int *inliers, int *outliers, float *reprojectionDistance);

/* ---- local-map maintenance (SURVEY.md section 8f rank 3) -------------------------------------------
 * Gaussian3f sensor model (pinholepointprojector.cpp:93-133, basemath/gaussian.h, gaussian3.h:26-36),
 * Merger::merge (merger.cpp:15-119).  A Gaussian is 24 floats + a flag word:
 *   g[0..2] mean, g[3..11] covariance (column-major 3x3), g[12..14] information vector,
 *   g[15..23] information matrix; flags bit 0 = _momentsUpdated, bit 1 = _infoUpdated
 * (the reference keeps both forms with lazy conversion through Matrix3f::inverse()). */
#define ORC_GAUSS_FLOATS 24
#define ORC_GAUSS_MOMENTS 1
#define ORC_GAUSS_INFO 2
/* unProject(points, gaussians, index, depth): gaussians of the valid pixels in raster order */
int orc_unproject_gaussians(const float *depth, int rows, int cols, const float K[9], const float iKRt[16],
                            float minD, float maxD, float baseline, float alpha, float *points, int *index,
                            float *gauss, int *gflags);
/* Gaussian3fVector::transformInPlace (skipped, like Cloud::transformInPlace, when T is the identity) */
void orc_gaussians_transform(const float T[16], int n, float *gauss, int *gflags);
/* Merger::merge.  All arrays are compacted in place; returns the new point count.  collapsed (n ints, may be
 * NULL) receives _collapsedIndices; omegaP/omegaN/statsM may be NULL. */
int orc_merge(int n, float *points, float *normals, float *statsM, float *omegaP, float *omegaN, float *gauss,
              int *gflags, int rows, int cols, const float K[9], const float T[16], float minD, float maxD,
              float distanceThreshold, float normalThreshold, float maxPointDepth, int *collapsed);

#ifdef __cplusplus
}
#endif
#endif

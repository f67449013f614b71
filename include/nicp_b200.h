/*
 * nicp_b200.h -- C-ABI of the B200-native NICP registration hot path.
 *
 * Drop-in boundary for g2o_frontend's pwn_core (reference paths below are relative to
 * /root/reference/g2o_frontend/pwn_core/).  The reference's seam is the C++ class API of
 * namespace pwn; its only GPU precedent is the flat function API of
 * pwn_cuda/cudaaligner.h:59-80 (createContext / initComputation / simpleIteration / getHb with
 * raw float* / int*, column-major 4x4, status return).  This header is the same kind of seam:
 * extern "C", plain pointers and sizes, int status codes, no exceptions, no torch types.
 * include/pwn/ holds the C++ pwn:: classes (same names, setters and defaults as the reference)
 * implemented over these entry points.
 *
 * Conventions
 *   - matrices: column-major float32 (Eigen default).  4x4 isometries as float[16], K as float[9].
 *   - images: row-major rows x cols (cv::Mat_).  Index images int32 (-1 = empty), depth float32
 *     metres (empty z-buffer pixel = FLT_MAX, pinholepointprojector.cpp:41).
 *   - points/normals on the host side: 4 floats per element (x,y,z,w), w=1 / w=0
 *     (homogeneousvector4f.h:17-83).  Information matrices: 6 floats per point, the upper
 *     triangle xx,xy,xz,yy,yz,zz of the 3x3 block (informationmatrix.h:13-84 stores a 4x4 whose
 *     last row/column are zero; the reference's U*D*U^T is symmetric up to float rounding, the
 *     device keeps the row<=col entries).
 *   - every host pointer may be pageable or pinned memory; calls are synchronous unless stated.
 *   - there is NO CPU fallback: every entry point fails with NICP_ERR_CUDA when no device works.
 */
#ifndef NICP_B200_H
#define NICP_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NICP_OK 0
#define NICP_ERR_INVALID 1   /* bad argument (null handle, zero-sized image, capacity exceeded) */
#define NICP_ERR_CUDA 2      /* a CUDA runtime call or kernel failed; see nicp_last_error() */
#define NICP_ERR_ALLOC 3

/* Largest image frame preparation (nicp_depth_to_cloud, nicp_raw_depth_to_cloud(_batch), nicp_multi_depth_to_cloud,
 * nicp_multi_raw_depth_to_cloud_batch, nicp_stats_compute, the sharded closers) builds a cloud for; for a
 * MultiPointProjector the limits apply to the composite image (cols = sum of the cameras' heights).  A larger image is
 * rejected with NICP_ERR_INVALID before anything is uploaded.
 *   NICP_MAX_PREP_COLS    the row pass of the integral image stages 10 float channels of one row in the 227 KB of
 *                         shared memory a block may have (six 1920x1080 cameras, 6480 columns, do not fit)
 *   NICP_MAX_PREP_PIXELS  2^24: point indices, cloud sizes and window counts come from float32 pixel counts, which are
 *                         exact integers only up to 2^24 (eight 1920x1200 cameras, 18.4 M pixels, exceed it) */
#define NICP_MAX_PREP_COLS 5810
#define NICP_MAX_PREP_PIXELS 16777216

typedef struct nicp_context nicp_context; /* one per host thread / GPU (not thread-safe, like pwn_core) */
typedef struct nicp_cloud nicp_cloud;     /* device-resident pwn::Cloud (cloud.h:20-187) */

/* PointProjector + PinholePointProjector state (pointprojector.cpp:6-13, pinholepointprojector.cpp:5-13) */
typedef struct {
  float K[9];          /* camera matrix, column-major */
  int rows, cols;      /* image size */
  float min_distance;  /* default 0.01 */
  float max_distance;  /* default 6.0 */
} nicp_projector;

/* MultiPointProjector (multipointprojector.h:14-78): up to NICP_MAX_CAMERAS child pinholes, each added with
 * addPointProjector(projector, sensorOffset, width, height).  camera[i].rows / .cols hold that call's width /
 * height (the child's setImageSize(width, height), multipointprojector.h:61-78).  The composite image is the
 * one the Aligner really produces for this projector -- the base-class z-buffer PointProjector::project
 * (pointprojector.cpp:17-40) over the per-point MultiPointProjector::project (multipointprojector.cpp:157-205):
 * rows = max width (pixel u), cols = sum of heights (pixel v + column offset of the camera), the first camera
 * that sees a point wins, empty depth pixels are 0 (not FLT_MAX).  unProject is defined as the inverse of
 * that layout, points ordered by camera then raster order inside the camera's column block (the reference's
 * own cv::Rect slicing, multipointprojector.cpp:71-72, is inconsistent with it; see DESIGN.md). */
#define NICP_MAX_CAMERAS 8
typedef struct {
  int num_cameras;
  nicp_projector camera[NICP_MAX_CAMERAS];
  float sensor_offset[NICP_MAX_CAMERAS][16];  /* ChildProjectorInfo::sensorOffset */
} nicp_multi_projector;

/* StatsCalculatorIntegralImage (statscalculatorintegralimage.cpp:6-12) +
 * Point/NormalInformationMatrixCalculator (informationmatrixcalculator.h:100-150) */
typedef struct {
  float world_radius;               /* 0.1 */
  int min_image_radius;             /* 10 */
  int max_image_radius;             /* 30 */
  int min_points;                   /* 50 */
  float curvature_threshold;        /* 0.02  (stats) */
  float omega_curvature_threshold;  /* 0.02  (information matrices) */
  float flat_omega_p[3];            /* diag(1000,1,1) */
  float flat_omega_n[3];            /* diag(100,100,100) */
  float nonflat_omega_n[3];         /* diag(1,1,1); non-flat Omega_P is U diag(1/eigenvalues) U^T */
} nicp_stats_params;

/* CorrespondenceFinder (correspondencefinder.cpp:9-18), Linearizer (linearizer.cpp:9-15),
 * Aligner (aligner.cpp:13-32) */
typedef struct {
  float inlier_distance_threshold;         /* 0.5 */
  float inlier_normal_angular_threshold;   /* cos(pi/6) */
  float flat_curvature_threshold;          /* 0.02 */
  float inlier_curvature_ratio_threshold;  /* 1.3 */
  float inlier_max_chi2;                   /* 9e3 */
  int robust_kernel;                       /* 1 */
  int outer_iterations;                    /* 10 */
  int inner_iterations;                    /* 1 */
} nicp_align_params;

/* SE3Prior (se3_prior.h / se3_prior.cpp:8-71) as added by Aligner::addRelativePrior / addAbsolutePrior */
typedef struct {
  int kind;                  /* 0 = SE3RelativePrior, 1 = SE3AbsolutePrior */
  float mean[16];
  float reference[16];       /* reference transform (absolute prior only) */
  float information[36];     /* column-major 6x6 */
} nicp_prior;

/* Fixed 256-byte result record of one alignment: what Aligner exposes after align()
 * (aligner.h:115,314-332) plus PwnMatcherBase::matchClouds' image statistics
 * (pwn_tracker2/pwn_matcher_base.cpp:167-196).  This is also the record the batched /
 * multi-GPU path gathers. */
typedef struct {
  float T[16];                  /* Aligner::T() */
  float omega[36];              /* Aligner::omega() */
  float error;                  /* Aligner::error(): chi2 of the last loop linearisation */
  int inliers;                  /* Aligner::inliers() */
  int num_correspondences;      /* CorrespondenceFinder::numCorrespondences() of the last iteration */
  int image_non_zeros;          /* MatcherResult::image_nonZeros */
  int image_inliers;
  int image_outliers;
  float image_reprojection_distance;
  int status;                   /* NICP_OK or an error code for this pair */
  float translational_eigen_ratio;
  float rotational_eigen_ratio;
  float reserved[2];            /* roofline accounting: sums over the outer iterations of [0] pixels
                                   whose two index images are both valid, [1] accepted correspondences */
} nicp_align_result;

/* ---- context -------------------------------------------------------------------------- */
int nicp_create(int device, nicp_context **ctx);
void nicp_destroy(nicp_context *ctx);
const char *nicp_last_error(void);
int nicp_synchronize(nicp_context *ctx);
/* 1 if the library was built with --fmad=false (verification build), else 0 */
int nicp_is_verification_build(void);
/* number of kernel launches issued by this context since creation */
long long nicp_launch_count(const nicp_context *ctx);
/* Optional live kernel timing for the roofline report: when enabled, CUDA events are recorded on the
 * context's stream around every fused correspondence+linearise launch and every reference projection
 * launch of nicp_align / nicp_align_batch; totals (ms, launch count) since the last enable. */
int nicp_set_kernel_timing(nicp_context *ctx, int enable);
int nicp_get_kernel_timing(const nicp_context *ctx, double *corr_lin_ms, long long *corr_lin_launches,
                           double *project_ms, long long *project_launches);
/* the CUDA stream (cudaStream_t) this context launches on, for event timing by the caller */
void *nicp_stream(nicp_context *ctx);

/* ---- host-side helpers shared by the pwn:: classes (same bits as the device code) ------------ */
/* PinholePointProjector::_updateMatrices (pinholepointprojector.cpp:17-31): KRt = [K R^-1, K t_inv],
 * iKRt = [R K^-1, t] for a projector with camera matrix K and pose T.  Either output may be NULL. */
void nicp_update_matrices(const float K[9], const float T[16], float KRt[16], float iKRt[16]);
/* v2t / t2v (bm_se3.h:36-52): 6-vector (t, qx, qy, qz) <-> isometry */
void nicp_v2t(const float v[6], float T[16]);
void nicp_t2v(const float T[16], float v[6]);

/* ---- clouds (cloud.h) ------------------------------------------------------------------- */
int nicp_cloud_create(nicp_context *ctx, int capacity, nicp_cloud **cloud);
void nicp_cloud_destroy(nicp_cloud *cloud);
int nicp_cloud_size(const nicp_cloud *cloud);
/* host -> device.  normals4/curvature/omega_p6/omega_n6 may be NULL (zero-filled). */
int nicp_cloud_upload(nicp_context *ctx, nicp_cloud *cloud, int n, const float *points4,
                      const float *normals4, const float *curvature, const float *omega_p6,
                      const float *omega_n6);
/* device -> host; any output may be NULL */
int nicp_cloud_download(nicp_context *ctx, const nicp_cloud *cloud, float *points4, float *normals4,
                        float *curvature, float *omega_p6, float *omega_n6);
/* Stats (stats.h:13-121) if the cloud was built with keep_stats: 4x4 column-major per point
 * (eigenvectors + mean), eigenvalues (3), n.  Returns NICP_ERR_INVALID if not materialised. */
int nicp_cloud_download_stats(nicp_context *ctx, const nicp_cloud *cloud, float *stats16,
                              float *eigenvalues3, int *n_points);
/* Cloud::transformInPlace (cloud.cpp:173-186) */
int nicp_cloud_transform(nicp_context *ctx, nicp_cloud *cloud, const float T[16]);
/* Cloud::add (cloud.cpp:145-171): append a copy of src transformed by T (points, normals, curvature, information
 * matrices; Stats are not carried over).  Fails with NICP_ERR_INVALID if dst's capacity is too small. */
int nicp_cloud_append(nicp_context *ctx, nicp_cloud *dst, const nicp_cloud *src, const float T[16]);

/* ---- local-map maintenance (SURVEY.md section 8f rank 3) -------------------------------------------
 * Gaussian3f (basemath/gaussian.h): 24 floats per point -- mean (3), covariance (column-major 3x3),
 * information vector (3), information matrix (3x3) -- plus a flag word saying which form is valid
 * (the reference keeps both with lazy conversion through Matrix3f::inverse()). */
#define NICP_GAUSS_FLOATS 24
#define NICP_GAUSS_MOMENTS 1 /* Gaussian::_momentsUpdated */
#define NICP_GAUSS_INFO 2    /* Gaussian::_infoUpdated */
/* The sensor-model gaussians PinholePointProjector::unProject(points, gaussians, index, depth) produces
 * (pinholepointprojector.cpp:93-133: J = iK [z 0 c; 0 z r; 0 0 1], cov = J diag(3, 3, alpha z^2 / (baseline fx + alpha z)) J^T)
 * followed by Gaussian3fVector::transformInPlace(sensor_offset) (gaussian3.h:26-36), attached to a cloud that was
 * built from the SAME depth image, projector and sensor offset by nicp_depth_to_cloud (one gaussian per point, raster
 * order).  PinholePointProjector defaults: baseline 0.075, alpha 0.1 (pinholepointprojector.cpp:5-13). */
int nicp_cloud_compute_gaussians(nicp_context *ctx, nicp_cloud *cloud, const float *depth, const nicp_projector *proj,
                                 float baseline, float alpha, const float sensor_offset[16]);
/* 1 if the cloud carries gaussians.  nicp_cloud_transform / nicp_cloud_append carry them along (cloud.cpp:145-186). */
int nicp_cloud_has_gaussians(const nicp_cloud *cloud);
int nicp_cloud_download_gaussians(nicp_context *ctx, const nicp_cloud *cloud, float *gauss24, int *flags);
int nicp_cloud_upload_gaussians(nicp_context *ctx, nicp_cloud *cloud, const float *gauss24, const int *flags);
/* Merger (merger.cpp:5-13 defaults) */
typedef struct {
  float distance_threshold; /* 0.1 */
  float normal_threshold;   /* cosf(10 deg) */
  float max_point_depth;    /* 10 */
} nicp_merge_params;
/* Merger::merge(cloud, transform) (merger.cpp:15-119) with the Merger's image size = proj->rows x proj->cols: projects the
 * cloud with the projector at `transform`, fuses every point that lands on another point's pixel within the distance /
 * normal thresholds into that z-buffer winner (information-form addition in the reference's order), moves the winners to
 * the mean of their gaussian and removes the fused points (order preserving).  The cloud must carry gaussians.
 * collapsed (host, one int per input point, may be NULL) receives Merger::_collapsedIndices. */
int nicp_merge(nicp_context *ctx, nicp_cloud *cloud, const nicp_projector *proj, const float transform[16],
               const nicp_merge_params *params, int *collapsed, int *new_size);
/* VoxelCalculator::compute(cloud, resolution) (voxelcalculator.cpp:15-73): keeps the first point of every occupied voxel
 * of side `resolution` (voxel = truncated point * (1/resolution)), output ordered by voxel (x, then y, then z).  The
 * reference's map comparator (voxelcalculator.h:40-46) is not a strict weak ordering; this is the lexicographic order
 * it intends (DESIGN.md).  representatives (host, capacity = current size, may be NULL) receives the kept input indices. */
int nicp_voxelize(nicp_context *ctx, nicp_cloud *cloud, float resolution, int *representatives, int *new_size);

/* ---- depth image helpers (pwn_static.cpp:5-68) ----------------------------------------------- */
/* DepthImage_convert_16UC1_to_32FC1 followed by DepthImage_scale(step) on the device.
 * out has (rows/step) x (cols/step) floats.  step <= 1 skips the scaling. */
int nicp_depth_prepare(nicp_context *ctx, const uint16_t *raw, int rows, int cols, float depth_scale,
                       int step, float max_depth_cov, float *out);

/* ---- frame preparation --------------------------------------------------------------------- */
/* PinholePointProjector::unProject (pinholepointprojector.cpp:68-91): points only, compacted in
 * raster order.  iKRt from PinholePointProjector::_updateMatrices.  index may be NULL. */
int nicp_unproject(nicp_context *ctx, const float *depth, int rows, int cols, const float iKRt[16],
                   float min_distance, float max_distance, nicp_cloud *cloud, int *index);
/* PinholePointProjector::projectIntervals (pinholepointprojector.cpp:135-147) */
int nicp_project_intervals(nicp_context *ctx, const float *depth, const nicp_projector *proj,
                           float world_radius, int *interval);
/* DepthImageConverterIntegralImage::compute (depthimageconverterintegralimage.cpp:15-55):
 * unProject + projectIntervals + PointIntegralImage + StatsCalculatorIntegralImage +
 * Point/NormalInformationMatrixCalculator + Cloud::transformInPlace(sensor_offset).
 * index (rows*cols) may be NULL.  keep_stats != 0 also materialises pwn::Stats.
 * ASYNCHRONOUS when index is NULL: the call returns once the work is queued on the context's stream (the cloud is
 * consumed in stream order by every later call on this context).  A pageable `depth` has been staged by the time
 * the call returns; a PINNED `depth` is read by the copy engine later, so it must stay unchanged until the next
 * synchronous call on this context (or nicp_synchronize) returns.  With index != NULL the call is synchronous. */
int nicp_depth_to_cloud(nicp_context *ctx, const float *depth, const nicp_projector *proj,
                        const nicp_stats_params *sp, const float sensor_offset[16], int keep_stats,
                        nicp_cloud *cloud, int *index);
/* same, from a raw 16-bit image: convert (depth_scale) + DepthImage_scale(step) + the above;
 * proj describes the camera AFTER scaling (PwnMatcherBase::makeCloud, pwn_matcher_base.cpp:46-75).
 * Same asynchrony as nicp_depth_to_cloud; the raw image is uploaded on a second stream into one of two staging
 * images, so with pinned `raw` buffers the upload of frame i+1 overlaps the kernels of frame i. */
int nicp_raw_depth_to_cloud(nicp_context *ctx, const uint16_t *raw, int raw_rows, int raw_cols,
                            float depth_scale, int step, float max_depth_cov, const nicp_projector *proj,
                            const nicp_stats_params *sp, const float sensor_offset[16], int keep_stats,
                            nicp_cloud *cloud, int *index);
/* The same for n frames with one launch set per sub-batch of up to 8 frames (grid.z = frame): what a tracker's cloud
 * cache or a loop closer does frame by frame (pwn_tracker2/pwn_cloud_cache.cpp:60-102 -> PwnMatcherBase::makeCloud,
 * pwn_matcher_base.cpp:46-75) when it (re)builds the clouds of many frames.  One frame does not fill a B200 -- its two
 * order-preserving prefix-sum passes are bound by latency -- a batch does.  All frames share the raw size, step,
 * projector, statistics parameters and sensor offset; clouds[i] receives frame i (distinct clouds, capacity >= pixels).
 * Results are bit-identical to n calls of nicp_raw_depth_to_cloud.  ASYNCHRONOUS like it (no index images are returned);
 * pinned raw buffers must stay unchanged until the next synchronous call on this context returns. */
int nicp_raw_depth_to_cloud_batch(nicp_context *ctx, int n, const uint16_t *const *raws, int raw_rows, int raw_cols,
                                  float depth_scale, int step, float max_depth_cov, const nicp_projector *proj,
                                  const nicp_stats_params *sp, const float sensor_offset[16], int keep_stats,
                                  nicp_cloud *const *clouds);
/* ---- stage-level virtuals of the converter (SURVEY.md section 8b) ------------------------------------------------
 * StatsCalculatorIntegralImage::compute(normals, statsVector, points, indexImage) with the calculator's _intervalImage
 * (statscalculator.h:36, statscalculatorintegralimage.h:37 / .cpp:14-82): PointIntegralImage::compute over
 * (index_image, points), then per pixel the window statistics.  points4 = n x 4 floats; index_image / interval_image =
 * rows x cols (index -1 / interval -1 = skip).  Outputs (n entries each, any may be NULL): normals4 (w = 0), stats16
 * (column-major 4x4: eigenvectors + mean, identity where nothing was computed), eigenvalues3, n_points, curvature
 * (Stats::curvature(), stats.h:98-103). */
int nicp_stats_compute(nicp_context *ctx, const float *points4, int n, const int *index_image, const int *interval_image,
                       int rows, int cols, const nicp_stats_params *sp, float *normals4, float *stats16, float *eigenvalues3,
                       int *n_points, float *curvature);
/* PointInformationMatrixCalculator::compute / NormalInformationMatrixCalculator::compute(informationMatrix, statsVector,
 * imageNormals) (informationmatrixcalculator.h:83,123,158 / .cpp:9-58): 6 floats per point (upper triangle), zero where
 * the normal is zero.  Either output may be NULL. */
int nicp_information_compute(nicp_context *ctx, int n, const float *normals4, const float *stats16, const float *eigenvalues3,
                             const float *curvature, const nicp_stats_params *sp, float *omega_p6, float *omega_n6);
/* PointIntegralImage::compute (pointintegralimage.cpp:7-44) of the last nicp_depth_to_cloud call:
 * 10 channels per pixel, interleaved [rows][cols][10] = n,x,y,z,xx,xy,xz,yy,yz,zz (test hook) */
int nicp_last_integral_image(nicp_context *ctx, float *integral10);
int nicp_last_interval_image(nicp_context *ctx, int *interval);

/* ---- projection ---------------------------------------------------------------------------- */
/* PinholePointProjector::project (pinholepointprojector.cpp:33-66).  KRt from _updateMatrices. */
int nicp_project(nicp_context *ctx, const nicp_cloud *cloud, const float KRt[16], int rows, int cols,
                 float min_distance, float max_distance, int *index, float *depth);

/* ---- correspondence + linearisation (stage level) ----------------------------------------- */
/* CorrespondenceFinder::compute (correspondencefinder.cpp:20-118) fused with Linearizer::update
 * (linearizer.cpp:17-115) for the same T, given the two index images (host).  corr_image
 * (rows*cols, may be NULL) receives the accepted reference index per pixel or -1; H column-major. */
int nicp_correspond_linearize(nicp_context *ctx, const nicp_cloud *reference, const nicp_cloud *current,
                              const int *reference_index, const int *current_index, int rows, int cols,
                              const float T[16], const nicp_align_params *ap, float H[36], float b[6],
                              float *error, int *inliers, int *num_correspondences, int *corr_image);
/* Linearizer::update over an explicit correspondence list (n pairs of (referenceIndex, currentIndex)) */
int nicp_linearize(nicp_context *ctx, const nicp_cloud *reference, const nicp_cloud *current,
                   const int *correspondences, int n, const float T[16], const nicp_align_params *ap,
                   float H[36], float b[6], float *error, int *inliers);

/* ---- alignment ------------------------------------------------------------------------------ */
/* Aligner::align() (aligner.cpp:49-150): all iterations on the device, one synchronisation at the end. */
int nicp_align(nicp_context *ctx, const nicp_cloud *reference, const nicp_cloud *current,
               const nicp_projector *proj, const nicp_align_params *ap,
               const float reference_sensor_offset[16], const float current_sensor_offset[16],
               const float initial_guess[16], const nicp_prior *priors, int num_priors,
               float frame_inlier_depth_threshold, nicp_align_result *result);
/* state of the last nicp_align on this context (what CorrespondenceFinder / Linearizer expose after
 * align(), pwn_matcher_base.cpp:156-171): any pointer may be NULL.  correspondences receives
 * num_correspondences (referenceIndex, currentIndex) pairs in raster order; H/b are the
 * linearisation of _computeStatistics at the final T. */
int nicp_align_get_state(nicp_context *ctx, int *reference_index, float *reference_depth,
                         int *current_index, float *current_depth, int *correspondences,
                         float H[36], float b[6]);
/* per-iteration trace of the last nicp_align: T at the start of each outer iteration (16), H (36),
 * b (6), error, inliers, numCorrespondences = 61 floats per iteration (test hook) */
int nicp_align_get_trace(nicp_context *ctx, float *trace61, int max_iterations);

/* Batched alignment of n independent pairs (loop-closure candidate verification,
 * pwn_tracker2/pwn_closer.cpp:83-182).  initial_guesses = n x 16 floats.  Results of pair i are
 * identical to nicp_align on pair i.  (Priors per pair: nicp_align_batch_priors below.) */
int nicp_align_batch(nicp_context *ctx, int n, const nicp_cloud *const *references,
                     const nicp_cloud *const *currents, const nicp_projector *proj,
                     const nicp_align_params *ap, const float reference_sensor_offset[16],
                     const float current_sensor_offset[16], const float *initial_guesses,
                     float frame_inlier_depth_threshold, nicp_align_result *results);

/* The same with SE(3) priors per pair, as the trackers add them before every match (odometry / IMU priors,
 * pwn_tracker2/pwn_tracker.cpp:150-160 -> Aligner::addRelativePrior / addAbsolutePrior, aligner.cpp:97-108): pair i owns
 * priors[prior_offsets[i] .. prior_offsets[i + 1]) (prior_offsets has n + 1 entries, prior_offsets[0] = 0; NULL = no
 * priors).  Results of pair i are identical to nicp_align on pair i with its priors. */
int nicp_align_batch_priors(nicp_context *ctx, int n, const nicp_cloud *const *references,
                            const nicp_cloud *const *currents, const nicp_projector *proj,
                            const nicp_align_params *ap, const float reference_sensor_offset[16],
                            const float current_sensor_offset[16], const float *initial_guesses,
                            const nicp_prior *priors, const int *prior_offsets,
                            float frame_inlier_depth_threshold, nicp_align_result *results);

/* ---- multi-GPU: pair-wise sharding over the devices of ONE process (SURVEY.md section 8e) ---------------------------
 * The reference's loop closer walks the candidate pairs of a partition serially, building the clouds of both frames and
 * matching them (PwnCloser::processPartition, pwn_tracker2/pwn_closer.cpp:83-182).  Here the pair list is cut into
 * contiguous blocks, one per device (block g = pairs [g n / G, (g + 1) n / G): order the list so that pairs sharing a
 * current frame are adjacent); every device prepares the clouds of the frames its block references from the raw images
 * and aligns its block on its own stream, one worker thread and one context per device.  Pairs are independent, so there
 * is no data-path exchange; the records land in the caller's array.  A pair's record does not depend on the number of
 * devices, on the block it fell into or on its neighbours (same bits as nicp_align on that pair).
 * devices may name a GPU more than once (two workers sharing a device). */
typedef struct nicp_shard_pool nicp_shard_pool;
int nicp_shard_pool_create(const int *devices, int n_devices, nicp_shard_pool **pool);
void nicp_shard_pool_destroy(nicp_shard_pool *pool);
int nicp_shard_pool_size(const nicp_shard_pool *pool);
/* frames in, records out: raws[f] = raw 16-bit image of frame f (all raw_rows x raw_cols, converted like
 * nicp_raw_depth_to_cloud; sensor_offset is the sensor pose used for the frame preparation and for both sides of every
 * alignment, as PwnMatcherBase does), pair i = (reference_frame[i], current_frame[i]) with initial_guesses + 16 i (NULL:
 * identity).  Worker g takes pairs [g n / G, (g + 1) n / G) and walks them in windows: the longest runs of consecutive
 * pairs whose distinct frames fit in its frame cap, building only the frames a window needs and does not hold yet.  The
 * cap is max(2, 0.5 * device memory / (112 B * image pixels) / workers on that device), about 2 600 frames at 640 x 480 on
 * a 180 GB GPU, so a block of a closer's partition is one window; NICP_SHARD_FRAMES, read when the pool is created, lowers
 * it.  A worker keeps one cloud cache for this entry and nicp_multi_align_frames_sharded, which starts over when the image
 * size changes.  Arguments are checked before any worker starts (raw size, frame indices, null images); synchronous. */
int nicp_align_frames_sharded(nicp_shard_pool *pool, int n_frames, const uint16_t *const *raws, int raw_rows, int raw_cols,
                              float depth_scale, int step, float max_depth_cov, const nicp_projector *proj,
                              const nicp_stats_params *sp, const float sensor_offset[16], int n_pairs,
                              const int *reference_frame, const int *current_frame, const float *initial_guesses,
                              const nicp_align_params *ap, float frame_inlier_depth_threshold, nicp_align_result *results);

/* ---- MultiPointProjector (BASELINE config 5) -------------------------------------------------------- */
/* MultiPointProjector::computeImageSize (multipointprojector.cpp:7-18) */
void nicp_multi_image_size(const nicp_multi_projector *mp, int *rows, int *cols);
/* DepthImageConverterIntegralImage::compute with a MultiPointProjector: depth is the composite image */
int nicp_multi_depth_to_cloud(nicp_context *ctx, const float *depth, const nicp_multi_projector *mp,
                              const nicp_stats_params *sp, const float sensor_offset[16], int keep_stats,
                              nicp_cloud *cloud, int *index);
/* PointProjector::project (base z-buffer) of a MultiPointProjector whose rig pose is T */
int nicp_multi_project(nicp_context *ctx, const nicp_cloud *cloud, const nicp_multi_projector *mp, const float T[16],
                       int *index, float *depth);
/* Aligner::align() with a MultiPointProjector */
int nicp_multi_align(nicp_context *ctx, const nicp_cloud *reference, const nicp_cloud *current,
                     const nicp_multi_projector *mp, const nicp_align_params *ap,
                     const float reference_sensor_offset[16], const float current_sensor_offset[16],
                     const float initial_guess[16], const nicp_prior *priors, int num_priors,
                     float frame_inlier_depth_threshold, nicp_align_result *result);
/* Rig frames from raw 16-bit images, n frames at a time: the rig counterpart of nicp_raw_depth_to_cloud_batch.
 * raws[f * num_cameras + i] is camera i of frame f as the sensor delivers it, raw_rows[i] x raw_cols[i] (row = pixel v,
 * column = pixel u).  Each image is converted (depth_scale) and scaled (DepthImage_scale(step), in sensor orientation) like
 * nicp_raw_depth_to_cloud, then transposed into the composite image of nicp_multi_depth_to_cloud:
 *   composite rows = max over cameras of width_i, composite cols = sum of height_i,
 *   composite[u][colOff_i + v] = scaled image i at (v, u), camera i owning columns [colOff_i, colOff_i + height_i),
 *   rows [width_i, rows) of that block are empty (0).
 * width_i = mp->camera[i].rows and height_i = mp->camera[i].cols (addPointProjector(p, offset, width, height)); mp describes
 * the rig AFTER scaling, so raw_rows[i] / step must equal height_i and raw_cols[i] / step width_i.  Every frame's cloud is
 * bit-identical to nicp_multi_depth_to_cloud of that composite.  clouds[f] receives frame f (distinct clouds, capacity >=
 * composite pixels).  One launch set takes clamp(8 * 640 * 480 / composite pixels, 1, 8) frames (1 at 1280 x 3840), so its
 * scratch stays within that of 8 pinhole 640x480 frames.  ASYNCHRONOUS like nicp_raw_depth_to_cloud_batch (no index images are returned); pinned raw buffers
 * must stay unchanged until the next synchronous call on this context returns. */
int nicp_multi_raw_depth_to_cloud_batch(nicp_context *ctx, int n, const uint16_t *const *raws, const int *raw_rows,
                                        const int *raw_cols, float depth_scale, int step, float max_depth_cov,
                                        const nicp_multi_projector *mp, const nicp_stats_params *sp,
                                        const float sensor_offset[16], int keep_stats, nicp_cloud *const *clouds);
/* Batched rig alignment of n independent pairs (a rig loop closer verifying one frame against many candidates), with
 * priors per pair as in nicp_align_batch_priors (priors / prior_offsets may be NULL).  Record i is identical, byte for
 * byte, to nicp_multi_align on pair i with the same guess and priors.  A lock-step chunk holds at most
 * max(1, 256 * 640 * 480 / composite pixels) pairs (32 B of scratch per pixel and pair: 16 pairs at 1280 x 3840), or
 * NICP_BATCH_SLOTS when that is lower. */
int nicp_multi_align_batch(nicp_context *ctx, int n, const nicp_cloud *const *references,
                           const nicp_cloud *const *currents, const nicp_multi_projector *mp,
                           const nicp_align_params *ap, const float reference_sensor_offset[16],
                           const float current_sensor_offset[16], const float *initial_guesses,
                           const nicp_prior *priors, const int *prior_offsets,
                           float frame_inlier_depth_threshold, nicp_align_result *results);
/* The rig counterpart of nicp_align_frames_sharded: raw rig frames in, records out, over the workers of a shard pool.
 * raws[f * num_cameras + i] is camera i of frame f, raw_rows[i] x raw_cols[i] in every frame, as in
 * nicp_multi_raw_depth_to_cloud_batch; pair i = (reference_frame[i], current_frame[i]) with initial_guesses + 16 i (NULL:
 * identity) and priors as in nicp_multi_align_batch (priors / prior_offsets may be NULL); sensor_offset is the rig pose
 * used for the frame preparation and for both sides of every alignment.  Blocks, windows, frame cap and cloud cache are
 * those of nicp_align_frames_sharded, with the composite image: the cap is about 160 frames at 1280 x 3840 on a 180 GB
 * GPU (in current-major order the candidates stay resident and only the current frames rotate).
 * Record i is byte-identical to nicp_multi_align on the clouds nicp_multi_raw_depth_to_cloud_batch builds from its two
 * frames, whatever the device list, the workers per device or the cap.  Arguments are checked before any worker starts
 * (frame indices, null images, raw sizes, prior_offsets); synchronous. */
int nicp_multi_align_frames_sharded(nicp_shard_pool *pool, int n_frames, const uint16_t *const *raws, const int *raw_rows,
                                    const int *raw_cols, float depth_scale, int step, float max_depth_cov,
                                    const nicp_multi_projector *mp, const nicp_stats_params *sp,
                                    const float sensor_offset[16], int n_pairs, const int *reference_frame,
                                    const int *current_frame, const float *initial_guesses,
                                    const nicp_prior *priors, const int *prior_offsets,
                                    const nicp_align_params *ap, float frame_inlier_depth_threshold,
                                    nicp_align_result *results);

#ifdef __cplusplus
}
#endif
#endif

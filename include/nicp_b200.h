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
/* The rig counterpart of nicp_cloud_compute_gaussians; depth is the composite image the cloud was built from by
 * nicp_multi_depth_to_cloud / nicp_multi_raw_depth_to_cloud_batch; baseline, alpha: mp->num_cameras floats each (> 0).
 * The gaussian of a point of camera i at composite pixel (r, c), depth z, is child i's sensor model above at its pixel
 * (u, v) = (r, c - colOff_i), in the moments form: mean = the rig point (bit-identical to the cloud's point before the
 * sensor offset), covariance R_i (J diag(3, 3, alpha_i z^2 / (baseline_i fx_i + alpha_i z)) J^T) R_i^T with R_i the
 * rotation of sensor_offset[i] of the rig (skipped when that offset is the identity); then sensor_offset as above.  One
 * gaussian per point, in the cloud's point order.  This is the project's definition (DESIGN.md, known deviations), not
 * pinned to the reference's MultiPointProjector.  A depth image whose valid pixels differ in number from the cloud's
 * points is rejected with NICP_ERR_INVALID. */
int nicp_multi_cloud_compute_gaussians(nicp_context *ctx, nicp_cloud *cloud, const float *depth,
                                       const nicp_multi_projector *mp, const float *baseline, const float *alpha,
                                       const float sensor_offset[16]);
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
/* Local map from n raw pinhole frames in one call.  Frame i is prepared like nicp_raw_depth_to_cloud (keep_stats 0), gets
 * the sensor-model gaussians of nicp_cloud_compute_gaussians (baseline, alpha, sensor_offset) and is appended to `map` with
 * poses + 16 * i (column-major 4x4) like nicp_cloud_append, in frame order, behind the points the map already holds (with
 * or without gaussians).  Then, if merge_params != NULL, nicp_merge(map, proj, merge_transform, merge_params); then, if
 * voxel_resolution > 0, nicp_voxelize(map, voxel_resolution).  The map is byte-identical to that chain of calls.  Frames
 * are prepared in launch sets of up to 8 as in nicp_raw_depth_to_cloud_batch; the gaussians come from the set's device
 * depth images and each set is appended by one launch, with no host round trip per frame.  The frame clouds of one set
 * are scratch of the context, reused by the next set and the next call.
 * Outputs (each may be NULL): appended_size = points the frames added; new_size = the map's final size; collapsed
 * (nicp_merge) and representatives (nicp_voxelize) need room for map->capacity ints.  If the appended points do not fit,
 * the call returns NICP_ERR_INVALID with new_size = the size the map would need, and the map keeps its size and its points.
 * Synchronous. */
int nicp_raw_depth_to_local_map(nicp_context *ctx, int n, const uint16_t *const *raws, int raw_rows, int raw_cols,
                                float depth_scale, int step, float max_depth_cov, const nicp_projector *proj,
                                const nicp_stats_params *sp, const float sensor_offset[16], float baseline, float alpha,
                                const float *poses, const nicp_merge_params *merge_params,
                                const float merge_transform[16], float voxel_resolution, nicp_cloud *map,
                                int *appended_size, int *new_size, int *collapsed, int *representatives);
/* The rig counterpart of nicp_raw_depth_to_local_map: raws[f * num_cameras + i] is camera i of frame f, raw_rows /
 * raw_cols as in nicp_multi_raw_depth_to_cloud_batch; each frame gets the gaussians of nicp_multi_cloud_compute_gaussians
 * (baseline, alpha: one per camera, > 0).  The merge step (if merge_params != NULL) is nicp_merge(map, merge_proj,
 * merge_transform, merge_params) with a pinhole merge view (merge_proj and merge_transform are then required).  The map
 * is byte-identical to the chain of single calls (nicp_multi_raw_depth_to_cloud_batch of one frame,
 * nicp_multi_cloud_compute_gaussians, nicp_cloud_append, then nicp_merge and nicp_voxelize).  A launch set holds
 * clamp(8 * 640 * 480 / composite pixels, 1, 8) frames; the frame clouds of one set are scratch of the context.  Outputs,
 * a map too small and synchronisation as in nicp_raw_depth_to_local_map. */
int nicp_multi_raw_depth_to_local_map(nicp_context *ctx, int n, const uint16_t *const *raws, const int *raw_rows,
                                      const int *raw_cols, float depth_scale, int step, float max_depth_cov,
                                      const nicp_multi_projector *mp, const nicp_stats_params *sp,
                                      const float sensor_offset[16], const float *baseline, const float *alpha,
                                      const float *poses, const nicp_projector *merge_proj,
                                      const nicp_merge_params *merge_params, const float merge_transform[16],
                                      float voxel_resolution, nicp_cloud *map, int *appended_size, int *new_size,
                                      int *collapsed, int *representatives);
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
/* The dense tail of Aligner::_computeStatistics (aligner.cpp:172-198) on n caller-given linearisations (test hooks):
 * H = n x 36 (column-major 6x6), T = n x 16 (column-major 4x4) -> omega = n x 36, ratios = n x 2 (translational,
 * rotational eigen-ratio).  Every NaN among the outputs is the quiet NaN 0x7fc00000.
 * nicp_statistics_tail runs the kernel that finishes a batch's records on the device (it ends the state of the last
 * nicp_align: nicp_align_get_state / _get_trace fail until the next one); nicp_statistics_tail_host needs no context and
 * runs the host function that finishes a single nicp_align's record.  The two agree bit for bit. */
int nicp_statistics_tail(nicp_context *ctx, int n, const float *H, const float *T, float *omega, float *ratios);
int nicp_statistics_tail_host(int n, const float *H, const float *T, float *omega, float *ratios);

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
 * size changes; its clouds are reused as storage only, every call prepares the frames it references again (a frame store,
 * below, keeps them across calls).  Arguments are checked before any worker starts (raw size, frame indices, null images); synchronous. */
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

/* ---- frame store: loop-closure frames resident on a shard pool across calls -------------------------------------------
 * An incremental closer matches each new map node against candidates that earlier steps already used
 * (MapCloser::process -> PwnCloser::processPartition, pwn_tracker2/pwn_closer.cpp:83-182) and keeps their clouds between
 * steps (PwnCloudCache, pwn_tracker2/pwn_cloud_cache.cpp:60-102).  A frame store holds the raw frames of one pinhole camera
 * or one rig under caller-chosen 64-bit ids (e.g. BOSS node ids); each worker of the pool keeps the clouds of the frames its
 * pairs used, and a later call finds them there.
 *   - Records: record i of nicp_frame_store_align is byte-identical to nicp_align / nicp_multi_align, with the pair's guess
 *     and priors, on the clouds nicp_raw_depth_to_cloud_batch / nicp_multi_raw_depth_to_cloud_batch build from its two
 *     frames, whatever the device list, the workers per device, the frame cap, the store's history or what is resident.
 *   - Placement and windows: those of nicp_align_frames_sharded (worker g takes pairs [g n / G, (g + 1) n / G)), but each
 *     worker's slot table is keyed by frame id and persists across calls.  A window keeps the resident clouds it uses;
 *     missing frames go to empty slots first, then to new clouds while the worker holds fewer than its frame cap, then to
 *     the least recently used slots the window does not use.  The cap is that of the sharded entries (NICP_SHARD_FRAMES
 *     lowers it), applied per store and per worker.  The cloud cache of the sharded entries is separate: a worker holds up
 *     to the cap for those entries and up to the cap for each store, so several full caches on one GPU add up.
 *   - Lazily built: nicp_frame_store_add only copies the raw images to host memory; a frame is prepared the first time a
 *     window on some worker needs it, and again only after it was evicted there.  Keep the candidates of one current frame
 *     in the same order (e.g. by id) from call to call so that each worker keeps seeing the same slice of them.
 *   - Every argument is checked in the calling thread before any worker starts, and a rejected call changes nothing: null
 *     handles or arrays, an id added twice (in one call or already in the store), remove / align naming an id that is not
 *     in the store, bad prior_offsets.  A worker that fails mid-call leaves no slot claiming a frame it did not finish.
 *   - nicp_shard_pool_destroy releases the device clouds of the pool's stores; every later call on such a store except
 *     nicp_frame_store_destroy returns NICP_ERR_INVALID (nicp_frame_store_size returns -1).
 *   - A pool and its stores are used from one host thread at a time, like a context.  Calls are synchronous. */
typedef struct nicp_frame_store nicp_frame_store;
/* the frame description, fixed for the store's lifetime and validated like nicp_align_frames_sharded /
 * nicp_multi_align_frames_sharded validate theirs: raw size, depth_scale, step, max_depth_cov, projector (or rig),
 * statistics parameters and the sensor offset (NULL: identity) used for the preparation and both sides of every alignment */
int nicp_frame_store_create(nicp_shard_pool *pool, int raw_rows, int raw_cols, float depth_scale, int step,
                            float max_depth_cov, const nicp_projector *proj, const nicp_stats_params *sp,
                            const float sensor_offset[16], nicp_frame_store **store);
int nicp_multi_frame_store_create(nicp_shard_pool *pool, const int *raw_rows, const int *raw_cols, float depth_scale,
                                  int step, float max_depth_cov, const nicp_multi_projector *mp,
                                  const nicp_stats_params *sp, const float sensor_offset[16], nicp_frame_store **store);
void nicp_frame_store_destroy(nicp_frame_store *store);
/* copies n frames: frame f has id ids[f] and raw images raws[f * num_cameras + i] (one camera for a pinhole store), as in
 * nicp_multi_align_frames_sharded; the caller may free them on return.  Every image must be exactly raw_rows[i] x
 * raw_cols[i] (raw_rows x raw_cols for a pinhole store) as given when the store was created: the call copies that many
 * pixels from each pointer and cannot see the caller's size (capi.FrameStore.add checks the shapes) */
int nicp_frame_store_add(nicp_frame_store *store, int n, const long long *ids, const uint16_t *const *raws);
/* forgets n frames: their raw copies are freed and no worker serves their clouds again (an id added again later is
 * prepared from its new images) */
int nicp_frame_store_remove(nicp_frame_store *store, int n, const long long *ids);
/* frames in the store, -1 for a null store or one whose pool was destroyed */
int nicp_frame_store_size(const nicp_frame_store *store);
/* pair i = (reference_ids[i], current_ids[i]) with initial_guesses + 16 i (NULL: identity); priors / prior_offsets as in
 * nicp_multi_align_batch (may be NULL), for pinhole and rig stores alike */
int nicp_frame_store_align(nicp_frame_store *store, int n_pairs, const long long *reference_ids,
                           const long long *current_ids, const float *initial_guesses, const nicp_prior *priors,
                           const int *prior_offsets, const nicp_align_params *ap, float frame_inlier_depth_threshold,
                           nicp_align_result *results);
/* since the store was created, summed over the workers and over the windows of every call: frames a window prepared,
 * and frames a window found resident (either output may be NULL) */
int nicp_frame_store_counters(const nicp_frame_store *store, long long *frames_built, long long *frames_reused);

/* ---- batched keyframe tracking: many independent depth sequences on a shard pool ---------------------------------------
 * One sequence's poses depend on each other (PwnTracker::processFrame, pwn_tracker/pwn_tracker.cpp:106-282), but separate
 * sequences (offline odometry over a recorded dataset, many robots, a parameter sweep over one log) do not.  A tracker keeps
 * the keyframe state of S sequences resident on the workers of a pool; one step takes one frame of each listed sequence.
 *   - Semantics: each listed sequence does exactly what pwn::SequentialTracker::processFrame (include/pwn/tracker.h) does on
 *     that frame, with the tracker's sensor offset on every frame and setScale(step).  The cloud is prepared as
 *     nicp_raw_depth_to_cloud / nicp_multi_raw_depth_to_cloud_batch prepare it (keep_stats 0).  A sequence without a keyframe
 *     takes the cloud as its keyframe (keyT = globalT) and aligns nothing; its odometry is ignored.  Otherwise
 *     guess = keyT^-1 * globalT * odometry (then fixLastRow), and the keyframe (reference) is aligned against the new cloud
 *     (current): the record is byte-identical to nicp_align / nicp_multi_align with that guess, no priors and the sensor
 *     offset on both sides.  Then globalT = keyT * T if inliers > 0, else globalT * guess; the rotation is re-orthogonalised
 *     when the sequence's frame counter is a multiple of 50; fixLastRow; and the new cloud becomes the keyframe
 *     (keyT = globalT) when (float)inliers / (float)(rows * cols) < new_frame_inliers_fraction (composite pixels for a rig).
 *     The pose arithmetic is float32 in the operation order of include/pwn/compat.h, so it matches the C++ class bit for bit.
 *   - Placement and memory: sequence s lives on worker floor(s * G / S) for the tracker's lifetime and owns two device
 *     clouds there (keyframe and current frame), allocated at create; a keyframe switch swaps the two, nothing is copied.
 *     Creation fails with NICP_ERR_INVALID when a worker's sequences need more clouds (two each) than its frame cap (that of
 *     the sharded entries; NICP_SHARD_FRAMES lowers it).
 *   - One step: every argument is checked in the calling thread first (null arrays or images, a sequence outside [0, S) or
 *     listed twice, a destroyed pool).  Each worker with listed sequences makes one batched prep of their frames and one
 *     batched alignment of those that have a keyframe, in listed order, and is synchronised before the call returns.  The
 *     sequences' state is committed only after every worker succeeded: a rejected or failed step changes no sequence.  A
 *     record whose status is not NICP_OK fails the step with that status.
 *   - nicp_shard_pool_destroy releases the trackers' clouds; every later call on such a tracker except
 *     nicp_tracker_destroy returns NICP_ERR_INVALID (nicp_tracker_size returns -1).  Calls are synchronous; a pool and its
 *     trackers are used from one host thread at a time. */
typedef struct {
  float global_T[16];        /* SequentialTracker::globalT() after this frame */
  float relative_T[16];      /* lastRelative(): the aligner's T (identity when aligned = 0) */
  float guess[16];           /* initial guess the alignment started from, after fixLastRow (identity when aligned = 0) */
  int frame;                 /* frames this sequence had processed before this one (SequentialTracker::_counter) */
  int aligned;               /* 0 for a sequence's first frame after create / reset: nothing to align against */
  int keyframe;              /* lastWasKeyframe() */
  int num_keyframes;         /* numKeyframes() */
  nicp_align_result record;  /* the alignment's record; zeroed with status NICP_OK when aligned = 0 */
} nicp_track_result;

typedef struct nicp_tracker nicp_tracker;
/* the frame description, fixed for the tracker's lifetime and validated like nicp_frame_store_create /
 * nicp_multi_frame_store_create validate theirs (proj describes the camera after scaling, as in nicp_raw_depth_to_cloud;
 * sensor_offset NULL: identity); ap and frame_inlier_depth_threshold are those of every alignment */
int nicp_tracker_create(nicp_shard_pool *pool, int n_sequences, int raw_rows, int raw_cols, float depth_scale, int step,
                        float max_depth_cov, const nicp_projector *proj, const nicp_stats_params *sp,
                        const float sensor_offset[16], const nicp_align_params *ap, float frame_inlier_depth_threshold,
                        float new_frame_inliers_fraction, nicp_tracker **tracker);
int nicp_multi_tracker_create(nicp_shard_pool *pool, int n_sequences, const int *raw_rows, const int *raw_cols,
                              float depth_scale, int step, float max_depth_cov, const nicp_multi_projector *mp,
                              const nicp_stats_params *sp, const float sensor_offset[16], const nicp_align_params *ap,
                              float frame_inlier_depth_threshold, float new_frame_inliers_fraction, nicp_tracker **tracker);
void nicp_tracker_destroy(nicp_tracker *tracker);
/* n_sequences; -1 for a null tracker or one whose pool was destroyed */
int nicp_tracker_size(const nicp_tracker *tracker);
/* one frame for each of n distinct sequences: raws[k * num_cameras + i] is camera i of sequence sequences[k]'s frame (one
 * camera for a pinhole tracker), exactly the raw size given at create; odometry + 16 k is that frame's initialGuess
 * (NULL: identity); results[k] receives its result */
int nicp_tracker_step(nicp_tracker *tracker, int n, const int *sequences, const uint16_t *const *raws,
                      const float *odometry, nicp_track_result *results);
/* the listed sequences start over: no keyframe, global pose identity, counters 0 */
int nicp_tracker_reset(nicp_tracker *tracker, int n, const int *sequences);

#ifdef __cplusplus
}
#endif
#endif

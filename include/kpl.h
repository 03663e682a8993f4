/*
 * kpl.h -- C ABI of the B200-native Keypoint-Learning detection path (libkpl_b200.so).
 *
 * This is the drop-in boundary.  Every entry point replaces one piece of the reference's
 * pcl::keypoints::KeypointLearningDetector / TestDetector path; the citations (file:line) are
 * into the reference tree (CVLAB-Unibo/Keypoint-Learning).  Plain C, POD only, no torch / PCL /
 * OpenCV types.  All functions return KPL_OK (0) or a KPL_E_* code; the message of the last
 * failure on a context is available through kpl_last_error().  There is no CPU fallback: every
 * compute entry point fails with KPL_E_CUDA when no sm_100 device is usable.
 *
 * Threading: one context per host thread / per GPU; calls on one context must be serialised by
 * the caller (the reference detector is equally non-reentrant, include/KeypointLearning.h:180-204).
 * Ownership: input pointers are borrowed for the duration of the call; outputs are caller
 * allocated; the context owns all device memory and releases it in kpl_destroy().
 */
#ifndef KPL_B200_H_
#define KPL_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define KPL_API
#else
#define KPL_API __attribute__((visibility("default")))
#endif

typedef struct kpl_ctx kpl_ctx;

enum kpl_status {
    KPL_OK = 0,
    KPL_E_INVALID = 1,        /* bad argument / parameter combination                                   */
    KPL_E_FOREST = 2,         /* forest missing, unreadable or empty  (loadForest -> false, hpp:165-174)  */
    KPL_E_SIZE_MISMATCH = 3,  /* normals/points size mismatch         (initCompute -> false, hpp:149-153) */
    KPL_E_NONFINITE = 4,      /* non-finite input point (a point without a finite NORMAL is not an error:
                                 it gets no score, as in runForest hpp:277, see kpl_stats.n_unscored)      */
    KPL_E_VARCOUNT = 5,       /* annuli*bins != forest var_count                                          */
    KPL_E_CUDA = 6,           /* CUDA runtime failure or no usable device                                 */
    KPL_E_GRID = 7,           /* uniform grid would exceed 2^31-2 cells / point outside a forced grid     */
    KPL_E_NOMEM = 8,
    KPL_E_IO = 9,
    KPL_E_UNSUPPORTED = 10,
    KPL_E_NCCL = 11,          /* NCCL missing (libnccl.so.2 not loadable) or a collective failed              */
    KPL_E_HALO = 12           /* slab-sharded call: a k-NN normal that an owned point depends on was clipped
                                 by the slab edge -- widen kpl_slab_plan.normal_support_cells                */
};

enum kpl_normals_mode {
    KPL_NORMALS_GIVEN = 0,   /* setNormals() was called                      (KeypointLearning.h:108-109)       */
    KPL_NORMALS_KNN = 1,     /* pcl::NormalEstimation::setKSearch(k)         (main_test_detector.cpp:162-169)    */
    KPL_NORMALS_RADIUS = 2   /* NormalEstimation::setRadiusSearch(r_feat)    (impl/KeypointLearning.hpp:130-137) */
};

/* Per-point roles for slab-sharded clouds (no counterpart in the reference, which is single process).  kpl_detect* with a
 * role array refuses draws-remove NMS (KPL_E_UNSUPPORTED): such a caller drives one slab by itself and cannot see the
 * neighbours' decisions its own depend on; the kpl_shard_* entry points exchange them. */
enum kpl_role { KPL_ROLE_HALO = 0, KPL_ROLE_SCORE = 1, KPL_ROLE_OWNED = 3 };

/* Mirrors the detector's setters (include/KeypointLearning.h:81-90,102-155) and the TestDetector
 * command line (src/main_test_detector.cpp:53-91,105-106). */
typedef struct kpl_params {
    float radius_features;    /* setRadiusSearch          default 20   (main_test_detector.cpp:65)   */
    float radius_nms;         /* setNonMaxRadius          default 4    (:66)                         */
    double threshold;         /* setPredictionThreshold   default (double)0.85f (:67)                */
    int32_t n_annulus;        /* setNAnnulus              default 5    (:105)                        */
    int32_t n_bins;           /* setNBins                 default 10   (:106)                        */
    int32_t non_maxima;       /* setNonMaxima             default 1                                  */
    int32_t draws_remove;     /* setNonMaximaDrawsRemove  default 0 in TestDetector (:128)           */
    float draws_threshold;    /* setNonMaximaDrawsThreshold (uninitialised in the reference; 0 here) */
    int32_t normals_mode;     /* enum kpl_normals_mode, used when no normals are passed              */
    int32_t k_normals;        /* 10 (main_test_detector.cpp:167)                                     */
    float viewpoint[3];       /* PCD VIEWPOINT / sensor_origin_, (0,0,0)                             */
    int32_t flip_normals;     /* --flipNormals (:173-179), applied to normals computed here          */
    int32_t cells_per_radius; /* grid resolution: cell = r_feat*(1+2^-20)/cells_per_radius, default 4 */
    int32_t grid_forced;      /* 1: use the grid below (slab of a larger cloud): a point's cell is    */
    double grid_origin[3];    /*    floor((v - grid_origin)/cell) - grid_offset, which must lie in     */
    int32_t grid_dims[3];     /*    [0, grid_dims); origin is the GLOBAL one so keys order globally    */
    int32_t grid_offset[3];
    int32_t slab_interior_lo; /* forced grid only: 1 = the cloud continues beyond the low / high x face of the   */
    int32_t slab_interior_hi; /*    local grid (a slab of a larger cloud): a k-NN normal search that would have   */
    int32_t slab_guard_cells; /*    to look beyond such a face fails with KPL_E_HALO, except for points in the    */
                              /*    outermost slab_guard_cells columns at that face (nothing kept depends on them) */
    int32_t slab_owned_lo;    /* forced grid only: the local columns [lo, hi) hold every point with a scoring role    */
    int32_t slab_owned_hi;    /*    (hi > lo; 0,0 = not stated).  A hint kept for ABI stability: the feature kernel's    */
                              /*    query list is built from the roles themselves, unscored points get no lanes at all   */
    int32_t uniform_sampling_centre; /* kpl_uniform_sample: 0 = PCL 1.8.0's literal rule (closest to the voxel INDEX vector taken as
                                        a point), 1 = closest to the voxel centre                                        */
    int32_t eigen32_normalize;/* per-annulus row.normalize() (hpp:360-365): 0 = divide by the norm (Eigen >= 3.3, default),   */
                              /*    1 = multiply by 1/norm (Eigen 3.2.x DenseBase::operator/=); <= 1 ulp per feature       */
    int32_t report_fragile;   /* 1: flag the points with a near-split forest decision (kpl_stats.n_fragile_points,
                                 kpl_fetch_u8 "fragile"); costs ~2 % of the detection, default 0                   */
} kpl_params;

/* Device-time breakdown of the last detect call (CUDA events on the context stream), ms. */
typedef struct kpl_timings {
    float grid_ms, normals_ms, features_ms, forest_ms, nms_ms, total_ms;
} kpl_timings;

/* Exact work counters of the last detect call (used for the roofline byte model, SURVEY.md 8d). */
typedef struct kpl_stats {
    int64_t n_points;         /* points in the call                                   */
    int64_t n_scored;         /* points that received a score                         */
    int64_t feature_pairs;    /* sum over scored points of voting neighbours (self excluded) */
    int64_t candidate_pairs;  /* distance tests executed by the feature kernel        */
    int64_t n_above_threshold;
    int64_t n_keypoints;
    int64_t grid_cells;
    int32_t grid_dims[3];
    int32_t kernel_launches;  /* kernels launched by the last call                    */
    double grid_origin[3];
    double grid_cell;
    int32_t fast_math;        /* 1: the self-tested FMA-corrected sqrt/div sequences were used (bit-identical) */
    int32_t nms_rounds;       /* draws-remove NMS: resolution rounds of the last call (one host synchronisation each); 0 without */
    int64_t n_unscored;       /* points without a finite normal: score NaN, never a keypoint (hpp:277)        */
    int64_t n_near_threshold; /* scored points with |score - threshold| <= 1e-5: the decisions a 1e-5 score
                                 difference against another implementation could flip                         */
    int64_t n_fragile_points; /* (kpl_params.report_fragile) scored points for which at least one split decided by forest_->predict
                                 (hpp:281) had |x[var] - thr| <= 1e-5: a feature difference of the tolerated
                                 size sends that tree the other way and moves the score by 1/ntrees            */
    int32_t host_syncs;       /* cudaStreamSynchronize calls the last call made                               */
    int32_t n_views;          /* kpl_detect_batch(_forests): views in the call, frames for the organized batch (1 otherwise) */
} kpl_stats;

/* ---- lifetime ------------------------------------------------------------------------------- */
KPL_API int kpl_create(int device, kpl_ctx** out);            /* new KeypointLearningDetector (main_test_detector.cpp:123) */
KPL_API void kpl_destroy(kpl_ctx* ctx);                       /* ~KeypointLearningDetector   (KeypointLearning.h:93-97)    */
KPL_API const char* kpl_last_error(const kpl_ctx* ctx);
KPL_API const char* kpl_version(void);
KPL_API int kpl_device_count(void);                           /* usable (compute capability 10.x) devices; 0 without one */
/* Run on a caller-owned cudaStream_t.  NULL selects the context's own NON-BLOCKING stream, which is not ordered
 * after work on the legacy default stream: a caller working on the default stream passes cudaStreamLegacy. */
KPL_API int kpl_set_stream(kpl_ctx* ctx, void* cuda_stream);

/* ---- parameters ----------------------------------------------------------------------------- */
KPL_API int kpl_params_default(kpl_params* p);                /* ctor defaults + TestDetector values                        */
KPL_API int kpl_set_params(kpl_ctx* ctx, const kpl_params* p);
KPL_API int kpl_get_params(const kpl_ctx* ctx, kpl_params* p);

/* ---- forest --------------------------------------------------------------------------------- */
/* loadForest(path): opencv_ml_rtrees YAML or YAML.gz -> flat device arrays (impl/KeypointLearning.hpp:159-176). */
KPL_API int kpl_load_forest(kpl_ctx* ctx, const char* path);
/* Same from already-flattened host arrays: node i is a leaf iff var[i] < 0; go left iff x[var] <= thr. */
KPL_API int kpl_set_forest(kpl_ctx* ctx, int32_t ntrees, int32_t nnodes, const int32_t* roots, const int32_t* var,
                           const float* thr, const int32_t* left, const int32_t* right, const float* value,
                           int32_t var_count);
KPL_API int kpl_forest_info(const kpl_ctx* ctx, int32_t* ntrees, int32_t* nnodes, int32_t* var_count, int32_t* max_depth);

/* ---- a SET of forests scored from one feature pass (kpl_detect_forests) ---------------------------- */
/* The forest set holds forest 0 -- the one kpl_load_forest / kpl_set_forest install, which also drop every other forest --
 * and up to KPL_MAX_FORESTS - 1 forests appended by kpl_add_forest(_arrays) as forests 1, 2, ...; *index_out (may be NULL)
 * receives the new forest's index.  Adding needs forest 0 (KPL_E_FOREST without it) and fails with KPL_E_INVALID once the
 * set is full; a failed add leaves the set as it was.  kpl_forest_info keeps describing forest 0, and every entry point
 * other than kpl_detect_forests, kpl_detect_batch_forests and kpl_detect_batch_organized_forests (and their _device
 * variants) scores with forest 0 only, whatever else is loaded. */
#define KPL_MAX_FORESTS 16
KPL_API int kpl_add_forest(kpl_ctx* ctx, const char* path, int32_t* index_out);
KPL_API int kpl_add_forest_arrays(kpl_ctx* ctx, int32_t ntrees, int32_t nnodes, const int32_t* roots, const int32_t* var,
                                  const float* thr, const int32_t* left, const int32_t* right, const float* value,
                                  int32_t var_count, int32_t* index_out);
KPL_API int kpl_forest_count(const kpl_ctx* ctx, int32_t* count_out);

/* ---- the hot path, host buffers (what detector->compute() binds to) --------------------------- */
/* xyz: n points, 3 floats each at xyz_stride bytes (16 = pcl::PointXYZ, 12 = packed).
 * normals: NULL (estimate per params.normals_mode) or n normals, 3 floats each at normals_stride bytes
 *          (32 = pcl::Normal).  role: NULL or n bytes of enum kpl_role.
 * scores_out: NULL or n floats (forest response, impl/KeypointLearning.hpp:287; NaN for unscored roles).
 * kp_idx_out: capacity n int32, ascending indices of the keypoints (keypoints_indices_, hpp:252-253).  */
KPL_API int kpl_detect(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, const float* normals, int32_t normals_stride,
                       const uint8_t* role, int64_t n, float* scores_out, int32_t* kp_idx_out, int64_t* n_kp_out);

/* The same, also filling the keypoint CLOUD detectKeypoints returns (hpp:246-253): kp_xyzi_out (NULL or capacity 4*n floats)
 * receives x, y, z of each keypoint and its response as the fourth float, in the order of kp_idx_out. */
KPL_API int kpl_detect_xyzi(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, const float* normals, int32_t normals_stride,
                            const uint8_t* role, int64_t n, float* scores_out, int32_t* kp_idx_out, float* kp_xyzi_out,
                            int64_t* n_kp_out);

/* pcl::NormalEstimation::compute as TestDetector uses it (main_test_detector.cpp:162-169):
 * normals_out = n x (nx, ny, nz, curvature). Mode / k / viewpoint / flip come from the params. */
KPL_API int kpl_normals(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, int64_t n, float* normals_out);

/* The normals KeypointLearningDetector::initCompute estimates itself for an ORGANIZED surface when none were set
 * (impl/KeypointLearning.hpp:138-145): pcl::IntegralImageNormalEstimation, SIMPLE_3D_GRADIENT, setNormalSmoothingSize
 * (smoothing_size; the reference passes 5.0).  xyz: height x width points in row-major order, NaN = no measurement.
 * normals_out = n x (nx, ny, nz, curvature = NaN), NaN where PCL leaves the normal undefined (image border, depth
 * discontinuities, NaN points).  Viewpoint from the params. */
KPL_API int kpl_normals_organized(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, int32_t width, int32_t height,
                                  float smoothing_size, float* normals_out);

/* pcl::UniformSampling as TestDetector's --subSampling uses it (main_test_detector.cpp:145-157): one point
 * per leaf-sized voxel -- PCL 1.8.0 keeps the one closest to the voxel's integer index vector (sic; see
 * kpl_params.uniform_sampling_centre), ties: lower index.  idx_out (capacity n) receives the ascending original
 * indices of the survivors, *m_out their number. */
KPL_API int kpl_uniform_sample(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, int64_t n, float leaf,
                               int32_t* idx_out, int64_t* m_out);

/* computePointsForTrainingFeatures (impl/KeypointLearning.hpp:299-318): rows of A*B floats for the
 * m given point indices (NULL: all points, m == n). */
KPL_API int kpl_features(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, const float* normals, int32_t normals_stride,
                         int64_t n, const int32_t* indices, int64_t m, float* features_out);

/* pcl::KdTreeFLANN::nearestKSearch(point, 1, ...) as TrainDetector snaps its positive / negative samples onto
 * cloud indices before computePointsForTrainingFeatures (src/main_train_detector.cpp:419-436): for each of the m
 * query points (3 floats at q_stride bytes) the index of the nearest cloud point (ties: lower index) and,
 * when d2_out != NULL, the squared distance. */
KPL_API int kpl_nearest(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, int64_t n, const float* queries, int32_t q_stride,
                        int64_t m, int32_t* idx_out, float* d2_out);

/* searchForNeighbors / tree_->radiusSearch semantics (hpp:213,334): per point the number of
 * neighbours with d2 < (float)(r*r) (self included) and the wrapping 64-bit sum of
 * (index+1)*0x9E3779B97F4A7C15 over them; either output may be NULL. */
KPL_API int kpl_radius_stats(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, int64_t n, double radius,
                             int32_t* counts_out, uint64_t* hash_out);
/* Explicit neighbour lists (ascending index) of m query points; two-call protocol:
 * indices_out == NULL fills offsets_out[m+1] only. */
KPL_API int kpl_radius_neighbors(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, int64_t n, double radius,
                                 const int32_t* queries, int64_t m, int64_t* offsets_out, int32_t* indices_out);

/* ---- the hot path, device-resident buffers (inputs already in HBM; outputs stay there) -------- */
/* d_xyz4: n float4 (x,y,z,*).  d_normals4: NULL or n float4 (nx,ny,nz,*).  d_role: NULL or n bytes.
 * d_scores: NULL or n floats.  d_kp_idx: n int32.  The call enqueues on the context stream and
 * synchronises once at the end to return n_kp. */
KPL_API int kpl_detect_device(kpl_ctx* ctx, const void* d_xyz4, const void* d_normals4, const void* d_role, int64_t n,
                              void* d_scores, void* d_kp_idx, int64_t* n_kp_out);

/* ---- one cloud, every forest of the set (several descriptors' forests, forest sweeps) ---------------- */
/* The K forests of the set (kpl_forest_count) score one cloud from ONE feature pass: grid, normals and the annuli x bins
 * histograms are computed once, and the feature kernel walks all K forests from each histogram.  Forest k's results are
 * bit-identical to kpl_detect on the same cloud with only forest k loaded and params.threshold = thresholds[k]
 * (thresholds NULL: params.threshold for every forest; compared in double, hpp:207).  Inputs as in kpl_detect, without a
 * role array; the grid follows the params as in kpl_detect (a forced grid included).  Outputs are forest-major:
 * scores_out: NULL or K*n floats, forest k's at k*n.  kp_idx_out (capacity K*n): ascending point indices per forest;
 * kp_offsets_out[K + 1]: forest k's keypoints are kp_idx_out[kp_offsets_out[k] .. kp_offsets_out[k+1]).
 * Every forest must match annuli*bins (var_count, and no split beyond it): KPL_E_VARCOUNT names the forest.  K*n must not
 * exceed 2 147 483 000.  kpl_stats: feature_pairs, candidate_pairs and n_scored count the one feature pass;
 * n_above_threshold, n_near_threshold, n_keypoints, n_fragile_points and nms_rounds are sums over the forests.  With
 * report_fragile, kpl_fetch_u8("fragile") returns K*n bytes, forest-major.  Host round trips: those of kpl_detect_device
 * whatever K is (plus one per draws-remove round of each forest, plus one for the results). */
KPL_API int kpl_detect_forests(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, const float* normals, int32_t normals_stride,
                               int64_t n, const double* thresholds, float* scores_out, int32_t* kp_idx_out, int64_t* kp_offsets_out);
/* Device-resident cloud: d_scores NULL or K*n floats, d_kp_idx K*n int32, d_kp_offsets K + 1 int64, all on the device
 * (thresholds stays a HOST array of K doubles or NULL); *n_kp_out = keypoints of all forests. */
KPL_API int kpl_detect_forests_device(kpl_ctx* ctx, const void* d_xyz4, const void* d_normals4, int64_t n, const double* thresholds,
                                      void* d_scores, void* d_kp_idx, void* d_kp_offsets, int64_t* n_kp_out);

/* ---- a batch of independent views in one pass (BASELINE.json configs[4]) ------------------------ */
/* TestDetector handles one view per process run (main_test_detector.cpp:142-187); a caller with many small views
 * (a 200 k-point view is ~1.5 waves of the feature kernel) passes them CONCATENATED: view v is the points
 * [view_offsets[v], view_offsets[v+1]) of xyz (and of normals when given).  Every view is processed exactly as a
 * kpl_detect call on it alone would (own bounding box, own canonical grid and accumulation order: bit-identical
 * scores and keypoints), but all views share one stacked grid, one launch per stage and one set of host round trips.
 * Draws-remove NMS included: no r_nms neighbourhood spans two views and every view keeps its own index order, so the
 * resolution rounds over the stacked grid decide all views at once (one host round trip per round for the whole batch).
 * scores_out: NULL or n floats.  kp_idx_out (capacity n): VIEW-LOCAL keypoint indices, view after view, ascending
 * inside a view; kp_offsets_out[n_views + 1]: view v's keypoints are kp_idx_out[kp_offsets_out[v] .. kp_offsets_out[v+1]). */
KPL_API int kpl_detect_batch(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, const float* normals, int32_t normals_stride,
                             const int64_t* view_offsets, int32_t n_views, float* scores_out, int32_t* kp_idx_out,
                             int64_t* kp_offsets_out);
/* Same with device-resident clouds; view_offsets stays a HOST array, d_kp_offsets is n_views + 1 int64 on the device. */
KPL_API int kpl_detect_batch_device(kpl_ctx* ctx, const void* d_xyz4, const void* d_normals4, const int64_t* view_offsets,
                                    int32_t n_views, void* d_scores, void* d_kp_idx, void* d_kp_offsets, int64_t* n_kp_out);
/* Every forest of the set over a batch of views (evaluating several descriptors' forests over a dataset of views): one
 * stacked grid, one normal estimation and one feature pass whose tail walks the K forests (kpl_forest_count), then each
 * forest's NMS.  For forest k and view v the scores (compared as bits) and keypoints are those of kpl_detect_batch on
 * the same views with only forest k loaded and params.threshold = thresholds[k] (thresholds: NULL or K doubles on the
 * host, as in kpl_detect_forests).  Outputs are forest-major, then view-major: scores_out NULL or K*n floats, forest k's
 * at k*n in concatenated point order; kp_idx_out (capacity K*n): VIEW-LOCAL indices, ascending within a range;
 * kp_offsets_out[K*n_views + 1]: the range of (k, v) is kp_idx_out[kp_offsets_out[k*n_views + v] .. [k*n_views + v + 1]).
 * Refusals as kpl_detect_batch, plus those of kpl_detect_forests (KPL_E_VARCOUNT names the forest; K*n above
 * 2 147 483 000 is KPL_E_INVALID before the device is touched).  kpl_stats as kpl_detect_forests, with n_views = n_views;
 * with report_fragile, kpl_fetch_u8("fragile") returns K*n bytes, forest-major.  Host round trips: those of
 * kpl_detect_batch(_device) whatever K is (plus one per draws-remove round of each forest); kernel launches: K - 1 more
 * (one NMS per further forest).  K = 1 is kpl_detect_batch. */
KPL_API int kpl_detect_batch_forests(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, const float* normals, int32_t normals_stride,
                                     const int64_t* view_offsets, int32_t n_views, const double* thresholds,
                                     float* scores_out, int32_t* kp_idx_out, int64_t* kp_offsets_out);
/* Device-resident views: d_scores NULL or K*n floats, d_kp_idx K*n int32, d_kp_offsets K*n_views + 1 int64, all on the
 * device; view_offsets and thresholds stay HOST arrays.  *n_kp_out = keypoints of all forests and views. */
KPL_API int kpl_detect_batch_forests_device(kpl_ctx* ctx, const void* d_xyz4, const void* d_normals4, const int64_t* view_offsets,
                                            int32_t n_views, const double* thresholds, void* d_scores, void* d_kp_idx,
                                            void* d_kp_offsets, int64_t* n_kp_out);

/* ---- a batch of ORGANIZED frames of one size (depth-camera streams; the 2.5-D views of BASELINE.json configs[4]) ---- */
/* n_frames organized frames of width x height points each, row-major, frame after frame (NaN = no measurement); xyz at
 * xyz_stride bytes per point.
 * normals: NULL -> pcl::IntegralImageNormalEstimation(SIMPLE_3D_GRADIENT, smoothing_size) per frame (hpp:138-145, as
 *          kpl_normals_organized), flipped towards viewpoints[3f..3f+2] (viewpoints NULL: params.viewpoint for every
 *          frame); else the caller's per-pixel normals at normals_stride bytes (viewpoints ignored).
 * The points with finite x, y, z (pcl::isFinite) of each frame are detected as kpl_detect would detect them alone, in
 * ascending pixel order: the results of every frame are bit-identical to the single-frame organized path.  normals_mode
 * and flip_normals are ignored, as on that path.  The integral images of up to 256 MiB of frames ((W+1)(H+1)*24 B per
 * frame) are built per launch; a larger batch runs in chunks on the stream, without a host round trip between them.
 * scores_out: NULL or n_frames*width*height floats in pixel order (NaN: non-finite pixel or no finite normal).
 * kp_idx_out (capacity n_frames*width*height): FRAME-LOCAL pixel indices r*width + c, ascending within a frame;
 * kp_offsets_out[n_frames + 1]: frame f's keypoints are kp_idx_out[kp_offsets_out[f] .. kp_offsets_out[f+1]).  A frame
 * without a finite point gets an empty range; a batch without any returns KPL_OK and no keypoint.
 * kpl_stats describe the detection over the finite points (n_points = their number, n_views = n_frames); in kpl_timings
 * normals_ms includes the integral images and the compaction, total_ms covers the whole call.  kpl_fetch("normals")
 * then returns the normals of the finite points, frame after frame.  Host round trips: one for the per-frame finite
 * counts plus those of kpl_detect_batch_device (plus one for the results).
 * KPL_E_INVALID: width, height or n_frames < 1, more than 2 147 483 000 points, a smoothing size that is not finite and
 * > 0, a bad stride, a NULL input or output, a forced grid in the params.  KPL_E_FOREST without a forest. */
KPL_API int kpl_detect_batch_organized(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, const float* normals,
                                       int32_t normals_stride, int32_t width, int32_t height, int32_t n_frames,
                                       float smoothing_size, const float* viewpoints, float* scores_out,
                                       int32_t* kp_idx_out, int64_t* kp_offsets_out);
/* Device-resident frames (float4 per pixel); viewpoints stay a HOST array; d_scores: NULL or n_frames*width*height
 * floats; d_kp_idx: n_frames*width*height int32; d_kp_offsets: n_frames + 1 int64.  The keypoint offsets are computed on
 * the device: no round trip beyond those of kpl_detect_batch_device and the per-frame finite counts. */
KPL_API int kpl_detect_batch_organized_device(kpl_ctx* ctx, const void* d_xyz4, const void* d_normals4, int32_t width,
                                              int32_t height, int32_t n_frames, float smoothing_size,
                                              const float* viewpoints, void* d_scores, void* d_kp_idx,
                                              void* d_kp_offsets, int64_t* n_kp_out);
/* Every forest of the set over a batch of organized frames, from one feature pass (as kpl_detect_batch_forests).  For
 * forest k and frame f the scores (as bits, NaN payloads included) and keypoints are those of kpl_detect_batch_organized
 * with only forest k loaded and params.threshold = thresholds[k] (NULL or K doubles on the host).  Forest-major, then
 * frame-major: scores_out NULL or K*n_frames*width*height floats in pixel order, forest k's at k*n_frames*width*height
 * (NaN on non-finite pixels in every slice); kp_idx_out (capacity K*n_frames*width*height): FRAME-LOCAL pixel indices,
 * ascending within a range; kp_offsets_out[K*n_frames + 1]: the range of (k, f) is [kp_offsets_out[k*n_frames + f],
 * kp_offsets_out[k*n_frames + f + 1]).  A frame without a finite point gets an empty range in every forest; a batch
 * without any returns KPL_OK, K*n_frames + 1 zero offsets and all-NaN scores.  Refusals as kpl_detect_batch_organized
 * plus those of kpl_detect_forests (K*n_frames*width*height above 2 147 483 000: KPL_E_INVALID before the device is
 * touched).  kpl_stats as kpl_detect_forests over the finite points, n_views = n_frames; with report_fragile,
 * kpl_fetch_u8("fragile") returns K x (finite points) bytes, forest-major.  Host round trips: those of
 * kpl_detect_batch_organized(_device) whatever K is (plus one per draws-remove round of each forest); kernel launches:
 * K - 1 more.  K = 1 is kpl_detect_batch_organized. */
KPL_API int kpl_detect_batch_organized_forests(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, const float* normals,
                                               int32_t normals_stride, int32_t width, int32_t height, int32_t n_frames,
                                               float smoothing_size, const float* viewpoints, const double* thresholds,
                                               float* scores_out, int32_t* kp_idx_out, int64_t* kp_offsets_out);
/* Device-resident frames; viewpoints and thresholds stay HOST arrays; d_scores NULL or K*n_frames*width*height floats,
 * d_kp_idx K*n_frames*width*height int32, d_kp_offsets K*n_frames + 1 int64, all on the device. */
KPL_API int kpl_detect_batch_organized_forests_device(kpl_ctx* ctx, const void* d_xyz4, const void* d_normals4, int32_t width,
                                                      int32_t height, int32_t n_frames, float smoothing_size,
                                                      const float* viewpoints, const double* thresholds, void* d_scores,
                                                      void* d_kp_idx, void* d_kp_offsets, int64_t* n_kp_out);

/* ---- ONE large cloud over the GPUs of a node: x slabs + halo over NCCL (BASELINE.json configs[3]) ---------- */
/* The reference is a single process (main_test_detector.cpp:123-187 drives one detector); this is the layer a
 * multi-GPU driver binds to.  The cloud is cut along x at CELL-COLUMN boundaries of the canonical grid of the WHOLE
 * cloud; rank r owns the columns [cuts[r], cuts[r+1]).  Per detection every rank
 *   1. sends its boundary strips (halo = reach(radiusFeatures) + normal_support_cells columns, 16 B per point, 32 B
 *      with caller normals) to its two neighbours and receives theirs                      [ncclSend/ncclRecv]
 *   2. builds the grid of [left halo | owned | right halo] with the GLOBAL origin (same cell keys, hence the same
 *      accumulation order, hence bit-identical floats as the single-GPU run), estimates normals for all of it (unless
 *      the caller gave them: kpl_shard_set_slab_normals) and scores the points it OWNS -- every point of the cloud is
 *      scored exactly once
 *   3. exchanges the 4-byte scores of the strips, so that NMS sees the neighbours' scores  [ncclSend/ncclRecv]
 *   4. runs threshold + NMS for its owned points; rank 0 gathers the ascending GLOBAL keypoint index list.
 * A k-NN normal search that the slab edge would clip fails the call on every rank with KPL_E_HALO (widen
 * normal_support_cells); with caller normals nothing is estimated, so this cannot happen and a plan with
 * normal_support_cells = 0 (halo = max(reach_feat, reach_nms)) is the one to use.  draws-remove NMS: every rank classifies and decides its OWNED points only; the states of the
 * strip points (1 B per point) go to the neighbours after the classification and after every resolution round, and all
 * ranks stop on the same global count of undecided candidates -- one host synchronisation per round
 * (kpl_stats.nms_rounds).  The result is the single-GPU one. */
#define KPL_MAX_RANKS 64
typedef struct kpl_slab_plan {
    double origin[3];              /* grid origin = bounding-box minimum of the whole cloud                        */
    double cell;                   /* r_feat * (1 + 2^-20) / cells_per_radius                                       */
    int32_t dims[3];               /* grid dimensions of the whole cloud                                            */
    int32_t world;                 /* number of slabs / ranks                                                       */
    int32_t reach_feat, reach_nms; /* search reach of the two radii in cells                                        */
    int32_t normal_support_cells;  /* columns of k-NN support beyond reach_feat                                     */
    int32_t halo;                  /* max(reach_feat + normal_support_cells, reach_nms) columns per interior side   */
    int32_t cuts[KPL_MAX_RANKS + 1];
    int64_t n_points;
    double cost[KPL_MAX_RANKS];    /* modelled cost of each rank (neighbour pairs + per-point work), for reports    */
} kpl_slab_plan;

typedef struct kpl_shard kpl_shard;

typedef struct kpl_shard_info {
    int64_t n_owned, n_left, n_right;     /* points owned / received from the left / right neighbour              */
    int64_t send_left, send_right;        /* points sent to the neighbours per detection                          */
    int64_t halo_bytes;                   /* bytes this rank sends per detection (positions + scores, + normals when given) */
    int32_t local_dims[3], local_offset[3];
    int32_t rank, world;
    float exchange_ms;                    /* device time of the two exchanges of the last detection               */
    float gather_ms;                      /* device time of the keypoint gather + sort (rank 0)                   */
} kpl_shard_info;

/* Host only (no GPU needed): balanced cuts for `world` slabs.  The cost of a rank is modelled from the cloud itself:
 * neighbour pairs of the points it owns (cell histogram convolved with the search box) plus the per-point work of
 * everything it holds including the halo.  Fails with KPL_E_INVALID when the grid has too few columns for `world`
 * slabs of at least `halo` columns. */
KPL_API int kpl_slab_plan_make(const float* xyz, int32_t xyz_stride, int64_t n, const kpl_params* p, int32_t world,
                               int32_t normal_support_cells, kpl_slab_plan* out);
/* Host only: ascending indices of the points rank `rank` owns; idx_out capacity n. */
KPL_API int kpl_slab_partition(const kpl_slab_plan* plan, const float* xyz, int32_t xyz_stride, int64_t n, int32_t rank,
                               int32_t* idx_out, int64_t* m_out);

/* 128-byte NCCL unique id (ncclGetUniqueId): create on one rank, hand to the others by the host's own means. */
KPL_API int kpl_nccl_unique_id(void* id128_out);
/* Joins the communicator (ncclCommInitRank: blocks until all `plan->world` ranks called it).  nccl_id128 == NULL
 * creates a rank of an IN-PROCESS group instead (no NCCL: the ranks are driven together by kpl_shard_detect_group,
 * strips move by cudaMemcpyPeerAsync) -- for hosts without NCCL and for tests on a single GPU. */
KPL_API int kpl_shard_create(kpl_ctx* ctx, const kpl_slab_plan* plan, int32_t rank, const void* nccl_id128, kpl_shard** out);
KPL_API void kpl_shard_destroy(kpl_shard* s);
/* Replace the plan (same world size) without rebuilding the communicator -- e.g. after KPL_E_HALO, with a plan made
 * for a larger normal_support_cells; kpl_shard_set_slab(_normals) must follow (the normals are cleared). */
KPL_API int kpl_shard_set_plan(kpl_shard* s, const kpl_slab_plan* plan);
/* The points this rank owns (host, ascending global index; kpl_slab_partition) and their global indices.  Uploads
 * them and exchanges the strip sizes: once per resident slab, not per detection. */
KPL_API int kpl_shard_set_slab(kpl_shard* s, const float* xyz_owned, int32_t xyz_stride, const int32_t* gidx_owned, int64_t n_owned);
/* kpl_shard_set_slab plus the caller's normals of the owned points (same order as xyz_owned; 3 floats at normals_stride
 * bytes, 32 = pcl::Normal).  A non-finite normal is not an error: that point gets no score, as in kpl_detect.
 * As in kpl_detect, normals_mode, k_normals, flip_normals and viewpoint are then ignored (so is the radius-mode halo
 * requirement).  The normal strips of the halo travel in the same exchange as the positions.  Every rank must call the
 * same variant (set_slab or set_slab_normals); otherwise the call fails with KPL_E_INVALID on every rank before any
 * strip moves (NCCL: here, in the strip-size all-gather; in-process group: in kpl_shard_detect_group).  A later plain
 * kpl_shard_set_slab returns the rank to estimated normals. */
KPL_API int kpl_shard_set_slab_normals(kpl_shard* s, const float* xyz_owned, int32_t xyz_stride, const float* normals_owned,
                                       int32_t normals_stride, const int32_t* gidx_owned, int64_t n_owned);
/* New coordinates for the same partition (a detection loop that streams its slab from the host every step). */
KPL_API int kpl_shard_upload(kpl_shard* s, const float* xyz_owned, int32_t xyz_stride);
/* New normals for the same partition (pairs with kpl_shard_upload); KPL_E_INVALID on a slab set without normals. */
KPL_API int kpl_shard_upload_normals(kpl_shard* s, const float* normals_owned, int32_t normals_stride);
/* One detection (all ranks call it).  scores_owned_out: NULL or n_owned floats (host).  kp_global_out (rank 0; NULL
 * elsewhere): ascending global keypoint indices, capacity kp_capacity; *n_kp_out = global keypoint count on every rank. */
KPL_API int kpl_shard_detect(kpl_shard* s, float* scores_owned_out, int32_t* kp_global_out, int64_t kp_capacity, int64_t* n_kp_out);
/* The same for the ranks of an in-process group, driven together from one host thread; outputs are per-rank arrays
 * (entries may be NULL), the global list lands in kp_global_out. */
KPL_API int kpl_shard_detect_group(kpl_shard** shards, int32_t world, float** scores_owned_out, int32_t* kp_global_out,
                                   int64_t kp_capacity, int64_t* n_kp_out);
KPL_API int kpl_shard_get_info(const kpl_shard* s, kpl_shard_info* out);
/* Device pointer of the owned scores of the last detection (n_owned floats), for callers that keep results on the GPU. */
KPL_API const void* kpl_shard_device_scores(const kpl_shard* s);

/* ---- introspection --------------------------------------------------------------------------- */
/* kpl_detect* score each point inside the feature kernel and do not write the A*B feature rows
 * (the cv::Mat of impl/KeypointLearning.hpp:366-369) to memory; on != 0 keeps them for kpl_fetch. */
KPL_API int kpl_set_keep_intermediates(kpl_ctx* ctx, int on);
KPL_API int kpl_get_timings(const kpl_ctx* ctx, kpl_timings* t);
KPL_API int kpl_get_stats(const kpl_ctx* ctx, kpl_stats* s);
/* Device copies of intermediate results of the last call, for parity tests: what = "normals"
 * (n x 4 floats, original order) or "features" (n x A*B floats, original order). */
KPL_API int kpl_fetch(kpl_ctx* ctx, const char* what, float* out, int64_t capacity_floats);
/* Byte masks of the last detect call, original order: what = "fragile" (see kpl_stats.n_fragile_points); K*n bytes,
 * forest-major, after kpl_detect_forests. */
KPL_API int kpl_fetch_u8(kpl_ctx* ctx, const char* what, uint8_t* out, int64_t capacity);

#ifdef __cplusplus
}
#endif
#endif /* KPL_B200_H_ */

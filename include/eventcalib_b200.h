/* eventcalib_b200 — C ABI of the B200-native EventCalib hot path.
 *
 * Plain C, plain pointers and sizes, no exceptions, no torch / Eigen / OpenCV types.  Every entry point
 * returns ECB_OK (0) or a negative ecb_status; ecb_last_error(ctx) gives the text.  A context owns one
 * CUDA device + stream and all device buffers; distinct contexts may be used from distinct host threads
 * (the reference calls DBSCAN::Run from hardware_concurrency()-2 threads, eventCameraCalib.cpp:181-187).
 * There is NO CPU fallback: without a CUDA device every compute call fails with ECB_ERR_CUDA.
 *
 * Reference interfaces replaced (paths relative to /root/reference/modules/camera_calibration/):
 *   ecb_load_events_*      Event::operator>> (event/include/opengv2/event/Event.hpp:41-47) + the load loop
 *                          (event_camera_calib/test/eventCameraCalib.cpp:154-163)
 *   ecb_frontend_run       EventFrame::EventFrame (event/src/EventFrame.cpp:10-36) +
 *                          CirclesEventFrame::extractFeatures up to findCirclesGrid
 *                          (event_camera_calib/src/CirclesEventFrame.cpp:61-312) incl. fitCircle (:361-415)
 *   ecb_dbscan_run[_batch] DBSCAN<Eigen::Vector2d,double>::Run (dbscan/include/dbscan.h:115-177)
 *   ecb_fit_circles        CirclesEventFrame::fitCircle (CirclesEventFrame.cpp:361-415)
 *   ecb_cost_*             EventCalibSpline::optimize association loop (src/EventCalibSpline.cpp:157-192),
 *                          CalibReprojectionError::operator() (include/.../EventCalibSpline.hpp:168-229) as
 *                          Ceres evaluates it (residual, Jacobian, Huber, quaternion local parameterisation)
 *                          and the normal-equation build that feeds the LM step.
 */
#ifndef EVENTCALIB_B200_H
#define EVENTCALIB_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ecb_ctx ecb_ctx;

typedef enum {
    ECB_OK = 0,
    ECB_FAILED = 1,            /* mirrors DBSCAN::ERROR_TYPE::FAILED (dbscan.h:46-48,121-123) */
    ECB_ERR_CUDA = -1,         /* no device / CUDA runtime error */
    ECB_ERR_ARG = -2,          /* bad argument */
    ECB_ERR_UNSUPPORTED = -3,  /* input outside what the device path handles (see ecb_last_error) */
    ECB_ERR_STATE = -4         /* call order (e.g. no events loaded) */
} ecb_status;

/* per-problem status bits reported by the device kernels */
#define ECB_PB_OK 0u
#define ECB_PB_DUPLICATE 2u     /* duplicate pixels inside one front-end problem (cannot happen after the per-pixel dedupe);
                                   ecb_dbscan_run* re-runs such inputs on the general path instead of reporting this */
#define ECB_PB_CLUSTER_CAP 4u   /* more kept clusters than max_clusters: tables truncated, labels still exact */
#define ECB_PB_RANGE 8u         /* pixel outside the sensor / bitmap */

/* ---- context ------------------------------------------------------------------------------------- */
/* stream: a cudaStream_t (as void*) to run on, or NULL for a context-owned stream. */
int ecb_ctx_create(int device, void *stream, ecb_ctx **out);
void ecb_ctx_destroy(ecb_ctx *ctx);
const char *ecb_last_error(const ecb_ctx *ctx);
/* number of kernels of this library launched through ctx so far */
uint64_t ecb_launch_count(const ecb_ctx *ctx);
int ecb_synchronize(ecb_ctx *ctx);
/* Per-kernel device timing (CUDA events on the context stream around every launch; no extra syncs).
 * ecb_stage_ms: durations of the most recent launch of each stage, out[ECB_N_STAGES]; synchronizes. */
#define ECB_STAGE_INGEST 0
#define ECB_STAGE_BOUNDS 1
#define ECB_STAGE_WINDOW 2
#define ECB_STAGE_CLUSTER 3
#define ECB_STAGE_PAIR 4
#define ECB_STAGE_ASSOC 5
#define ECB_STAGE_NORMAL_EQ 6
#define ECB_STAGE_COST 7
#define ECB_STAGE_ORDER 8
#define ECB_STAGE_BFS 9
#define ECB_N_STAGES 10
int ecb_set_profiling(ecb_ctx *ctx, int on);
int ecb_stage_ms(ecb_ctx *ctx, float *out);
const char *ecb_version(void);
/* number of CUDA devices visible to the process (0 without a driver / device): a multi-GPU host creates one context per device */
int ecb_device_count(void);

/* ---- a1: event ingest ---------------------------------------------------------------------------- */
/* Sensor size in pixels (Camera.width / Camera.height of the YAML). Must be set before loading events. */
int ecb_set_sensor(ecb_ctx *ctx, int width, int height);
/* records: n packed 25-byte reference records (f64 t, f64 x, f64 y, u8 polarity), time sorted.
 * _host copies host->device inside the call; _device expects a device pointer (16-byte aligned).
 * The records are unpacked to the SoA layout the kernels use (f64 t[n], u32 x|y<<15|pol<<31).
 * Events with non-integer or out-of-sensor coordinates, or an unsorted stream, make the call fail
 * with ECB_ERR_UNSUPPORTED (the reference would accept them; this path does not, loudly). */
int ecb_load_events_host(ecb_ctx *ctx, const void *records, int64_t n);
int ecb_load_events_device(ecb_ctx *ctx, const void *d_records, int64_t n);
int64_t ecb_num_events(const ecb_ctx *ctx);

/* ---- a2-a5: batched window front end --------------------------------------------------------------- */
typedef struct {
    double dbscan_eps;          /* CirclesEventFrame::Params (CirclesEventFrame.cpp:35-48) */
    uint32_t dbscan_min_pts;    /* dbscan_startMinSample */
    uint32_t cluster_min;       /* clusterMinSample */
    int32_t knn_num;
    int32_t fit_circle;         /* 0: mutual-nearest medians (example.yaml default), 1: fitted circles */
    double radius_threshold;    /* circleRadiusThreshold_ (CirclesEventFrame.cpp:16-33) */
    uint32_t rows_cols;         /* pattern rows*cols (need that many kept clusters per polarity, :127-129) */
    int32_t order_mode;         /* 0: pid = first-arrival order; 1: libstdc++ unordered_set iteration order
                                   (the reference's order, EventFrame.cpp:12-35) */
    uint32_t max_clusters;      /* kept-cluster table capacity per (window,polarity).  0 (recommended): automatic — the
                                   tables grow until every window fits (the reference has no cap,
                                   CirclesEventFrame.cpp:89-117) and the context keeps the capacity for later runs;
                                   > 0: fixed capacity, windows with more kept clusters are truncated and flagged
                                   ECB_PB_CLUSTER_CAP */
    uint32_t median_mode;       /* cluster centre = member with the median norm (CirclesEventFrame.cpp:137-147):
                                   0: slot size/2 of the members sorted by (norm, pid) — order independent;
                                   1: the reference's pick: std::nth_element (libstdc++) over the members in DBSCAN's
                                      BFS pop order — differs from 0 only when several members share the median norm */
} ecb_frontend_params;

typedef struct {
    int64_t ev_lo, ev_hi;       /* event index range of the CLOSED window [t0,t1] */
    int32_t n_points[2];        /* [0]=negative, [1]=positive unique surviving pixels (pid count) */
    int32_t n_clusters[2];      /* raw DBSCAN clusters */
    int32_t n_kept[2];          /* after the clusterMinSample filter */
    int32_t n_candidates;       /* candidate circles (pairs) */
    uint32_t status;            /* ECB_PB_* bits */
    int64_t point_offset[2];    /* offset of this window's points in the flat per-polarity arrays */
} ecb_window_summary;

/* windows: n_win closed intervals [t0,t1] (host doubles, interleaved).  Runs window selection, per-pixel
 * dedupe, +/- cancellation, DBSCAN on both polarities, the cluster-size filter, medians, pairing and
 * circle fit for every window in one batch. Results stay on the device until fetched. */
int ecb_frontend_run(ecb_ctx *ctx, const double *windows, int n_win, const ecb_frontend_params *params);
int ecb_frontend_summary(ecb_ctx *ctx, ecb_window_summary *out, int n_win);
/* total number of point slots per polarity (size of the flat arrays below) */
int64_t ecb_frontend_total_points(ecb_ctx *ctx, int polarity);
/* flat per-polarity arrays: xy (2 doubles per point, pid order per window) and labels (cluster id in
 * discovery order, -1 = Noise) */
int ecb_frontend_points(ecb_ctx *ctx, int polarity, double *xy, int32_t *labels);
/* per window up to max_cand candidates: pi, ni (kept-cluster indices), cx, cy, r  -> out[n_win][max_cand][5] */
int ecb_frontend_candidates(ecb_ctx *ctx, double *out, int max_cand);
/* kept-cluster table of one window/polarity: raw cluster id, size, median pid  (each up to cap entries) */
int ecb_frontend_clusters(ecb_ctx *ctx, int window, int polarity, int32_t *raw_id, int32_t *size,
                          int32_t *median_pid, int cap);
/* a6: CirclesEventFrame::rectifyFeatures (CirclesEventFrame.cpp:417-609) for n_frames windows of the last run, batched over
 * frames x board circles.  image_points[n_frames][n_circles][5][2]: the projected circle centre and its four quadrant
 * points (:431-456; cv::projectPoints stays on the caller's side, it needs the OpenCV initialisation).  Per circle: radius
 * search over the window's points, quadrant-wise +-inlier_threshold band, expansion to whole DBSCAN clusters, circle fit,
 * sanity gates.  out[n_frames][n_circles][3] = rectified cx, cy, r (r < 0: feature deleted, :461,:560,:573);
 * frame_ok[n_frames] (optional) = the frame verdict of :585-609 (edge scores — skipped when fit_circle — and the 20 % rule)
 * for a rows x cols (a)symmetric pattern.  inlier_threshold is 3 px in the reference (:475). */
int ecb_frontend_rectify(ecb_ctx *ctx, const int32_t *window_index, int n_frames, int n_circles,
                         const double *image_points, double inlier_threshold, int rows, int cols, int asymmetric,
                         double *out, int32_t *frame_ok);
/* device pointers of the results of the last run (for callers that keep working on the GPU) */
int ecb_frontend_device_ptrs(ecb_ctx *ctx, void **d_summary, void **d_candidates, int *cand_stride);

/* ---- a3: the DBSCAN::Run boundary ---------------------------------------------------------------- */
/* xy: n x 2 doubles in pid order — ANY finite doubles, duplicates included, any eps (the reference's template takes every
 * T with operator[], dbscan.h:40,70).  Distinct integer pixels with 1 <= eps <= 15 (what the calibration front end
 * produces) run on the sensor-plane bitmap kernel; everything else runs on the general path (grid hash: cell =
 * floor((p - min) / eps), in-tree radix sort by cell key, 3 x 3 cell search, the kd query's strict pruning rule replayed on
 * the emulated insertion tree for the pairs it can affect).  Both give the reference's labels.
 * labels[n]: cluster id in the reference's discovery order, -1 = Noise.
 * Returns ECB_FAILED for n<1 or min_pts<1 exactly like the reference; ECB_ERR_UNSUPPORTED only for NaN / infinite
 * coordinates, NaN eps and problems of 2^21 points or more. */
int ecb_dbscan_run(ecb_ctx *ctx, const double *xy, int n, double eps, uint32_t min_pts, int32_t *labels,
                   int32_t *n_clusters);
/* batch: problem k is xy[offsets[k] .. offsets[k+1]); labels is flat; n_clusters[n_problems]; status
 * (optional) receives ECB_PB_* bits per problem */
int ecb_dbscan_run_batch(ecb_ctx *ctx, const double *xy, const int64_t *offsets, int n_problems, double eps,
                         uint32_t min_pts, int32_t *labels, int32_t *n_clusters, uint32_t *status);

/* Same, plus `Clusters` as the reference builds them (dbscan.h:92,143-162,229-259): cluster c (discovery order) holds
 * cluster_sizes[c] members, listed consecutively in `members` in the reference's order (the seed, then core points in
 * the order expandCluster's FIFO pops them; neighbours enumerated like kd_nearest_range does).  Noise = the pids with
 * label -1, ascending.  cluster_sizes and members need room for n entries. */
int ecb_dbscan_run_ordered(ecb_ctx *ctx, const double *xy, int n, double eps, uint32_t min_pts, int32_t *labels,
                           int32_t *n_clusters, int32_t *cluster_sizes, uint32_t *members);
/* batch form: problem k's sizes start at cluster_sizes[offsets[k]] (n_clusters[k] entries) and its member lists at
 * members[offsets[k]] (one entry per core point) */
int ecb_dbscan_run_batch_ordered(ecb_ctx *ctx, const double *xy, const int64_t *offsets, int n_problems, double eps,
                                 uint32_t min_pts, int32_t *labels, int32_t *n_clusters, uint32_t *status,
                                 int32_t *cluster_sizes, uint32_t *members);

/* DBSCAN<T,Float>::Run(V, dim, eps, min) for dim = 1 .. 4 (dbscan.h:115-177): pts = n x dim doubles.  cluster_sizes and
 * members are optional (both or neither): ordered `Clusters` as above.  dim < 1 returns ECB_FAILED like the reference. */
int ecb_dbscan_run_nd(ecb_ctx *ctx, const double *pts, int n, int dim, double eps, uint32_t min_pts, int32_t *labels,
                      int32_t *n_clusters, int32_t *cluster_sizes, uint32_t *members);

/* ---- a5: batched circle fit ---------------------------------------------------------------------- */
/* set k = points xy[offsets[k]..offsets[k+1]) (union of a + and a - index set); out[k] = cx, cy, r */
int ecb_fit_circles(ecb_ctx *ctx, const double *xy, const int64_t *offsets, int n_sets, double *out);

/* ---- a7-a12: cost evaluation of the dynamic-calibration objective ------------------------------------ */
/* Spline structure (EventCalibSpline ctor, src/EventCalibSpline.cpp:63-91): n_splines segments, n_cp[s] control
 * points each, knots = concatenation of the (n_cp[s] + 4) clamped cubic knot vectors.  Control points are passed to
 * the evaluation calls as flat arrays over all segments: rot_cp 4 doubles each (x,y,z,w), trans_cp 3 doubles each.
 * huber_delta = 0.2 * circle_radius in the reference (:197). */
int ecb_cost_setup(ecb_ctx *ctx, int n_splines, const int32_t *n_cp, const double *knots, double circle_radius,
                   double huber_delta);
/* Rotation model of the residual blocks (the reference's `useSO3` switch, eventCameraCalib.cpp:204-209):
 *   0 (default) CalibReprojectionError      — normalised quaternion B-spline, EigenQuaternionParameterization (hpp:158-250)
 *   1           CalibReprojectionError_SO3 — cumulative SO(3) B-spline R0 * prod exp(beta_j log(R_{j-1}^-1 R_j)) with
 *               LocalParameterizationSO3 (hpp:65-156, BsplineSO3.hpp:190-221); rot_cp are then Sophus::SO3d coefficients (x,y,z,w)
 * Also selects the Plus operation of the host LM step (ecb_lm_options.rotation_model must match). */
int ecb_cost_set_rotation_model(ecb_ctx *ctx, int use_so3);
/* Intrinsics held constant in the spline optimisation.  Bit i of mask = intrinsic i in the order fx fy cx cy k1 k2 k3 k4 k5 (the
 * order of every intrinsics array here).  k1 .. k5 are the coefficients of the INVERSE radial polynomial of the spline stage, not
 * OpenCV's distortion coefficients (the YAML's Fix_K* keys name those).  0 (default): all 9 are free, as in the reference.
 * The optimisation is the reduced problem, what Ceres does with a SubsetManifold on the intrinsics block: the rows and columns of
 * the constant intrinsics in J^T J and their entries of J^T r are zeroed once the normal equations are assembled, so their step is
 * exactly 0 and they keep their start values exactly (==).  The parameter-tolerance test still uses |x| of the full vector.
 * ecb_covariance then returns the covariance conditional on the constant intrinsics: Z = the inverse of H restricted to the free
 * parameters, exact zeros in the rows and columns of the constant ones, dimension = D - popcount(mask).
 * A property of the context: it survives ecb_cost_setup.  ecb_calibrate and ecb_covariance read it at each call,
 * ecb_lm_device_create captures it.  Changing it makes ecb_pose_covariance return ECB_ERR_STATE until the next ecb_covariance.
 * mask > 0x1FF returns ECB_ERR_ARG. */
int ecb_cost_set_constant_intrinsics(ecb_ctx *ctx, uint32_t mask);
/* total control points, total span blocks (sum of n_cp-3), residual count, doubles in the packed result */
int ecb_cost_layout(ecb_ctx *ctx, int32_t *total_cp, int32_t *total_spans, int64_t *n_residuals, int64_t *out_doubles);
/* Residual blocks from the loaded events (association loop of optimize(), :157-192, with findCenter,
 * CirclesEventFrame.hpp:50-65): kf_time[K] ascending key-frame stamps, kf_circles[K][n_circles][3] = (cx, cy, r) of
 * each frame's features (r < 0 marks an absent feature), landmarks_xyz[n_circles][3] the board points. */
int ecb_cost_associate(ecb_ctx *ctx, const double *kf_time, const double *kf_circles, int n_keyframes, int n_circles,
                       const double *landmarks_xyz, double motion_time_step, int64_t *n_residuals);
/* The same with the three tables already in device memory (the counterpart of ecb_load_events_device: a caller that keeps the
 * key frames on the GPU across optimisations does not pay their upload per call; the tables are read during this call only). */
int ecb_cost_associate_device(ecb_ctx *ctx, const double *d_kf_time, const double *d_kf_circles, int n_keyframes, int n_circles,
                              const double *d_landmarks_xyz, double motion_time_step, int64_t *n_residuals);
int ecb_cost_get_association(ecb_ctx *ctx, int64_t *event_index, int32_t *circle_id, int64_t cap);
/* ... or explicit residual blocks (host arrays, ordered by (spline, time)) */
int ecb_cost_set_residuals(ecb_ctx *ctx, const double *obs_xy, const double *lm_xyz, const double *t,
                           const int32_t *spline, int64_t n);
/* cost = sum 1/2 rho(r^2)  (Ceres Evaluate without Jacobians; LM step acceptance) */
int ecb_cost_eval(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, double *cost);
/* Normal equations in the tangent space, packed per knot span s (33 local parameters: intrinsics 9 | rotation
 * tangent of control points s..s+3, 3 each | translation of the same control points, 3 each):
 *   out[s*1122 .. +1089) = J^T J of the span's residual blocks (33x33, full symmetric, row major)
 *   out[s*1122+1089 .. +33) = J^T r ;  out[n_spans*1122] = cost
 * d_out: device buffer to fill (e.g. one a collective will all-reduce), or NULL for the context's own;
 * h_out: optional host copy; cost: optional.  Deterministic (fixed-order reductions). */
int ecb_cost_normal_eq(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, void *d_out,
                       double *h_out, double *cost);

/* ---- how well the model fits: the residuals of the calibration and their statistics --------------------------------------
 * r_k is the raw residual of record k, ||X_w - L|| - circle_radius before the Huber loss (CalibReprojectionError; the rotation
 * model of ecb_cost_set_rotation_model selects the quaternion or the SO(3) spline).  It is a DISTANCE ON THE BOARD PLANE, in the
 * units of the board points and of circle_radius, NOT in pixels.  Records are in the order of ecb_cost_get_association (record k
 * pairs with event_index[k] and circle_id[k]), or in the order given to ecb_cost_set_residuals.  The point (intrinsics, rot_cp,
 * trans_cp) has the layout of ecb_cost_eval.  Record indices are 32-bit: n_residuals < 2^32 (ECB_ERR_UNSUPPORTED otherwise).
 * Both calls read this context's records only: with several GPUs every shard reports its own share. */
/* r_k of every record, FP64.  d_out: device buffer of n_residuals doubles, or NULL for a context-owned one; h_out: optional host
 * copy.  Asynchronous on the context's stream unless h_out is given. */
int ecb_cost_residuals(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, double *d_out,
                       double *h_out);
/* Statistics of a group of residuals.  mean = sum / count and RMS = sqrt(sum_sq / count) are left to the caller.  A residual is
 * down-weighted when r^2 > huber_delta^2 (the linear branch of the Huber loss).  cost = sum rho(r^2) / 2, the group's share of
 * ecb_cost_eval.  Every field is a sum or a max, so the results of several shards combine by a fixed-order sum. */
typedef struct {
    int64_t count, n_downweighted;
    double sum, sum_sq, max_abs;   /* of r (board units, not pixels); max_abs = 0 for an empty group */
    double cost;
} ecb_residual_group;
#define ECB_RESIDUALS_BY_KEYFRAME 0     /* the key frame the association used: nearest stamp to the event, ties -> the earlier */
#define ECB_RESIDUALS_BY_CIRCLE 1       /* circle_id: n_circles groups */
#define ECB_RESIDUALS_BY_SENSOR_CELL 2  /* (floor(v / c)) * ceil(W / c) + floor(u / c) of the observation (u, v), row major */
/* Statistics of the residuals at the point, grouped by `by`:
 *   BY_KEYFRAME: kf_time[n_keyframes] are the host stamps given to the association (n_keyframes must equal its K, else
 *                ECB_ERR_ARG); K groups.
 *   BY_CIRCLE: n_circles groups, as given to the association.
 *   BY_SENSOR_CELL: cells of cell_px x cell_px pixels of the sensor W x H of ecb_set_sensor, ceil(W/c) * ceil(H/c) groups;
 *                an observation outside [0, W) x [0, H) (explicit residuals only) counts in `total` only.
 * *n_groups (if non-NULL) is always set.  cap < *n_groups returns ECB_ERR_ARG and writes nothing else; groups = NULL with cap = 0
 * is a pure size query (ECB_OK, nothing computed).  total (optional): all records.  Zero residuals give all-zero groups.
 * Errors: unknown `by`, cell_px < 1, or kf_time == NULL for BY_KEYFRAME: ECB_ERR_ARG.  BY_KEYFRAME or BY_CIRCLE on residuals of
 * ecb_cost_set_residuals, BY_KEYFRAME after events were loaded since the association, BY_SENSOR_CELL without ecb_set_sensor:
 * ECB_ERR_STATE.  Deterministic: repeated calls are bit-identical (stable radix sort by group, fixed-order reductions, no
 * floating-point atomics).  Synchronises the context's stream. */
int ecb_cost_residual_groups(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, int by,
                             const double *kf_time, int n_keyframes, int cell_px, ecb_residual_group *groups, int cap,
                             int *n_groups, ecb_residual_group *total);
/* Outlier rejection: removes record k from this context when !(|r_k| <= max_abs_residual), r_k exactly as ecb_cost_residuals
 * returns it at the point (so a non-finite r_k is always removed), or when drop_keyframe[j] != 0 for the key frame j the record
 * counts under in ECB_RESIDUALS_BY_KEYFRAME (nearest stamp to the event, ties -> the earlier frame).  The kept records keep their
 * order.  drop_keyframe = NULL: no key-frame criterion; max_abs_residual = INFINITY: no residual criterion.  kf_time /
 * n_keyframes as in ecb_cost_residual_groups (the host stamps given to the association; only read with drop_keyframe).
 * *n_kept / *n_removed (optional) count this context's records.  When nothing is removed the records are left untouched.
 * The removal lasts until the next ecb_cost_associate[_device] or ecb_cost_set_residuals: ecb_cost_layout,
 * ecb_cost_get_association, both reports, ecb_cost_eval, ecb_cost_normal_eq[_exchange], ecb_calibrate, the device LM (it reads
 * the records at every evaluation, so one created before this call stays valid) and ecb_covariance see only the kept records.
 * A covariance computed before the call still answers ecb_pose_covariance: call ecb_covariance again for the kept records.
 * Errors: max_abs_residual NaN or negative, drop_keyframe without kf_time, or n_keyframes != the association's K: ECB_ERR_ARG.
 * No ecb_cost_setup, drop_keyframe on records of ecb_cost_set_residuals, or drop_keyframe after events were loaded since the
 * association: ECB_ERR_STATE.  n_residuals >= 2^32: ECB_ERR_UNSUPPORTED.  Zero records: ECB_OK, both counts 0.  No
 * floating-point atomics: deterministic.  Synchronises. */
int ecb_cost_reject(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, double max_abs_residual,
                    const double *kf_time, const uint8_t *drop_keyframe, int n_keyframes, int64_t *n_kept, int64_t *n_removed);
/* Re-association at a calibrated point (intrinsics / rot_cp / trans_cp as ecb_cost_eval): every loaded event i is matched again to
 * a board circle through the model instead of the detected ellipses of its key frame.  Candidates are the events that lie in a
 * spline segment, have a valid pixel and lie near their key frame (the nearest stamp of the association, ties -> the earlier one):
 * max_dt = 0 applies the association's own test (dt^2 < (5 motion_time_step)^2, so the candidates are exactly the association's),
 * max_dt > 0 keeps |t_i - t_kf| <= max_dt.  For a candidate: the pose at t_i on the spline (rotation model of the context), X_w =
 * the back-projection of the event pixel onto the board plane (the arithmetic of the residual), c* = the landmark of the
 * association nearest to X_w in FP64 over ALL n_circles (detected in that key frame or not; ties -> the smaller index; no circle
 * when X_w is not finite), e = ecb_rim_reprojection of (i, c*), the value ecb_cost_reprojection_errors returns for that record.
 * The event is kept iff |e| < gate_px (NaN never; 5 is the association's pixel tolerance).  The kept events replace the
 * records, in event order and in the layout of ecb_cost_associate; key frames, landmarks and K stay those of the association,
 * so the groupings, ecb_cost_reject with a mask and ecb_cost_get_association keep working.  Like an association, it undoes an
 * earlier rejection.  After ecb_cost_associate_device the stamps are read at the association's d_kf_time, which must still
 * hold them.  *n_residuals: the new record count; *n_same / *n_changed (same event, same / another circle), *n_new (event not
 * recorded before) and *n_lost (record whose event is not kept) compare with the records held just before the call (after any
 * rejection); all optional.  A device LM created before the call stays valid: it reads the records at every evaluation.  A
 * covariance computed before still answers ecb_pose_covariance: call ecb_covariance again for the new records.
 * Errors: gate_px NaN or <= 0, max_dt NaN or < 0: ECB_ERR_ARG.  No ecb_cost_setup, records of ecb_cost_set_residuals or of no
 * association, events loaded since the association: ECB_ERR_STATE.  A record count >= 2^32: ECB_ERR_UNSUPPORTED.  Zero kept
 * events: ECB_OK.  No floating-point atomics: repeated calls give bit-identical records.  Synchronises. */
int ecb_cost_reassociate(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, double gate_px,
                         double max_dt, int64_t *n_residuals, int64_t *n_same, int64_t *n_changed, int64_t *n_new,
                         int64_t *n_lost);

/* ---- the same fit in pixels: reprojection errors through the forward camera model --------------------------------------------
 * The spline stage's distortion is the inverse radial polynomial (undistorted = distorted * s(rho_d^2), s = 1 + k1 rho^2 + ... +
 * k5 rho^10, ecb_residual.h); projecting inverts g(rho) = rho s(rho^2) by safeguarded Newton (ecb_camera.h).  g is increasing
 * on [0, rho_fold) only, rho_fold^2 = the smallest positive root of h(u) = 1 + 3 k1 u + 5 k2 u^2 + ... + 11 k5 u^5, so points
 * whose undistorted radius reaches g(rho_fold) cannot be projected.
 * e_k, the reprojection error of record k in pixels: X_w = the event pixel o back-projected onto the board plane at the record's
 * pose (as in the residual), d = X_w - L, rim point P = L + radius d / |d| (the correspondence the residual measures), q = the
 * pixel of P; e_k = sign(|d| - radius) |q - o|, positive when the event lies outside the projected rim.  It is the residual's
 * correspondence seen in the image, NOT the distance to the projected ellipse of the circle.  e_k is NaN (not projectable)
 * when |d| = 0, when the event's own distorted radius is >= rho_fold (the model folds inside the sensor there), when P lies
 * behind the camera or past the fold, or when a value is not finite. */
/* host only: rho_fold of the inverse radial polynomial k[5] (+INFINITY when g is increasing everywhere) */
int ecb_inverse_radial_fold(const double *k, double *rho_fold);
/* e_k of every record, in the order of ecb_cost_residuals; NaN = not projectable.  d_out / h_out as ecb_cost_residuals;
 * n_invalid (optional) synchronises. */
int ecb_cost_reprojection_errors(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp,
                                 double *d_out, double *h_out, int64_t *n_invalid);
/* Statistics of a group of reprojection errors, in pixels.  count, sum, sum_sq and max_abs cover the valid records only (RMS =
 * sqrt(sum_sq / count)); an invalid record adds to n_invalid and to nothing else. */
typedef struct { int64_t count, n_invalid; double sum, sum_sq, max_abs; } ecb_reprojection_group;  /* pixels */
/* The groups of ecb_cost_residual_groups (by, kf_time, n_keyframes, cell_px, the size query, cap, every error code and the 2^32
 * record limit are the same) over e_k.  Deterministic: repeated calls are bit-identical.  Synchronises. */
int ecb_cost_reprojection_groups(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, int by,
                                 const double *kf_time, int n_keyframes, int cell_px, ecb_reprojection_group *groups, int cap,
                                 int *n_groups, ecb_reprojection_group *total);
/* circle centres of the key frames reprojected at their stamps: proj[K][n_circles][2], err[K][n_circles] = |proj - (cx,cy)|;
 * NaN for an absent feature (r < 0), a stamp outside every segment, or a point that cannot be projected.
 * kf_time / kf_circles / landmarks_xyz as ecb_cost_associate (host arrays); the pose is the spline of ecb_cost_setup at the
 * point, in the rotation model of the context.  This is the quantity calibrateCamera reports, against the detected centre: the
 * fitted ellipse centre is not the projected circle centre (OpenCV's circle-grid calibration has the same bias).  proj, err and
 * total are optional; total covers the present features (absent ones count nowhere, unprojectable ones in n_invalid).  Needs
 * ecb_cost_setup, reads no residual records.  Synchronises. */
int ecb_keyframe_reprojection(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp,
                              const double *kf_time, const double *kf_circles, int n_keyframes, int n_circles,
                              const double *landmarks_xyz, double *proj, double *err, ecb_reprojection_group *total);

/* Multi-GPU (one process per GPU): the same evaluation with the inter-GPU sum fused in.  Every rank owns a receive
 * buffer of ecb_exchange_buffer_bytes() bytes, ZERO-FILLED once, in device memory its peers can write (same process:
 * any cudaMalloc pointer with peer access; other processes: ecb_device_alloc + ecb_ipc_export / ecb_ipc_open).
 * recv_buffers[p] = rank p's buffer as seen from this process (own buffer at [rank]).  The span reduction writes this rank's
 * result into its slot of every peer's buffer over NVLink, publishes (epoch, span range, cost), waits for all ranks'
 * slots of this epoch and sums them in rank order into d_out (layout of ecb_cost_normal_eq; bit-identical on all ranks).
 * epoch: 1, 2, 3, ... — the same sequence on every rank; `cost` (optional) synchronises the stream.
 * phases: ECB_EXCHANGE_BOTH normally.  The receive side spins (one warp, bounded) until the peers' slots arrive, so
 * "ranks" that share ONE device must not enqueue it before every rank's send side (CUDA does not promise that two streams
 * of a device run concurrently): issue ECB_EXCHANGE_SEND on all of them first, then ECB_EXCHANGE_RECV. */
#define ECB_MAX_PEERS 16
#define ECB_EXCHANGE_SEND 1
#define ECB_EXCHANGE_RECV 2
#define ECB_EXCHANGE_BOTH 3
size_t ecb_exchange_buffer_bytes(ecb_ctx *ctx, int n_ranks);
int ecb_cost_normal_eq_exchange(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, int rank,
                                int n_ranks, void *const *recv_buffers, uint64_t epoch, int phases, void *d_out, double *cost);
/* plumbing for the receive buffers: device allocation (zero-filled) that can be exported to other processes of the node */
int ecb_device_alloc(ecb_ctx *ctx, size_t bytes, void **d_ptr);
int ecb_device_free(ecb_ctx *ctx, void *d_ptr);
int ecb_ipc_export(ecb_ctx *ctx, void *d_ptr, void *handle64);          /* 64-byte cudaIpcMemHandle_t */
int ecb_ipc_open(ecb_ctx *ctx, const void *handle64, void **d_ptr);     /* maps a peer's buffer (enables peer access) */
int ecb_ipc_close(ecb_ctx *ctx, void *d_ptr);
/* several GPUs driven from ONE process (one context per device): lets ctx's kernels store into ecb_device_alloc buffers of
 * peer_device (cudaDeviceEnablePeerAccess); receive buffers are then passed to the exchange as plain device pointers */
int ecb_enable_peer_access(ecb_ctx *ctx, int peer_device);

/* ---- a12: the LM step around the GPU normal equations (EventCalibSpline::optimize, src/EventCalibSpline.cpp:197-247) ---- */
typedef struct {
    int32_t max_iterations;        /* 50 (Ceres default; BASELINE config C4) */
    int32_t jacobi_scaling;        /* 1 */
    int32_t fixed_iterations;      /* != 0: convergence tests off, exactly max_iterations LM iterations (benchmark C4) */
    int32_t rotation_model;        /* 0: x+ = dq(delta) * x (EigenQuaternionParameterization); 1: x+ = x * exp(delta) (LocalParameterizationSO3) */
    double function_tolerance;     /* 1e-10 (EventCalibSpline.cpp:239-240) */
    double gradient_tolerance;     /* 1e-10 */
    double parameter_tolerance;    /* 1e-8 */
    double initial_radius, max_radius, min_radius;      /* 1e4, 1e16, 1e-32 */
    double min_relative_decrease;  /* 1e-3 */
    double min_lm_diagonal, max_lm_diagonal;            /* 1e-6, 1e32 */
} ecb_lm_options;

typedef struct {
    int32_t iterations, successful_steps, termination, reserved;
    double initial_cost, final_cost, gradient_max_norm, radius;
} ecb_lm_summary;

#define ECB_LM_RUNNING 0
#define ECB_LM_NO_CONVERGENCE 2       /* max_iterations reached */
#define ECB_LM_FUNCTION_TOLERANCE 3
#define ECB_LM_GRADIENT_TOLERANCE 4
#define ECB_LM_PARAMETER_TOLERANCE 5
#define ECB_LM_MIN_RADIUS 6
#define ECB_LM_FAILURE 7

typedef struct ecb_lm ecb_lm;
void ecb_lm_default_options(ecb_lm_options *o);
/* Host-only LM state machine (no CUDA): the caller evaluates, possibly all-reducing the packed normal equations
 * across GPUs in between.   begin(x, packed) -> { propose(candidate) -> [caller: cost(candidate)] -> feedback(cost)
 *   -> 1: accepted, caller evaluates packed at the candidate -> update(packed) | 0: rejected } until != RUNNING */
ecb_lm *ecb_lm_create(int n_splines, const int32_t *n_cp, const ecb_lm_options *opt);
void ecb_lm_destroy(ecb_lm *lm);
int ecb_lm_dimension(const ecb_lm *lm);
/* constant intrinsics of this state machine (mask as ecb_cost_set_constant_intrinsics); before ecb_lm_begin, ECB_ERR_STATE after */
int ecb_lm_set_constant_intrinsics(ecb_lm *lm, uint32_t mask);
int ecb_lm_begin(ecb_lm *lm, const double *intrinsics, const double *rot_cp, const double *trans_cp, const double *packed);
int ecb_lm_propose(ecb_lm *lm, double *cand_intrinsics, double *cand_rot_cp, double *cand_trans_cp);
int ecb_lm_feedback(ecb_lm *lm, double candidate_cost);
int ecb_lm_update(ecb_lm *lm, const double *packed);
int ecb_lm_state(const ecb_lm *lm, double *intrinsics, double *rot_cp, double *trans_cp, ecb_lm_summary *summary);
/* rows of (cost, gradient_max_norm, radius, accepted) per recorded evaluation; returns the row count */
int ecb_lm_trace(const ecb_lm *lm, double *out, int cap_rows);
/* single-GPU driver of the whole loop; parameters are updated in place */
int ecb_calibrate(ecb_ctx *ctx, int n_splines, const int32_t *n_cp, double *intrinsics, double *rot_cp, double *trans_cp,
                  const ecb_lm_options *opt, ecb_lm_summary *summary, double *trace, int trace_rows);

/* ---- the same loop with the state machine AND the linear solve on the device --------------------------------------------
 * The host only enqueues kernels: per iteration a band-arrow Cholesky of the damped system (one CTA per spline segment, the 9
 * intrinsics and the right-hand side as arrow rows), the candidate's cost, the accept / reject decision and — only if the step
 * was accepted, decided by a device flag — the normal equations at the new point.  Nothing crosses PCIe until the result is
 * read.  Several GPUs (one process per GPU, or several contexts of one process): every rank runs the same replicated state
 * machine on its own share of the residuals; the packed normal equations and the candidate costs are summed over the ranks
 * inside the kernels through the peer-mapped receive buffers of ecb_cost_normal_eq_exchange (sized by
 * ecb_exchange_buffer_bytes, zero-filled once), in rank order, so all ranks take bit-identical decisions.
 * fixed_iterations != 0 runs exactly max_iterations iterations (benchmark config C4): no convergence test, no MIN_RADIUS exit.
 * Call order: create (after ecb_cost_setup + association) -> [set_exchange] -> begin -> iterate(n) ... -> result. */
typedef struct ecb_lm_device ecb_lm_device;
int ecb_lm_device_create(ecb_ctx *ctx, int n_splines, const int32_t *n_cp, const ecb_lm_options *opt, ecb_lm_device **out);
void ecb_lm_device_destroy(ecb_lm_device *lm);
int ecb_lm_device_set_exchange(ecb_lm_device *lm, int rank, int n_ranks, void *const *recv_buffers);
/* uploads x, evaluates the normal equations at x, initialises the trust region (asynchronous) */
int ecb_lm_device_begin(ecb_lm_device *lm, const double *intrinsics, const double *rot_cp, const double *trans_cp);
/* enqueues n_iterations LM iterations (asynchronous; no-ops on the device once the state machine has terminated) */
int ecb_lm_device_iterate(ecb_lm_device *lm, int n_iterations);
/* synchronises: 1 while the state machine is running, 0 when it has terminated, < 0 on error */
int ecb_lm_device_running(ecb_lm_device *lm);
/* synchronises and reads back the parameters, the summary and up to trace_rows rows of (cost, gradient_max_norm, radius,
 * accepted 1 / rejected 0 / invalid -1) */
int ecb_lm_device_result(ecb_lm_device *lm, double *intrinsics, double *rot_cp, double *trans_cp, ecb_lm_summary *summary,
                         double *trace, int trace_rows);
/* begin + iterations until termination + result; parameters are updated in place */
int ecb_calibrate_device(ecb_lm_device *lm, double *intrinsics, double *rot_cp, double *trans_cp, ecb_lm_summary *summary,
                         double *trace, int trace_rows);

/* ---- uncertainty of the calibration: covariance of the intrinsics and the spline control points ----------------------------
 * x is the parameter point in the tangent space of the selected rotation model: control point c owns rows 6c .. 6c+5 (rotation
 * tangent 3, translation 3) of the flat order over all segments, the 9 intrinsics come last (D = 6 C + 9).  H = J^T J at x
 * (Huber corrector applied, as ecb_cost_normal_eq).  Z = H^-1 as ceres::Covariance returns it with default options (no sigma^2
 * scaling); the standard deviation of parameter i is sqrt(sigma2 Z_ii) with sigma2 = 2 cost / (n_residuals - D) (OpenCV's
 * calibrateCameraExtended convention).  Z is computed on the device: Cholesky factor of S H S (S = diag(H)^-1/2, 1 where the
 * diagonal is 0) with the LM's band-arrow factorisation, undamped, then the selected inverse of that factor, i.e. the entries of
 * Z on the band / arrow pattern: every control point's 6 x 6 block, any 4 consecutive control points (a pose on the spline), the
 * intrinsics.  FP64, deterministic.
 *   d_packed: NULL = evaluate the normal equations at x on this context; else an already-summed packed buffer on this context's
 *             device (layout of ecb_cost_normal_eq, e.g. the d_out of ecb_cost_normal_eq_exchange): every rank then computes the
 *             same result bit for bit
 *   n_residuals_total: residual count of sigma2; 0 = this context's count
 *   cov_intrinsics[9 x 9]; cov_band[6C x 24] = Z(j + r, j) at [j * 24 + r] (0 past the end of a segment); cov_cross[9 x 6C] =
 *   Z(intrinsic i, j) at [i * 6C + j].  Output pointers may be NULL.
 * A relative pivot L(j,j)^2 / M(j,j) <= 1e-12 or a zero diagonal (a control point without residuals, an intrinsic nothing
 * constrains) returns ECB_FAILED with summary->deficient_index = j and writes no covariance; deficient_index is -1 otherwise.
 * With constant intrinsics (ecb_cost_set_constant_intrinsics) Z is conditional on them: their rows and columns of cov_intrinsics and
 * cov_cross are exact zeros, they are never deficient, and dimension (the D of sigma2) counts the free parameters only. */
typedef struct {
    double cost, sigma2, min_relative_pivot;  /* sigma2 is NaN when n_residuals <= dimension */
    int64_t n_residuals;
    int32_t dimension, deficient_index;
} ecb_covariance_summary;
int ecb_covariance(ecb_ctx *ctx, int n_splines, const int32_t *n_cp, const double *intrinsics, const double *rot_cp,
                   const double *trans_cp, const void *d_packed, int64_t n_residuals_total, double *cov_intrinsics, double *cov_band,
                   double *cov_cross, ecb_covariance_summary *summary);

/* ---- uncertainty of the trajectory: 6 x 6 covariance of the pose at any time on the spline ------------------------------
 * For a time t, let s be the first segment whose knot range holds t (EventCalibSpline::time2splineIdx) and i its span.  The
 * pose (R^, t^) at t is what EventCalibSpline::evaluate returns for the rotation model in use.  The tangent of the output is
 * dtheta (body frame, R = R^ Exp(dtheta), radians) then dp = t - t^ (world frame, units of the translation control points).
 * cov = Sigma(t) = J Z_blk J^T with J (6 x 24) the derivative of (dtheta, dp) with respect to the tangent parameters of control
 * points i-3 .. i in the order and rotation model of ecb_covariance, and Z_blk their 24 x 24 block of Z.  No sigma^2 scaling:
 * the covariance is sigma2 Sigma (sigma2 of ecb_covariance_summary).
 * Uses the Z and x of the last successful ecb_covariance on ctx (with several GPUs every rank holds the same Z bit for bit);
 * ECB_ERR_STATE without one, or when ecb_cost_setup or ecb_cost_set_rotation_model ran after it.
 *   pose[n][7] = tx ty tz qx qy qz qw (the order of TrajectoryByEvent.txt); cov[n][36] = Sigma row major, exactly symmetric.
 *   pose and cov may each be NULL.  A time outside every segment, or NaN, gives a NaN row and is not counted in *n_valid.
 *   n == 0 is valid, n < 0 returns ECB_ERR_ARG.  A query's output does not depend on the batch it is in.  FP64.
 * ecb_pose_covariance takes host arrays (staged through device buffers); ecb_pose_covariance_device takes device arrays and is
 * asynchronous on the context's stream unless n_valid (a host pointer, may be NULL) is asked for. */
int ecb_pose_covariance(ecb_ctx *ctx, const double *times, int64_t n, double *pose, double *cov, int64_t *n_valid);
int ecb_pose_covariance_device(ecb_ctx *ctx, const double *d_times, int64_t n, double *d_pose, double *d_cov, int64_t *n_valid);

/* ---- motion of the trajectory: angular velocity, velocity and acceleration at any time on the spline ------------------------
 * For a time t, s, i and the pose (R^, t^) are those of ecb_pose_covariance.  Nd_j and Ndd_j are the first and second time
 * derivatives of the cubic basis functions N_{i-3..i} on the same clamped knots (NURBS-book A2.3, BsplineReal::dersBasisFuns).
 *   w_b  body-frame angular velocity, R^T dR/dt = [w_b]x, radians per time unit: quaternion model 2 vec(q~^* (x) q~') / |q~|^2
 *        with q~ = sum N_j Q_j, q~' = sum Nd_j Q_j; SO(3) model sum_k b'_k (E_{k+1} .. E_3)^T d_k with E_k = Exp(b_k d_k), d_k =
 *        Log(R_{k-1}^-1 R_k) and b' the cumulative sum of Nd.
 *   v_w  = sum Nd_j T_j (world frame, translation units per time unit); a_w = sum Ndd_j T_j (per time unit squared).
 *   motion[n][16] = tx ty tz qx qy qz qw (the pose of ecb_pose_covariance, bit for bit), wx wy wz, vx vy vz, ax ay az.
 *   cov[n][81] = Sigma_m(t) = J Z_blk J^T over (w_b, v_w, a_w), row major, exactly symmetric.  J (9 x 24) is the derivative with
 *   respect to the tangent parameters of control points i-3 .. i in the order and rotation model of ecb_covariance: per control
 *   point j a block d w_b / d delta_j, Nd_j I3 and Ndd_j I3.  No sigma^2 scaling, as for ecb_pose_covariance.
 * Every output pointer may be NULL.  A time outside every segment, or NaN, gives a NaN row and is not counted in *n_valid.
 * n == 0 is valid, n < 0 returns ECB_ERR_ARG.  A query's output does not depend on the batch it is in.  FP64.
 * The host variants take host arrays (staged through device buffers); the _device variants take device arrays and are
 * asynchronous on the context's stream unless n_valid (a host pointer, may be NULL) is asked for.
 * ecb_trajectory_motion[_device]: the motion at the control points rot_cp / trans_cp (host arrays, layout of ecb_cost_eval),
 * in the rotation model of the context; needs ecb_cost_setup only (ECB_ERR_STATE before it), no covariance. */
int ecb_trajectory_motion(ecb_ctx *ctx, const double *rot_cp, const double *trans_cp, const double *times, int64_t n,
                          double *motion, int64_t *n_valid);
int ecb_trajectory_motion_device(ecb_ctx *ctx, const double *rot_cp, const double *trans_cp, const double *d_times, int64_t n,
                                 double *d_motion, int64_t *n_valid);
/* ecb_motion_covariance[_device]: the motion and Sigma_m at the x of the last successful ecb_covariance on ctx, with its Z; the
 * ECB_ERR_STATE rules of ecb_pose_covariance. */
int ecb_motion_covariance(ecb_ctx *ctx, const double *times, int64_t n, double *motion, double *cov, int64_t *n_valid);
int ecb_motion_covariance_device(ecb_ctx *ctx, const double *d_times, int64_t n, double *d_motion, double *d_cov,
                                 int64_t *n_valid);

/* ---- camera-gyroscope calibration: rotation, time offset and bias from the trajectory's angular velocity ---------------------
 * Gyroscope sample i: stamp t_i (gyroscope clock, time units of the knots) and reading w_g,i (radians per time unit, gyroscope
 * frame).  Model, with w_c the body-frame (camera) angular velocity of ecb_trajectory_motion in the context's rotation model:
 *   w_g,i = R_gc w_c(t_i + d) + b + noise
 *   R_gc rotates camera-frame vectors into the gyroscope frame; d is the time offset (gyroscope stamp t is event time t + d); b the
 *   bias (radians per time unit).  Residual r_i = R_gc w_c(t_i + d) + b - w_g,i, cost = 1/2 sum |r_i|^2 (no robust loss).
 *   Parameters (delta, d, b) with R_gc = Exp(delta) R^_gc (left perturbation, gyroscope frame); Jacobian of r_i
 *   [ -[R^ w_c]x, R^ dw_c/dt, I3 ].  The trajectory is held fixed: the result is conditional on the spline, whose own
 *   covariance is not propagated.
 * Used samples: t_i and w_g,i finite, and t_i - D and t_i + D (D = max_offset) in the same segment (the first whose knot range
 * holds the time).  The set is fixed for the whole call.  Unsorted stamps are allowed.
 * 1. Scan: offsets d_m = D (2m - (M-1)) / (M-1), m = 0 .. M-1 (M = n_offsets, odd, d = 0 on the grid; M = 1: d_0 = 0) and
 *    cost_m = sum_used (|w_c(t_i + d_m)| - |w_g,i|)^2 / n_used (norms: no rotation needed).  scan_offset = d_m of the least cost
 *    (ties: the lowest m).
 * 2. Horn's closed-form rotation from the centred cross-covariance of (w_c(t_i + scan_offset), w_g,i), then b = mean w_g -
 *    R mean w_c.
 * 3. Levenberg-Marquardt on (delta, d, b), 7 parameters, or 6 when D = 0 (d held at exactly 0): the trust-region rules of
 *    ecb_lm on a dense Cholesky, with the tolerances and iteration limit of ecb_lm_default_options; the parameter and function
 *    tolerances are tested after a step is accepted (the last successful step is kept); a candidate with |d| > D is rejected
 *    like a cost increase.
 * 4. cov = Z = (J^T J)^-1 at the solution, 7 x 7 row major over (delta, d, b), not scaled (the covariance is sigma2 Z); with 6
 *    parameters the offset's row and column are 0.  sigma2 = 2 cost / (3 n_used - n_params), std = sqrt(sigma2 diag Z),
 *    rms = sqrt(sum |r_i|^2 / (3 n_used)).
 * Sums are deterministic (fixed-order reductions, no floating-point atomics): repeated calls are bit-identical.  FP64.
 * ECB_FAILED (out->status says why; out is filled as far as it was computed): fewer used samples than parameters
 * (ECB_GYRO_TOO_FEW_SAMPLES); the scan's least cost at m = 0 or M-1 with M > 1 (ECB_GYRO_OFFSET_AT_EDGE: widen max_offset);
 * J^T J rank deficient, least relative Cholesky pivot < 1e-12, e.g. motion about one axis only (ECB_GYRO_RANK_DEFICIENT: cov and
 * std NaN).
 * rot_cp: rotation control points (layout of ecb_cost_eval); gyro[n][4] = t wx wy wz.  offset_cost[n_offsets] (cost_m) and
 * residuals[n][3] (r_i at the solution, NaN rows for unused samples) may be NULL.  Needs ecb_cost_setup (ECB_ERR_STATE before it).
 * ECB_ERR_ARG: ctx, out or rot_cp NULL, n < 0, gyro NULL with n > 0, max_offset NaN, negative or infinite, n_offsets even, < 1 or
 * > 65535, n_offsets > 1 with max_offset 0, or n_offsets 1 with max_offset > 0. */
#define ECB_GYRO_OK 0
#define ECB_GYRO_TOO_FEW_SAMPLES 1
#define ECB_GYRO_OFFSET_AT_EDGE 2
#define ECB_GYRO_RANK_DEFICIENT 3
typedef struct {
    double q_gc[4];      /* R_gc as x y z w */
    double offset;       /* d */
    double bias[3];
    double cov[49];      /* Z over (delta, d, b), not scaled by sigma2 */
    double std[7];       /* sqrt(sigma2 diag Z) */
    double sigma2, cost, rms;
    double scan_offset;  /* the offset of the scan's least cost */
    int64_t n_used, n_unused;
    int32_t iterations, termination;  /* LM iterations and ECB_LM_* code */
    int32_t n_params, status;         /* 7, or 6 with max_offset = 0; ECB_GYRO_* */
} ecb_gyro_calibration;
int ecb_gyro_calibrate(ecb_ctx *ctx, const double *rot_cp, const double *gyro, int64_t n, double max_offset, int32_t n_offsets,
                       ecb_gyro_calibration *out, double *offset_cost, double *residuals);

#ifdef __cplusplus
}
#endif
#endif /* EVENTCALIB_B200_H */

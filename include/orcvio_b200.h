/*
 * orcvio_b200 -- C ABI of the B200-native OrcVIO filter-update path.
 *
 * The reference has no plugin/FFI layer: callers link liborcvio_estimator and call
 * the C++ class orcvio::OrcVIO directly (reference include/orcvio/orcvio.h:39-119,
 * CMakeLists.txt:76-83).  This header is the C-ABI shape of that class for the hot
 * path: plain pointers and sizes, column-major double matrices where the reference
 * passes Eigen::MatrixXd, no C++/torch types.  INTEGRATION.md shows the thin
 * Eigen facade a maintainer would put on top to keep the class signature.
 *
 * Every entry point runs its arithmetic in hand-written sm_100a CUDA kernels
 * (orcvio_b200/csrc).  There is no CPU fallback: without a CUDA device every compute
 * call returns ORCVIO_ERR_NO_DEVICE and prints the reason to stderr.
 */
#ifndef ORCVIO_B200_H
#define ORCVIO_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define ORCVIO_OK 0
#define ORCVIO_ERR_NO_DEVICE -1
#define ORCVIO_ERR_ARG -2
#define ORCVIO_ERR_CONFIG -3
#define ORCVIO_ERR_UNSUPPORTED -4
#define ORCVIO_ERR_CUDA -5
#define ORCVIO_ERR_CAPACITY -6

/* One tracked image feature: field-for-field MonoFeatureMeasurement
 * (reference include/orcvio/feat/feature_msg.h:14-44). */
typedef struct {
  unsigned long long id;
  double u, v;
  double u_init, v_init;
  double u_vel, v_vel;
  double u_init_vel, v_init_vel;
} OrcvioFeature;

/* One IMU sample: ImuData (reference include/sensors/ImuData.hpp:16-39). */
typedef struct {
  double t;
  double gyro[3];
  double acc[3];
} OrcvioImu;

/* Snapshot of the IMU state and of what the reference's getters return
 * (getTbw/getVel/getPpose/getPvel, reference src/orcvio.cpp:2962-3026). */
typedef struct {
  long long state_id;
  double time;
  double R[9];        /* body->world, row-major */
  double p[3];
  double v[3];
  double bg[3];
  double ba[3];
  double P_pose[36];  /* [p, theta] ordering, row-major (getPpose) */
  double P_vel[9];
  int n_clones;
  int dim;            /* covariance dimension D = 22 + 6 n_clones */
  int n_map_features; /* size of the map server */
} OrcvioState;

/* Per-frame counters for parity tests (which features were consumed and how). */
typedef struct {
  int n_candidates_lost;     /* MSCKF candidates of removeLostFeatures */
  int n_tri_invalid_lost;
  int n_gate_pass_lost;
  int n_candidates_prune;
  int n_tri_invalid_prune;
  int n_gate_pass_prune;
  int n_removed_clones;
  long long removed_ids[2];
  int zupt;                  /* 1: the frame took a zero-velocity update (checkZUPTFeat / checkZUPTIMU) */
  double zupt_chi2;          /* checkZUPTIMU only: chi2 of the stationarity test and |v| it was compared with */
  double zupt_vnorm;
} OrcvioFrameStats;

typedef struct orcvio_handle orcvio_handle;
typedef struct orcvio_batch orcvio_batch;

/* ---- orcvio::OrcVIO class mirror ------------------------------------------------- */
/* OrcVIO::OrcVIO(std::string& config_file), src/orcvio.cpp:45-50 */
/* Parses a config/*.yaml with the reader orcvio_initialize uses (OrcVIO::loadParameters, src/orcvio.cpp:62-415) and
 * says whether this path runs it: ORCVIO_OK, ORCVIO_ERR_CONFIG (unreadable) or ORCVIO_ERR_UNSUPPORTED, with the reason
 * in `why`.  Needs no device. */
int orcvio_config_check(const char* config_yaml_path, char* why, int why_cap);
orcvio_handle* orcvio_create(const char* config_yaml_path);
void orcvio_destroy(orcvio_handle* h);
/* OrcVIO::initialize(), src/orcvio.cpp:418-497.  1 = ok, 0 = yaml unreadable/unsupported. */
int orcvio_initialize(orcvio_handle* h);
/* initial_use_gt semantics (src/orcvio.cpp:514-544) for configs whose yaml has no GT block:
 * the static/dynamic initialisers are out of scope, so the caller supplies the state. */
int orcvio_set_initial_state(orcvio_handle* h, double t, const double quat_xyzw[4], const double p[3],
                             const double v[3], const double bg[3], const double ba[3]);
/* OrcVIO::processFeatures(msg, imu_msg_buffer), src/orcvio.cpp:500-661.
 * `imu` is the caller's buffer of *n_imu samples; like the reference the consumed prefix is
 * erased: the remaining samples are moved to the front and *n_imu is updated.
 * Returns 1 (published), 0 (not yet initialised / no IMU ahead of the image), <0 error. */
int orcvio_process_features(orcvio_handle* h, double t_img, const OrcvioFeature* feats, int n_feats,
                            OrcvioImu* imu, int* n_imu);
int orcvio_get_state(orcvio_handle* h, OrcvioState* out);
/* state_server.state_cov, column-major D x D (symmetric).  cap = capacity in doubles. */
int orcvio_get_cov(orcvio_handle* h, double* P, int cap, int* D);
/* getSwPoses, src/orcvio.cpp:3030-3042: per clone R (9, row-major) + p (3); ids optional. */
int orcvio_get_window(orcvio_handle* h, double* poses12, long long* ids, double* times, int cap);
/* getTcw, src/orcvio.cpp:2978-2988: camera pose (camera -> world rotation, row-major, and camera position) of the
 * clone of the current state id. */
int orcvio_get_tcw(orcvio_handle* h, double R_c2w[9], double t_c_w[3]);
/* The pose log processFeatures appends to (output_dir + "state_est_geo_feat.txt", src/orcvio.cpp:422, 640-645): one
 * "t tx ty tz qx qy qz qw" line per published frame, t relative to take-off.  path = NULL or "" closes it. */
int orcvio_set_pose_log(orcvio_handle* h, const char* path);
/* getMSCKFMapPointPositions, src/orcvio.cpp:3059-3062 */
int orcvio_get_map_points(orcvio_handle* h, long long* ids, double* xyz, int cap);
/* state_server.feature_states (hybrid MSCKF / EKF-SLAM mode, max_features_in_one_grid > 0), in state order: feature id,
 * state id of its anchor clone, inverse depth and obs_anchor (x, y) in the anchor camera (feature.hpp:243-246), world
 * position.  Column 22 + 6 N + k of the covariance belongs to entry k.  This is what getStableMapPointPositions /
 * getActiveMapPointPositions (src/orcvio.cpp:3046-3058) are served from. */
int orcvio_get_feature_states(orcvio_handle* h, long long* ids, long long* anchor_ids, double* inv_depth,
                              double* obs_anchor, double* xyz, int cap);
/* EKF-SLAM branches of the last frame (diagnostics / parity surface).  what = 0: features dropped from the state because
 * they were lost (src/orcvio.cpp:2221-2232; ids);  1: features of the state updated with their 2 rows (:2449-2495; ids,
 * flags = gate pass, gamma);  2: candidate new features (:2343-2446; ids, flags = entered the state, gamma of the MSCKF
 * gate);  3: anchor changes in pruneImuStateBuffer (:2665-2722; ids = triples feature id, old anchor, new anchor --
 * cap counts entries, i.e. 3 per change).  Returns the number of entries written. */
int orcvio_get_hybrid_log(orcvio_handle* h, int what, long long* ids, int* flags, double* gamma, int cap);
int orcvio_get_frame_stats(orcvio_handle* h, OrcvioFrameStats* out);
/* per-candidate log of the last frame: ids, phase (0 lost / 1 prune), status bits
 * (1 = triangulation valid, 2 = gate pass), gamma. */
int orcvio_get_candidate_log(orcvio_handle* h, long long* ids, int* phase, int* status, double* gamma,
                             int cap);

/* OrcVIO::constructObjectResidualJacobians, src/orcvio.cpp:2017-2151.
 * jac_sensor: rows x 6, Hf: rows x odim, res: rows (all column-major, in); outputs
 * Hx_out (rows x D), Hf_out (rows x odim), res_out with *rows_out valid rows.
 * Returns 1 if at least one timestamp is in the window, 0 otherwise. */
int orcvio_construct_object_jacobians(orcvio_handle* h, const double* jac_sensor, int rows,
                                      const double* timestamps, int n_ts, const double* Hf, int odim,
                                      const double* res, const int* zs_num, const double* cam_pose_se3,
                                      double* Hx_out, double* Hf_out, double* res_out, int* rows_out);
/* OrcVIO::removeLostObjects, src/orcvio.cpp:2154-2193.  Returns 1 updated, 0 rejected
 * (status_out: 0 updated, 1 empty, 2 disabled, 3 nullspace fail, 4 gate fail, 5 nan). */
int orcvio_remove_lost_objects(orcvio_handle* h, const double* Hx, const double* Hf, const double* res,
                               int rows, int odim, int* status_out, double* gamma_out);
/* test hooks, include/orcvio/orcvio.h:101-119 */
int orcvio_set_state_cov(orcvio_handle* h, int imu_dim, int num_clone);
int orcvio_set_win_pose_timestamps(orcvio_handle* h, const double* ts, int n);
int orcvio_fix_dcampose_dimupose_to_i(orcvio_handle* h);
/* overwrite the full filter state (parity tests start both sides from one snapshot) */
int orcvio_set_cov(orcvio_handle* h, const double* P, int D);

/* ---- multi-trajectory batch (SURVEY 8e): n independent filters advanced in lock-step -- */
orcvio_batch* orcvio_batch_create(const char* config_yaml_path, int n_filters);
void orcvio_batch_destroy(orcvio_batch* b);
int orcvio_batch_set_initial_state(orcvio_batch* b, int i, double t, const double quat_xyzw[4],
                                   const double p[3], const double v[3], const double bg[3],
                                   const double ba[3]);
/* One frame for every filter.  feats/imu are concatenated per filter with CSR offsets
 * (n_filters + 1 entries).  imu_used[i] receives the number of consumed IMU samples
 * (the prefix the reference would erase).  published[i] = processFeatures' return. */
int orcvio_batch_process(orcvio_batch* b, const double* t_img, const OrcvioFeature* feats,
                         const int* feat_off, const OrcvioImu* imu, const int* imu_off, int* imu_used,
                         int* published);
/* Whole-sequence replay of every filter of the batch (Monte-Carlo / multi-sequence replay, SURVEY 8e): the lock-step
 * loop over the frames runs inside the library, one orcvio_batch_process per frame.  Filter i: frames t_img[i*n_frames + f],
 * features feats[i][feat_off[i*(n_frames+1) + f] .. feat_off[i*(n_frames+1) + f + 1]), IMU stream imu[i][0 .. n_imu[i]);
 * before frame f the samples up to t_img + imu_window are offered, the filter consumes a prefix.  poses_out:
 * n_filters x n_frames x 7 (p, q xyzw -- a line of the reference's state_est_geo_feat.txt); ok_out[i] = every frame
 * published.  Several batches may replay concurrently from different host threads. */
int orcvio_batch_replay(orcvio_batch* b, int n_frames, const double* t_img, const OrcvioFeature* const* feats,
                        const int* feat_off, const OrcvioImu* const* imu, const int* n_imu, double imu_window,
                        double* poses_out, int* ok_out);
/* orcvio_batch_replay that also records what filter consistency needs.  state17_out: n_filters x n_frames x 17 = t (the
 * IMU state's own time), p (3), q xyzw (4), v (3), bg (3), ba (3) after every frame.  cov15_out: n_filters x n_frames x
 * 225, the leading 15 x 15 block of the covariance (error state [theta, v, p, b_g, b_a], row-major) after every frame,
 * captured on the device and downloaded once at the end of the call.  Either may be NULL; with both NULL this is
 * orcvio_batch_replay. */
int orcvio_batch_replay_states(orcvio_batch* b, int n_frames, const double* t_img, const OrcvioFeature* const* feats,
                               const int* feat_off, const OrcvioImu* const* imu, const int* n_imu, double imu_window,
                               double* poses_out, int* ok_out, double* state17_out, double* cov15_out);
/* Object pose initialisation, first step (ObjectFeatureInitializer::single_object_initialization without RANSAC,
 * src/obj/ObjectFeatureInitializer.cpp:99-111): findTransform (:265-341) -- similarity fit of the mean-shape keypoints
 * onto the triangulated ones, scale from the polyline lengths, rotation by Kabsch -- and, with se2_flag,
 * poseSE32SE2 (include/orcvio/utils/se3_ops.hpp:272-300) for a batch of objects on the device.  Points: 3 doubles
 * each, object o owns [off[o], off[o+1]); wTq16_out: row-major 4 x 4 per object; ok_out[o] = 0 for a degenerate
 * object (fewer than two points, zero-length polyline).  Host pointers. */
int orcvio_object_kabsch_init(const double* mean_pts, const double* world_pts, const int* off, int n_obj, int se2_flag,
                              double* wTq16_out, int* ok_out);
/* Object state optimiser (SURVEY 8f rank 2), the step immediately before stage 3, for a batch of n_obj objects of ONE
 * class (K <= 12 keypoints).  Object o owns the frames [frame_off[o], frame_off[o+1]): frames_wTc (16 doubles each,
 * row-major camera-to-world), zs (K x 2 per frame, NaN = keypoint not observed), zb (xmin ymin xmax ymax per frame).
 * Host pointers.
 *
 * orcvio_object_init = ObjectFeatureInitializer::single_object_initialization without RANSAC
 * (src/obj/ObjectFeatureInitializer.cpp:33-111): every keypoint observed in more than 3 frames is triangulated linearly
 * with the last observing frame as the anchor (single_triangulation_common, src/feat/FeatureInitializer.cpp:6-110);
 * with more than 3 such keypoints wTq = findTransform(mean, world) [poseSE32SE2 with se2_flag], else identity and
 * ok = 0.  kp_world_out (n_obj x K x 3, NaN where not triangulated) and kp_valid_out (n_obj x K) may be NULL. */
int orcvio_object_init(int n_obj, const int* frame_off, const double* frames_wTc, const double* zs, int K,
                       const double* kps_mean, int se2_flag, double* wTq16_out, int* ok_out, double* kp_world_out,
                       int* kp_valid_out);
/* orcvio_object_lm = ObjectFeatureInitializer::single_levenberg_marquardt up to the optimum (:346-381): minimises the
 * ObjectLM functor (keypoint reprojection, bounding-box / quadric, deformation and shape regularisers, weights4,
 * src/obj/ObjectLM.cpp:761-816) over (wTo, shape, keypoints) with the reference's Levenberg-Marquardt (factor 10),
 * started from (wTo_init, mean_shape, kps_mean).  flags: bit0 left perturbation, bit1 new bbox residual.
 * Outputs per object: wTo (16), shape (3), keypoints in the object frame (K x 3) and in the world frame
 * (transform_mean_keypoints_to_global; may be NULL), status = LevenbergMarquardtSpace::Status (success = not 0 / 5),
 * nfev, njev, |f| (each may be NULL), rounds_out = lock-step rounds = kernel launches (may be NULL).  The rows the
 * filter consumes at the optimum come from orcvio_object_residuals. */
int orcvio_object_lm(int n_obj, const int* frame_off, const double* frames_wTc, const double* zs, const double* zb, int K,
                     const double* kps_mean, const double* mean_shape, const double* weights4, int flags,
                     const double* wTo_init, double* wTo_out, double* shape_out, double* kps_out, double* kps_world_out,
                     int* status_out, int* nfev_out, int* njev_out, double* fnorm_out, int* rounds_out);
/* One evaluation of the ObjectLM model at given states (n_obj x [wTo 16 | shape 3 | keypoints 3K]):
 * out = n_obj x [|f| | J^T f (n) | J^T J (n x n)], n = 9 + 3K -- ObjectLM::operator() and ::df reduced to what the
 * optimiser consumes. */
int orcvio_object_lm_eval(int n_obj, const int* frame_off, const double* frames_wTc, const double* zs, const double* zb,
                          int K, const double* kps_mean, const double* mean_shape, const double* weights4, int flags,
                          const double* states, double* out);
/* The reference's two Levenberg-Marquardt known-answer problems (src/tests/test_levenberg_marquardt.cpp:64-140) through
 * the library's driver; which = 0: lmder1 example (x_out 3), 1: the quadratic (x_out 1); 2 / 3: MINPACK's Rosenbrock and
 * Freudenstein-Roth test functions from their standard starting points with lmder1's settings (x_out 2), whose answers
 * the CPU tests take from the real MINPACK (scipy.optimize.leastsq).  Needs no device. */
int orcvio_lm_known_answer(int which, double* x_out, int* status, int* nfev, int* njev, double* fnorm);
/* The reference's trajectory logger (System::publishGroundtruth, ros_wrapper/src/orcvio/src/System.cpp:885-943) for a
 * batch of trajectories, on the device: first-pose SE(3) alignment, then per trajectory the mean orientation error
 * (deg), mean position error (m), position RMSE (m) and final position error (m) -> out4 (n_traj x 4).  Poses are
 * n_traj x n_frames x 7 (p, q xyzw, Hamilton), host pointers. */
int orcvio_trajectory_metrics(const double* est_pose7, const double* gt_pose7, int n_traj, int n_frames, double* out4);
/* NEES of a batch of filter runs against their truth, on the device.  est17 / gt17: n_traj x n_frames x 17 (layout of
 * state17_out), cov15: n_traj x n_frames x 225 (cov15_out), host pointers.  flags: bit0 use_larvio, bit1
 * use_left_perturbation (the orientation error is Log(R R_est^T) if either is set, else Log(R_est^T R); v, p and the
 * biases are true - estimate).  nees8_out (n_traj x n_frames x 8): NEES of theta (dof 3), v (3), p (3), pose [theta, p]
 * (6), navigation [theta, v, p] (9), full IMU state (15), then |dtheta| in degrees and |dp| in metres; NaN when the
 * 15 x 15 block is not positive definite or an input is not finite.  summary9_out (n_frames x 9, may be NULL): per frame
 * over the valid trajectories, the ANEES of the six blocks, the RMS orientation error (deg), the RMS position error (m)
 * and the number of valid trajectories (fixed-order reduction: the same rows give the same bits).  The 95 % bounds of
 * the ANEES of a block of dof d over N runs are orcvio_chi2_quantile(0.025 | 0.975, N d) / N. */
int orcvio_trajectory_nees(const double* est17, const double* gt17, const double* cov15, int n_traj, int n_frames,
                           int flags, double* nees8_out, double* summary9_out);
/* summary9_out of orcvio_trajectory_nees from NEES rows alone (n_traj x n_frames x 8), e.g. rows gathered from several
 * ranks: the same kernel, so the same rows give the same bits as the summary of orcvio_trajectory_nees. */
int orcvio_nees_summary(const double* nees8, int n_traj, int n_frames, double* summary9_out);
/* The reference's KITTI-style relative error (python_scripts/trajectory_eval/traj_eval.py:61-90 -> the vendored
 * rpg_trajectory_evaluation: compute_trajectory_errors.py:10-67, trajectory.py:341-377, 309-339) for a batch of
 * trajectories on the device: for every sub-trajectory length the pairs (start, first pose closest to start + length
 * along the ground truth, tolerance 0.2 length) and the error of the relative motion.  out4: n_traj x n_len x 4 =
 * (samples, mean translation error in % of the length, mean rotation error in deg / m, mean translation error in m);
 * trans_error_pct (n_traj, may be NULL): write_kitti_errors_to_yaml's "TransError(%)".  scale (n_traj, may be NULL = 1):
 * the scale of the alignment, which the package applies to the estimated relative translation (sim3 only).  Poses as
 * above, n_frames <= 4096. */
int orcvio_kitti_relative_error(const double* est_pose7, const double* gt_pose7, int n_traj, int n_frames,
                                const double* lengths, int n_len, const double* scale, double* out4,
                                double* trans_error_pct);
/* Trajectory.align_trajectory + the translation part of compute_absolute_error of the same package (trajectory.py:211-275,
 * align_trajectory.py:27-79): Umeyama alignment gt ~ s R est + t over all frames, method 0 = "sim3", 1 = "se3" (s = 1),
 * for a batch of trajectories on the device.  out15 per trajectory: s, R (9, row-major), t (3), mean and rmse of the
 * absolute translation error (the mean is the "RMSE(m)" of write_kitti_errors_to_yaml). */
int orcvio_trajectory_align_ate(const double* est_pose7, const double* gt_pose7, int n_traj, int n_frames, int method,
                                double* out15);
int orcvio_batch_get_state(orcvio_batch* b, int i, OrcvioState* out);
int orcvio_batch_get_cov(orcvio_batch* b, int i, double* P, int cap, int* D);
int orcvio_batch_get_frame_stats(orcvio_batch* b, int i, OrcvioFrameStats* out);
/* consumed MSCKF features (gate-passed, both phases) summed over filters since creation */
long long orcvio_batch_feature_updates(orcvio_batch* b);
/* number of kernel launches issued since creation */
long long orcvio_batch_kernel_launches(orcvio_batch* b);

/* ---- stage-level entry points on a frozen snapshot (parity tests, stress bench) ------- */
/* Stage 1: Feature::checkMotion + triangulate_position (feature.hpp:353-396, 583-719) for
 * n_feat features; feature f uses observations [feat_off[f], feat_off[f+1]) whose camera
 * poses are cam_R (row-major 3x3, cam->world) / cam_t of clone obs_clone[k].
 * out_pos: world positions (3 per feature), out_status bit0 = valid, out_iters: outer/inner
 * iteration counts (2 per feature) for control-flow parity. */
int orcvio_triangulate(const double* cam_R, const double* cam_t, int n_clones, const int* feat_off,
                       const int* obs_clone, const double* obs_z, int n_feat, double translation_threshold,
                       double cost_threshold, double init_final_dist_threshold, double* out_pos,
                       int* out_status, int* out_iters, double* out_cost);

/* Stages 1,2,4,5 on one frozen window ("stack -> compress -> update", SURVEY 8d):
 * triangulate every feature, Jacobian + nullspace + gate, compression in the whitened form,
 * EKF update of (state, P).  clone_R/clone_p: body poses; P: D x D with D = 22 + 6 n_clones.
 * flags: bit0 use_larvio, bit1 use_left_perturbation, bit2 discard_large_update; any other bit
 * set is rejected with ORCVIO_ERR_ARG (the same flags, and the same check, for
 * orcvio_measurement_jacobians and orcvio_frame_create, which returns NULL).
 * Outputs (any may be NULL): P_out, delta_x (D), status per feature (bit0 tri valid, bit1
 * gate pass), gamma per feature, positions, updated clone poses (N x 12).  timings_us[8]:
 * device time per stage measured with CUDA events (tri, jac+gate, A = H' L, A^T A + Cholesky
 * of W, posterior, total) when non-NULL. */
int orcvio_snapshot_update(const double* clone_R, const double* clone_p, int n_clones,
                           const double* R_b2c, const double* t_c_b, const double* P_in,
                           const int* feat_off, const int* obs_clone, const double* obs_z, int n_feat,
                           int flags, double noise_feature_var, double chi2_p,
                           double translation_threshold, double cost_threshold,
                           double init_final_dist_threshold, double* P_out, double* delta_x,
                           int* status, double* gamma, double* positions, double* clone_out,
                           float* timings_us, int repeat);

/* Persistent form of orcvio_snapshot_update for a stream of frames (no allocation per call):
 * the same stages 1,2,4,5 -- removeLostFeatures' "stack -> compress -> update" chain,
 * src/orcvio.cpp:2498-2560 + measurementUpdate_hybrid :1766-1950 -- on one frame.
 *   orcvio_frame_update : host buffers in, host buffers out (H2D + kernels + D2H), the call a
 *                         host integration makes per frame;
 *   orcvio_frame_load / _run / _fetch : upload once, run the kernel chain `repeat` times on the
 *                         HBM-resident frame (each run restores the pristine window first),
 *                         device time in microseconds via CUDA events. */
typedef struct orcvio_frame orcvio_frame;
orcvio_frame* orcvio_frame_create(int n_clones_cap, int flags, double noise_feature_var, double chi2_p,
                                  double translation_threshold, double cost_threshold,
                                  double init_final_dist_threshold);
void orcvio_frame_destroy(orcvio_frame* f);
int orcvio_frame_update(orcvio_frame* f, const double* clone_R, const double* clone_p, int n_clones,
                        const double* R_b2c, const double* t_c_b, const double* P_in, const int* feat_off,
                        const int* obs_clone, const double* obs_z, int n_feat, double* P_out,
                        double* delta_x, int* status, double* gamma, double* clone_out);
/* Same call when the caller keeps the covariance on the device between frames: instead of the whole posterior
 * (D x D: 326 KB at 30 clones) only its leading 9 x 9 block comes back -- what getPpose / getPvel
 * (src/orcvio.cpp:3000-3027) are computed from -- row-major into P_lead9 (81 doubles). */
int orcvio_frame_update_pose_cov(orcvio_frame* f, const double* clone_R, const double* clone_p, int n_clones,
                                 const double* R_b2c, const double* t_c_b, const double* P_in, const int* feat_off,
                                 const int* obs_clone, const double* obs_z, int n_feat, double* P_lead9,
                                 double* delta_x, int* status, double* gamma, double* clone_out);
int orcvio_frame_load(orcvio_frame* f, const double* clone_R, const double* clone_p, int n_clones,
                      const double* R_b2c, const double* t_c_b, const double* P_in, const int* feat_off,
                      const int* obs_clone, const double* obs_z, int n_feat);
int orcvio_frame_run(orcvio_frame* f, int repeat, float* total_us, float* stage_us6);
int orcvio_frame_fetch(orcvio_frame* f, double* P_out, double* delta_x, int* status, double* gamma,
                       double* clone_out);
long long orcvio_frame_kernel_launches(orcvio_frame* f);
/* wall-clock split (us) of the last orcvio_frame_update: host work-list build + uploads, kernel launches,
 * wait + downloads, total -- explains the gap between the device-timed and the end-to-end figure */
int orcvio_frame_host_times(orcvio_frame* f, float* us4);
/* device time (us, CUDA events, mean over the last profiled orcvio_frame_run) of the two kernels the
 * stage split does not isolate: us2[0] = k_syrk (W = s^2 I + A^T A on the FP64 tensor cores, the
 * roofline kernel of bench.py), us2[1] = k_chol_prior (second stream, overlaps stages 1-2) */
int orcvio_frame_kernel_times(orcvio_frame* f, float* us2);

/* Stage 2 only, for element-wise parity of J1 (measurementJacobian_msckf, orcvio.cpp:1071-1168):
 * per observation H_x (2x6), H_e (2x6), H_f (2x3), r (2), row-major. */
int orcvio_measurement_jacobians(const double* clone_R, const double* clone_p, int n_clones,
                                 const double* R_b2c, const double* t_c_b, const double* positions,
                                 const int* feat_off, const int* obs_clone, const double* obs_z,
                                 int n_feat, int flags, double* Hx, double* He, double* Hf, double* r);

/* Hybrid EKF-SLAM feature rows, stage level (SURVEY 8a H1 / H2; feature_idp_dim 1, no Schmidt, no FEJ).
 * H1, measurementJacobian_ekf_1didp (orcvio.cpp:1356-1478): feature f is anchored in clone anchor[f] with inverse
 * depth inv_depth[f] along the anchor-frame bearing (f_an[2f], f_an[2f+1], 1); positions[3f..] is its world
 * position as the map server holds it.  Per observation (CSR feat_off / obs_clone / obs_z), row-major:
 * H_f (2), H_a (2x6, anchor pose), H_x (2x6, observing clone), H_e (2x6, extrinsics), r (2); an observation taken
 * by the anchor clone itself returns zeros (:1433-1441). */
int orcvio_ekf_measurement_jacobians(const double* clone_R, const double* clone_p, int n_clones,
                                     const double* R_b2c, const double* t_c_b, const int* anchor,
                                     const double* inv_depth, const double* f_an, const double* positions,
                                     const int* feat_off, const int* obs_clone, const double* obs_z, int n_feat,
                                     double* H_f, double* H_a, double* H_x, double* H_e, double* r);

/* H2, featureJacobian_ekf (orcvio.cpp:1575-1651) + gatingTestFeature with dof 2 (:1953-1976): the n_feat features
 * of the state (feature f = state column 22 + 6 n_clones + f) observed at z_cur[2f..] by the newest clone.
 * P: D x D covariance, D = 22 + 6 n_clones + n_feat (symmetric: row- or column-major).
 * Outputs: H (2 n_feat x D, row-major), r (2 n_feat), gamma (n_feat), pass (n_feat). */
int orcvio_ekf_feature_rows(const double* clone_R, const double* clone_p, int n_clones, const double* R_b2c,
                            const double* t_c_b, const int* anchor, const double* inv_depth, const double* f_an,
                            const double* positions, const double* z_cur, int n_feat, const double* P, int D,
                            double noise_var, double chi2_p, double* H, double* r, double* gamma, int* pass);

/* H4, updateFeatureCov_1didp (orcvio.cpp:3611-3773): feature feat_idx (state column 22 + 6 n_clones + feat_idx) moves its
 * anchor from clone old_idx to clone new_idx; p_w is its world position, inv_depth_new its inverse depth already
 * expressed in the new anchor.  P (D x D, symmetric) is updated in place: the feature's row / column becomes J P
 * (J P J^T on the diagonal).  J_out (D) optionally receives the 1 x D Jacobian. */
int orcvio_ekf_update_feature_cov(double* P, int D, const double* clone_R, const double* clone_p, int n_clones,
                                  const double* R_b2c, const double* t_c_b, int feat_idx, int old_idx, int new_idx,
                                  const double* p_w, double inv_depth_new, double* J_out);

/* H4, rmLostFeaturesCov (orcvio.cpp:3776-3828): P without the row / column of feature feat_idx, (D-1) x (D-1). */
int orcvio_ekf_remove_feature_cov(const double* P, int D, int n_clones, int feat_idx, double* P_out);

/* H2 + H3: featureJacobian_ekf_new (orcvio.cpp:1481-1572) and the new-feature sparsification of removeLostFeatures
 * (:2413-2443) for n_feat features about to enter the state (inputs as orcvio_ekf_measurement_jacobians; D = legacy state
 * dimension).  Per feature the rows of its non-anchor observations are reflected so that its (single-column) feature
 * part becomes h_2 e_0: H_1 (n_feat x D), h_2 (n_feat: the diagonal of H_2), r_1 (n_feat) are the initialisation rows of
 * measurementUpdate_hybrid; H_o (rows_out x D) / r_o the remaining, feature-free rows, in feature order. */
int orcvio_ekf_new_feature_rows(const double* clone_R, const double* clone_p, int n_clones, const double* R_b2c,
                                const double* t_c_b, const int* anchor, const double* inv_depth, const double* f_an,
                                const double* positions, const int* feat_off, const int* obs_clone,
                                const double* obs_z, int n_feat, int D, double* H_1, double* h_2, double* r_1,
                                double* H_o, double* r_o, int* rows_out);

/* The new-state part of measurementUpdate_hybrid (orcvio.cpp:1823-1832, 1903-1941; no Schmidt): P (D x D) and dx_leg (D)
 * are the posterior covariance and correction of the legacy state; HH = H_2^-1 H_1, dx_new = -HH dx_leg + H_2^-1 r_1,
 * P_aug ((D + n_new)^2) = [[P, -P HH^T], [-HH P, HH P HH^T + noise_var (H_2^T H_2)^-1]], symmetrised. */
int orcvio_ekf_delayed_init(const double* P, int D, const double* dx_leg, const double* H_1, const double* h_2,
                            const double* r_1, int n_new, double noise_var, double* dx_new, double* P_aug);

/* stateAugmentation (orcvio.cpp:963-1010) / the covariance part of pruneImuStateBuffer (:2916-2940) on a state with
 * feature states behind the n_clones clones (D = 22 + 6 n_clones + E): the new clone block (J P J^T, J = theta and p of the
 * IMU state) is inserted BEFORE the feature block -> P_out (D+6)^2, symmetrised; a clone's 6 rows / columns are dropped ->
 * P_out (D-6)^2. */
int orcvio_ekf_augment_cov(const double* P, int D, int n_clones, double* P_out);
int orcvio_ekf_remove_clone_cov(const double* P, int D, int n_clones, int clone_idx, double* P_out);

/* Legacy-state part of measurementUpdate_hybrid (orcvio.cpp:1808-1820, 1884-1901) on a state WITH inverse-depth feature
 * states behind the clones: P is D x D (D = 22 + 6 N + E <= 208, symmetric, rows / columns 15..21 zero), H the stacked
 * H_o (rows x D, row-major; its columns 0..21 are ignored: P is zero under the extrinsic columns and vision rows do not
 * touch the IMU block), r its residual.  dx = K r (D) and P_out = (I - K H) P, symmetrised (D x D). */
int orcvio_hybrid_update_dense(const double* P, int D, const double* H, const double* r, int rows, double noise_var,
                               double* dx, double* P_out);

/* Stage 3 (O1-O4): keypoint + bbox residuals and Jacobians of one object over T frames.
 * frames_wTc: T x 16 (row-major 4x4), wTo 16, shape 3, kps K x 3, zs T x K x 2 (NaN = not
 * observed), zb T x 4.  flags: bit0 left perturbation, bit1 new bbox residual.
 * Outputs: fvec (rows), fjac_cam (rows x 6, column-major), fjac_obj (rows x (9+3K),
 * column-major), zs_num (T), cam_pose_se3 (6 x T column-major), rows_out. */
int orcvio_object_residuals(const double* frames_wTc, int T, const double* wTo, const double* shape,
                            const double* kps, int K, const double* zs, const double* zb, int flags,
                            double* fvec, double* fjac_cam, double* fjac_obj, int* zs_num,
                            double* cam_pose_se3, int* rows_out);

/* Stage 6: IMU propagation of (state, P) over n samples (processModel, orcvio.cpp:727-823).
 * state16: R(9) v(3) p(3) + time at [15]; biases bg, ba; flags as above.
 * noise4: gyro, acc, gyro-bias, acc-bias variances. */
int orcvio_propagate(double* state16, const double* bg, const double* ba, const double* gyro_old,
                     const double* acc_old, const OrcvioImu* imu, int n, double* P, int D, int flags,
                     const double* noise4);

/* Host-side probe of the split-K plan of the compression GEMM (no device needed): out[0] rows per chunk, out[1] column
 * tiles, out[2] tile pairs, out[3] work units, out[4 .. 4 + pairs] first unit of every pair followed by the total,
 * out[15] rows per chunk of a diagonal pair (16 ints). */
int orcvio_syrk_plan_probe(int arows, const int* jrow0, int n_clones, int cta_budget, int* out);

/* device / build info */
int orcvio_device_count(void);
/* select the CUDA device used by handles created afterwards on this thread (one process per GPU) */
int orcvio_set_device(int device);
const char* orcvio_version(void);
/* measured FP64 peaks of the current device (TFLOP/s): plain DFMA and mma.sync m8n8k4 (DMMA);
 * the roofline denominators for the FP64 kernels (MEASURED_PEAKS.json carries only HBM / bf16) */
int orcvio_fp64_peak(double* dfma_tflops, double* dmma_tflops);
/* dependent-chain latencies in cycles: DFMA, sqrt, divide, rsqrt, shared load, __syncthreads(512), shuffle */
int orcvio_latency_probe(double* cycles7);
/* single-warp dependent latencies (cycles): DFMA, DMMA dependent, DMMA with 2 / 4 / 8 independent accumulators
   (per MMA), 64-bit shuffle + add, 16-byte shared load, fence.acq_rel.cta after a shared store, rcp.approx.f64, 0 */
int orcvio_latency_probe1(double* cycles10);
/* test / profiling hook: the one-CTA Cholesky both factorisation kernels are built on (csrc/chol.cuh).
 * A: m x m SPD row-major, X: nx x m carried rows; L: m x m lower factor, Xs = X C^-T; prof: 64 x 8
 * clock64() stamps per 8-column panel (may be NULL); us: mean kernel time over `reps` launches. */
int orcvio_chol_probe(int m, int nx, const double* A, const double* X, double* L, double* Xs,
                      long long* prof, int reps, float* us);
/* chi-square quantile used for the gating tables (boost::math::quantile(chi_squared(dof), p),
 * src/orcvio.cpp:481-494) */
double orcvio_chi2_quantile(double p, int dof);
/* per-kernel-class device time (ms) and counts accumulated while profiling is on:
 * tri, jac+gate, qr tiles, qr chain, update, propagate+augment */
int orcvio_batch_set_profiling(orcvio_batch* b, int on);
int orcvio_batch_get_phase_times(orcvio_batch* b, double* ms6, long long* n6);

/* ---- on-disk and wire formats either side of the path (host code, no device needed) ------------------------------
 * EuRoC / ASL csv files as the reference's app reads them (include/utils/DataReader.hpp:30-140): header line skipped,
 * time stamps in ns -> s, IMU rows "t, wx, wy, wz, ax, ay, az".  Return the number of rows in the file (rows beyond
 * `cap` are counted, not stored), or a negative error code. */
int orcvio_read_imu_csv(const char* path, OrcvioImu* out, int cap);
int orcvio_read_image_list_csv(const char* path, double* t_out, char* names, int name_stride, int cap);
/* Ground-truth csv (DatasetReader::load_gt_file, include/orcvio/dataset_reader.h:64-101): rows of 17 doubles
 * [t (s), q (4), p (3), v (3), b_gyro (3), b_accel (3)]; orcvio_gt_lookup is get_gt_state (:111-140): the state whose
 * stamp is closest to t when that is within 5 ms, else only an exact match; returns 1 when found. */
int orcvio_read_gt_csv(const char* path, double* out17, int cap);
int orcvio_gt_lookup(const double* gt17, int n, double t, double out17[17]);
/* The pose log of processFeatures (src/orcvio.cpp:640-645; written by orcvio_set_pose_log): rows of 8 doubles. */
int orcvio_read_pose_log(const char* path, double* out8, int cap);
/* orcvio_ros_msgs/ObjectLM (ros_wrapper/src/orcvio_ros_msgs/msg/ObjectLM.msg) in ROS 1 wire serialisation, matrices
 * as tf::matrixEigenToMsg lays them out (two dimensions, row-major): residual (rows x 1), jacobian_wrt_object_state
 * (rows x odim), jacobian_wrt_sensor_state (rows x 6), valid_camera_pose_mat (6 x n_poses), timestamps, zs_num --
 * exactly the arguments of constructObjectResidualJacobians.  pack returns the message length (buf may be NULL to
 * size it); unpack checks the layout and returns ORCVIO_OK. */
int orcvio_objectlm_pack(long long object_id, const double* residual, int rows, const double* jac_object, int odim,
                         const double* jac_sensor, const double* cam_pose_se3, int n_poses, const double* timestamps,
                         int n_ts, const int* zs_num, int n_zs, unsigned char* buf, int cap);
int orcvio_objectlm_unpack(const unsigned char* buf, int len, long long* object_id, double* residual, int* rows,
                           double* jac_object, int* odim, double* jac_sensor, double* cam_pose_se3, int* n_poses,
                           double* timestamps, int* n_ts, int* zs_num, int* n_zs, int cap_rows, int cap_odim, int cap_n);

#ifdef __cplusplus
}
#endif
#endif /* ORCVIO_B200_H */

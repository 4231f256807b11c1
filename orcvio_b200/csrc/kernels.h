// Shared kernel-side declarations: device data layouts, work-list records, launchers.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <algorithm>
#include "dmath.cuh"

namespace ob {

// ------------------------------------------------------------------ capacities / layouts
#define ORCVIO_MAX_OBS 32        // observations per feature == clones in the window (<= 32)
#define ORCVIO_LEG 22            // LEG_DIM (calib_imu_instrinsic = 0)

// clone record (doubles): body pose + cached camera pose (IMUState_Aug, imu_state.h:100-153)
constexpr int CL_R = 0;          // R body->world, row-major 3x3
constexpr int CL_P = 9;          // position
constexpr int CL_RC = 12;        // orientation_cam = R cam->world
constexpr int CL_PC = 21;        // position_cam
constexpr int CL_STRIDE = 24;

// IMU state record (doubles)
constexpr int IM_R = 0, IM_V = 9, IM_P = 12, IM_BG = 15, IM_BA = 18, IM_RBC = 21, IM_TCB = 30,
              IM_TD = 33, IM_TIME = 34, IM_ROLD = 35, IM_VOLD = 44, IM_POLD = 47, IM_GOLD = 50,
              IM_AOLD = 53, IM_DISCARDS = 56, IM_STRIDE = 64;

constexpr int FP_STRIDE = 4;     // feature position slot: x, y, z, pad
constexpr int FI_STRIDE = 4;     // inverse-depth record of a slot (hybrid mode): inv depth, obs_anchor x, y, pad

// filter flags
constexpr int FL_LARVIO = 1, FL_LEFT = 2, FL_DISCARD_LARGE = 4;

// candidate status bits
constexpr int ST_TRI_VALID = 1, ST_GATE_PASS = 2;
// candidate flags
constexpr int CAND_FORCE_TRI = 1;
constexpr int CAND_GATE_ONLY = 2;   // new EKF-SLAM feature: MSCKF rows only decide its gate (src/orcvio.cpp:2365-2370)

struct TriCfg {                  // Feature::OptimizationConfig, feature.hpp:41-63
  double translation_threshold, huber_epsilon, estimation_precision, initial_damping;
  int outer_max, inner_max;
  double cost_threshold, init_final_dist_threshold;
};

// One MSCKF candidate feature of one filter (built by the host bookkeeping every frame).
struct Cand {
  int filter;                    // filter index inside the batch
  int slot;                      // feature slot (position table)
  long long gen;                 // track serial: slot is initialised iff fgen[slot] == gen
  int flags;
  int tri_off, tri_m;            // observations used by the triangulation
  int jac_off, jac_m;            // observations used by the Jacobian / gate
  int row_off;                   // first row of this feature in its filter's stacked H
  int hblk_off;                  // offset (doubles) of its compact r x w block
  int s_blk, e_blk;              // first / last clone index touched by the Jacobian rows
  int cm_first_clone, cm_last_clone;   // checkMotion: first and last(-or-second-to-last) obs
  double cm_zu, cm_zv;           // first observation
};

struct TriArgs {
  const Cand* cand; int n_cand;
  const double* clones; size_t clone_stride;     // per-filter stride in doubles
  double* fpos; long long* fgen; int fcap;       // per-filter feature tables
  const int* obs_clone; const double* obs_z;
  TriCfg cfg;
  int* status; int* iters; double* cost;
  double* final_pos;             // optional, 3 per candidate: the solution in the last camera used (the anchor frame of
                                 // initializeInvParamPosition, feature.hpp:536-547)
  // direct mode (end-to-end frame call): when feat_off != nullptr the kernel runs over the caller's features in
  // their own order (candidate c == feature c, slot c, forced triangulation) without any Cand record, so it can
  // start while the host still sorts the candidates and builds the tiles; status is then indexed by feature
  const int* feat_off;
  int direct_n_clones, direct_n_obs;   // direct mode: bounds the kernel checks itself (it may start before the host
                                       // has validated the caller's lists; a malformed feature is just invalid)
  // per-candidate completion flags (optional): done[c] = epoch once the candidate's results are visible device-wide.
  // The Jacobian kernel, launched behind this one with programmatic stream serialisation, starts its candidates one by
  // one as they finish instead of waiting for the slowest LM chain of the grid.
  int* done; int epoch;
};

struct JacArgs {
  const Cand* cand; const int* cand_list; int n_list;   // indirection: size-class lists
  const double* clones; size_t clone_stride;
  const double* imu; const double* fpos; int fcap;
  const double* P; size_t p_stride; int ldp;
  const int* obs_clone; const double* obs_z;
  int flags; double sigma2; const double* chi2;  // chi2[dof], dof < 500
  int* status; double* gamma;
  const int* tri_status_f;                       // != nullptr: triangulation status by feature slot (direct mode)
  const int* tri_done; int tri_epoch;            // != nullptr: per-candidate completion flags of k_triangulate (see TriArgs)
  // direct mode (end-to-end frame call): feat_off != nullptr -> list entries are FEATURE indices of the caller's
  // list, the candidate record is derived on the fly (offsets of the feature's rows / block from rowoff_f /
  // hblkoff_f), status and gamma are indexed by feature
  const int* feat_off; const int* rowoff_f; const int* hblkoff_f;
  double* hblk; double* rblk;                    // compact projected blocks / residuals
  // optional raw per-observation outputs (orcvio_measurement_jacobians)
  double* raw_Hx; double* raw_He; double* raw_Hf; double* raw_r;
};

// Row tile of the stacked Jacobian: one CTA of k_aform forms its rows of the whitened matrix A.
struct Tile {
  int filter;
  int cand_begin, cand_end;      // candidates (sorted by s_blk inside a filter)
  int rows;                      // rows if every candidate passes the gate
  int c0_blk, c1_blk;            // clone-block window [c0, c1)
  int arow;                      // first row of this tile in the stacked A matrix
};

struct FilterWork {              // per filter, per update
  int N;                         // clones
  int D;                         // 22 + 6N (+ E inverse-depth feature states behind the clones: dense hybrid update)
  int tile_begin, tile_end;      // tiles of this filter, sorted by c0_blk
  int wmax_blk;                  // widest tile window (blocks)
  int active;                    // 0: skip this filter's update entirely
  int arow0, arows;              // rows of this filter in the stacked A matrix (upper bound)
  int jrow0[4];                  // staircase of A: first row (relative to arow0) with a structural non-zero in
                                 // column tile J (64 columns) of A; rows above it are skipped by k_syrk
  int dense_rows;                // dense rows behind the tiles' rows (hybrid mode: rows of the EKF-SLAM features)
};

struct AformArgs {               // inputs of k_aform: the gated rows of every tile
  const Cand* cand; const int* status;
  const int* status_f;                           // != nullptr: status by feature slot (direct-mode Jacobian pass)
  // direct mode (end-to-end frame call): no candidate records on the device at all -- order_f[c] is the feature
  // behind sorted candidate c, the rest comes from the per-feature arrays the early Jacobian pass already uses
  const int* order_f; const int* feat_off; const int* rowoff_f; const int* hblkoff_f; const int* sblk_f;
  const int* eblk_f;
  const double* hblk; const double* rblk;
  const Tile* tiles;
  const FilterWork* fw;
};

struct UpdArgs {
  const FilterWork* fw; int n_filters;
  double* P; size_t p_stride; int ldp;
  size_t r_stride; int ldr;                              // per-filter stride and ld of S
  double* T; double* S; size_t t_stride; int ldt;        // T: n x D, S: n x n (ld = ldr)
  double* yv;                                            // C^-1 v, per filter (ldr)
  double* imu; double* clones; size_t clone_stride;
  double* dx; int lddx;                                  // delta_x log per filter
  int flags; double sigma2;
};

// scratch of the whitened-form update (info_kernel.cu)
struct InfoBufs {
  double* Ls;            // per filter 22 x 22 : IMU block factor given the clones
  double* Amat;          // stacked A = [r' | H' L], lda = ldr (residual in column 0)
  double* part;          // split-K partials of A^T A: [filter][work unit][64 x 64]
  int max_units, cta_budget, group;        // part layout [filter][max_units]; SMs x waves; chunks per reduction group
  unsigned int* syrk_cnt; // split-K arrival counters [filter][SY_MAXP][1 + SY_MAXG] (zero between launches)
  int* tile_rows;        // gated rows per tile
  int* filter_rows;      // gated rows per filter (0 -> posterior == prior, P is left untouched)
  cudaEvent_t ls_done;   // recorded on the side stream behind k_imu_factor (Ls); the main stream waits for it before k_pinfo
};

struct PropSample { double t, w[3], a[3]; };

struct PropArgs {
  double* P; size_t p_stride; int ldp;
  double* imu;
  const PropSample* samples; const int* samp_off;        // CSR per filter
  const int* D;                                          // per filter current dimension
  int n_filters; int flags;
  double qc[4];                                          // gyro, acc, gyro-bias, acc-bias variances
};

struct AugArgs {
  double* P; size_t p_stride; int ldp;
  const double* imu; double* clones; size_t clone_stride;
  const int* N; int n_filters;                           // N = clones BEFORE augmentation
  const int* E;                                          // EKF-SLAM feature states behind the clones (nullptr: none)
};

struct RemoveArgs {
  double* P; size_t p_stride; int ldp;
  double* clones; size_t clone_stride;
  const int* N;                                          // clones before removal
  const int* rm;                                         // 2 per filter, ascending, -1 = none
  int n_filters;
  const int* E;                                          // EKF-SLAM feature states behind the clones (nullptr: none)
};

// Zero-velocity update (zupt_kernel.cu): checkZUPTIMU + measurementUpdate_ZUPT_vpq, src/orcvio.cpp:3129-3454
struct ZuptArgs {
  double* P; size_t p_stride; int ldp;
  double* imu; double* clones; size_t clone_stride;
  const PropSample* samples; const int* samp_off;        // imu_recent_zupt = the samples of this frame
  const int* N;                                          // clones AFTER augmentation (< 2: no ZUPT)
  const int* mode;                                       // 0 none, 1 update (feature test passed), 2 IMU chi2 test
  const double* chi2_check;                              // per filter chi2 threshold of the IMU test
  int* decision;                                         // out: 1 = the ZUPT update was applied
  double* info;                                          // out, 2 per filter: chi2, |v| of the IMU test
  double* dx; int lddx;
  int n_filters; int flags;
  double noise_v, noise_p, noise_q;                      // zupt_noise_{v,p,q}^2
};

// ---------------------------------------------------------------- hybrid MSCKF / EKF-SLAM mode (hybrid_kernel.cu)
// Features of the state (1-D inverse depth in an anchor clone, src/orcvio.cpp:1356-1651) and candidates for it.
struct HybFeat {                 // feature i of the state (column 22 + 6N + i), in state order; all are tracked now
  int slot, anchor;              // feature slot; clone index of the anchor
  double zu, zv;                 // its observation in the newest clone
};
struct HybNew {                  // candidate new EKF-SLAM feature (tracked long, its grid cell has room)
  int slot, anchor;
  int cand;                      // its gate-only MSCKF candidate (status decides whether it enters the state)
  int obs_off, obs_m;            // all of its observations in the observation pool
  int row_off;                   // first of its 2 (m - 1) - 1 dense rows (relative to the filter's dense rows)
};
struct HybWork {                 // per filter and frame
  int N, E;                      // clones; feature states before this frame's new ones
  int feat_begin, feat_end;      // HybFeat range (E entries)
  int new_begin, new_end;        // HybNew range
  int dense_off;                 // first dense row of this filter in the dense-row buffer
  int n_dense;                   // dense rows reserved: 2 E + sum over new candidates
  int arow_dense;                // row of the stacked A matrix where the dense rows go (relative to the filter's rows)
  int active;
};
struct HybArgs {
  const HybWork* hw; int n_filters;
  const HybFeat* feats; const HybNew* news;
  const double* clones; size_t clone_stride; const double* imu;
  double* fpos; double* fidp; int fcap;
  double* P; size_t p_stride; int ldp;
  const int* obs_clone; const double* obs_z;
  const int* status;             // candidate status (gate of the new candidates)
  double sigma2; double chi2_dof2;
  double* Hd; int ldh;           // dense rows [n | r] (window columns 22.., residual in column n = D - 22)
  double* H1; double* h2; double* r1; int new_cap;   // initialisation rows of the survivors, per filter new_cap
  double* scratch;               // unreflected rows of one new candidate at a time, per filter 64 x ldh
  int* ekf_pass; double* ekf_gamma;                  // per HybFeat
  int* new_ok;                                       // per HybNew: 1 = entered the state
  int* n_new;                                        // per filter: survivors
  const double* dx; int lddx;
};
void launch_hybrid_rows(const HybArgs& a, cudaStream_t s);
void launch_hybrid_aform(const HybArgs& a, const double* FT, size_t t_stride, int ldt, double* Amat, int lda,
                         const FilterWork* fw, int max_dense, cudaStream_t s);
void launch_hybrid_post(const HybArgs& a, cudaStream_t s);   // feature increments + delayed initialisation
// features only: invDepth += dx, world positions (after measurementUpdate_msckf of the prune phase)
void launch_hybrid_feature_increment(const HybArgs& a, cudaStream_t s);
// initializeInvParamPosition took the branch: the speculative solution of candidate `cand` becomes the position of
// slot (= filter * fcap + slot), serial gen; idp record <- its anchor-frame solution
struct CommitRec { int cand, slot; long long gen; };
void launch_hybrid_commit(const CommitRec* recs, int n, const double* final_pos, const double* spec_pos, double* fpos,
                          long long* fgen, double* fidp, cudaStream_t s);
// P <- P[keep, keep]: newidx (per filter ldp ints) maps an old state index to its new one, -1 = dropped
void launch_compact_cov(double* P, size_t p_stride, int ldp, const int* newidx, const int* D_old, int n_filters,
                        cudaStream_t s);
struct ReanchorRec {             // anchor change of one feature (src/orcvio.cpp:2665-2773, 3611-3773)
  int filter, slot, col;         // col >= 0: feature of the state (covariance row / column replaced); -1: outside
  int old_idx, new_idx;          // clone indices
  double zu, zv;                 // col < 0: the stored observation in the new anchor becomes obs_anchor
};
void launch_reanchor(const ReanchorRec* recs, const int* rec_off, int n_filters, const HybWork* hw,
                     const double* clones, size_t clone_stride, const double* imu, const double* fpos, double* fidp,
                     int fcap, double* P, size_t p_stride, int ldp, cudaStream_t s);
// host mirror of the EKF features: out[6 k ..] = position (3), inv depth, obs_anchor (2) of slots[k]
void launch_hybrid_gather(const int* filt, const int* slots, int n, const double* fpos, const double* fidp, int fcap,
                          double* out, cudaStream_t s);

// Records (and prints) a launch-configuration error; Batch polls launch_error_count().
void check_launch(const char* name);
int launch_error_count();
int env_int(const char* name, int dflt);   // tuning knobs (ORCVIO_* environment variables)

// Programmatic dependent launch (sm_90+): a kernel launched with launch_pdl() may be scheduled while the previous
// kernel of its stream is still running (once every CTA of that kernel has called pdl_launch_dependents() or
// exited); it runs its prologue (shared-memory zeroing, index arithmetic on host-provided lists) and then blocks in
// pdl_wait() until the previous kernel has completed and its writes are visible.  Launched the ordinary way the two
// device calls are no-ops.  Measured on the frame chain (B200, 2000 / 4096 features): no gain (207 -> 213 us, 252 -> 261 us),
// so the attribute is OFF by default; ORCVIO_PDL=1 turns it on.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <class... KArgs, class... Args>
inline void launch_pdl_if(bool on, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                          Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = on ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
template <class... KArgs, class... Args>
inline void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  static const int pdl_on = env_int("ORCVIO_PDL", 0);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl_on ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
#endif

void launch_triangulate(const TriArgs& a, cudaStream_t s);
void launch_jac_gate(const JacArgs& small_list, const JacArgs& large_list, cudaStream_t s);
void launch_info_update(const AformArgs& q, const UpdArgs& u, const InfoBufs& ib, int n_tiles, int max_tile_rows,
                        int max_w_blk, int max_N, cudaStream_t s, cudaStream_t s2, cudaEvent_t fork,
                        cudaEvent_t join, cudaEvent_t mid1, cudaEvent_t mid2, int* launches,
                        bool prior_in_flight = false, cudaEvent_t mid_syrk = nullptr, cudaEvent_t prior_t0 = nullptr,
                        cudaEvent_t prior_t1 = nullptr, int max_E = 0, const struct HybArgs* hyb = nullptr,
                        int max_dense = 0);
void launch_info_prior(const UpdArgs& u, const InfoBufs& ib, int max_N, cudaStream_t s2, cudaEvent_t fork,
                       cudaEvent_t join, cudaEvent_t t0 = nullptr, cudaEvent_t t1 = nullptr, int max_E = 0);
// System::publishGroundtruth for a batch of trajectories (metrics_kernel.cu); host pointers, pose = p (3) + q xyzw (4)
int trajectory_metrics(const double* est_pose7, const double* gt_pose7, int n_traj, int n_frames, double* out4);
// KITTI-style relative error (rpg_trajectory_evaluation as the reference's traj_eval.py calls it); host pointers
int kitti_relative_error(const double* est_pose7, const double* gt_pose7, int n_traj, int n_frames, const double* lengths,
                         int n_len, const double* scale, double* out4, double* trans_error_pct);
int umeyama_ate(const double* est_pose7, const double* gt_pose7, int n_traj, int n_frames, int known_scale, double* out15);
// filter consistency (consistency_kernel.cu): the leading 15 x 15 block of every filter's P into hist[filter, frame]
// (queued on the batch stream after a frame); NEES / ANEES of state records against the truth (host pointers)
void launch_capture_imu_cov(const double* P, size_t p_stride, int ldp, int n_filters, double* hist, int n_frames,
                            int frame, cudaStream_t s);
int trajectory_nees(const double* est17, const double* gt17, const double* cov15, int n_traj, int n_frames, int flags,
                    double* nees8, double* summary9);
int nees_summary(const double* nees8, int n_traj, int n_frames, double* summary9);
// findTransform (+ poseSE32SE2) for a batch of objects (kabsch_kernel.cu); host pointers
int kabsch_init(const double* mean_pts, const double* world_pts, const int* off, int n_obj, int se2, double* wTq16, int* ok);
// object state optimiser (objlm_kernel.cu); host pointers
int object_init(int n_obj, const int* frame_off, const double* frames_wTc, const double* zs, int K, const double* kps_mean,
                int se2, int min_obs, double* wTq16, int* ok, double* kp_world, int* kp_valid);
int object_lm(int n_obj, const int* frame_off, const double* frames_wTc, const double* zs, const double* zb, int K,
              const double* kps_mean, const double* mean_shape, const double* weights4, int flags, const double* wTo_init,
              double* wTo_out, double* shape_out, double* kps_out, double* kps_world_out, int* status, int* nfev,
              int* njev, double* fnorm, int* rounds_out);
int object_lm_eval(int n_obj, const int* frame_off, const double* frames_wTc, const double* zs, const double* zb, int K,
                   const double* kps_mean, const double* mean_shape, const double* weights4, int flags, const double* xs,
                   double* out);
int lm_known_answer(int which, double* x_out, int* status, int* nfev, int* njev, double* fnorm);
int syrk_debug_read(long long* out, int cap);   // ORCVIO_SYRK_DBG=1: phase time stamps of the last k_syrk launch
void launch_info_dense_factor(const UpdArgs& u, const InfoBufs& ib, const double* Hp, int ldh, int rows, int n,
                              cudaStream_t s);
void launch_info_dense_apply(const UpdArgs& u, const InfoBufs& ib, int n, cudaStream_t s);
void launch_project_dense(double* M, int rows, int ld, int nelim, int ncols, cudaStream_t s);
void launch_object_rows(const double* frames_wTc, int T, const double* wTo, const double* shape, const double* kps,
                        int K, const double* zs, const double* zb, int flags, const int* kp_row_off, int rows_kp,
                        int rows, double* fvec, double* fjac_cam, double* fjac_obj, double* cam_pose_se3,
                        cudaStream_t s);
void launch_object_construct(const double* jac_sensor, const double* Hf, const double* res, int rows_in, int odim,
                             const int* map5, const double* dcam_dimu, int n_kept, int leg, int D, int rows_out,
                             double* Hx_out, double* Hf_out, double* res_out, cudaStream_t s);
void launch_propagate(const PropArgs& a, cudaStream_t s);
void launch_augment(const AugArgs& a, cudaStream_t s);
void launch_remove(const RemoveArgs& a, cudaStream_t s);
void launch_zupt(const ZuptArgs& a, cudaStream_t s);

// tile sizing shared by host tiler and kernels
constexpr int QR_THREADS = 256;         // CTA of k_project_dense; candidates per tile (k_aform's rowbase[256])
constexpr int AFORM_TILE_ROWS = 64;     // row cap of a tile
// Split-K plan of W = s^2 I + A^T A for ONE filter (k_syrk).  A^T A is computed as 64 x 64 tiles (I <= J) over
// chunks of rows; column tile J of A is structurally zero above row jrow0[J] (features are sorted by first
// clone and A = H' L with L lower triangular), so pair (I, J) only covers rows [jrow0[J], arows).  The plan
// picks the rows per chunk (multiple of 32, >= 128) so that the work units of all pairs fill `cta_budget`
// (= SMs x waves).  A function of the filter alone: the chunking fixes the summation order, so a filter
// gives bit-identical results whether it runs alone or inside a batch.
constexpr int SY_TILE = 64, SY_MAXT = 4, SY_MAXP = 10, SY_MAXG = 32;
struct SyrkPlan {
  int kc, kcd, nt, npairs, total;   // rows per chunk of an off-diagonal / a diagonal pair
  int first[SY_MAXP + 1];        // first work unit of every pair (pair order: I outer, J >= I inner)
};
// A diagonal pair (I, I) only computes the 36 of its 64 8 x 8 fragments that are ever emitted (k_syrk), so its chunks
// are longer for the same time: 13/8 as measured (a 64-row slab of a diagonal unit costs 1.13 x its share of DMMAs).
// At the minimum chunk length (a frame of a few hundred rows: far fewer units than SMs, nothing to balance) a
// diagonal pair keeps the chunk length of the others: shorter chunks = a flatter summation tree for W = s^2 I + A^T A,
// and W's rounding is what the update amplifies on an ill-conditioned window (scripts/soak_parity.py).
__host__ __device__ inline int syrk_kcd(int kc) { return kc <= 128 ? kc : (kc * 13 / 8 + 31) / 32 * 32; }
__host__ __device__ inline SyrkPlan syrk_plan(const FilterWork& fw, int cta_budget) {
  SyrkPlan p;
  p.nt = (fw.D - ORCVIO_LEG + 1 + SY_TILE - 1) / SY_TILE;
  if (p.nt > SY_MAXT) p.nt = SY_MAXT;
  p.npairs = p.nt * (p.nt + 1) / 2;
  int rowsJ[SY_MAXT];
  long long tot16 = 0;
  for (int J = 0; J < p.nt; ++J) {
    rowsJ[J] = fw.arows - fw.jrow0[J];
    if (rowsJ[J] < 0) rowsJ[J] = 0;
    tot16 += (long long)rowsJ[J] * (16 * J + 10);      // J off-diagonal pairs + 8/13 of a diagonal one
  }
  int kc = (int)((tot16 + 16LL * cta_budget - 1) / (16LL * cta_budget));
  kc = (kc + 31) / 32 * 32;
  if (kc < 128) kc = 128;
  for (;;) {
    const int kcd = syrk_kcd(kc);
    int total = 0, q = 0;
    for (int I = 0; I < p.nt; ++I)
      for (int J = I; J < p.nt; ++J) {
        const int k = (I == J) ? kcd : kc;
        int c = (rowsJ[J] + k - 1) / k;
        if (c < 1) c = 1;
        p.first[q++] = total;
        total += c;
      }
    p.first[q] = total;
    p.total = total;
    if (total <= cta_budget || total <= p.npairs) break;
    kc += 32;
  }
  p.kc = kc;
  p.kcd = syrk_kcd(kc);
  return p;
}

}  // namespace ob

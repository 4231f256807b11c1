// Host side of the filter: bookkeeping of the reference's OrcVIO class (map server,
// window of clones, per-frame classification) for a batch of independent filters that
// advance in lock-step, driving the CUDA kernels.  A single filter is a batch of one.
#pragma once
#include <cuda_runtime.h>

#include <cstring>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <unordered_map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/orcvio_b200.h"
#include "config.h"
#include "kernels.h"

namespace ob {

struct Obs {
  long long sid;      // state id of the observing clone
  double z[2];        // (u + u_vel dt, v + v_vel dt)
  double vel[2];
};

struct Track {        // struct Feature, reference include/orcvio/feat/feature.hpp:34-265
  long long id = 0;
  int slot = -1;
  long long gen = 0;
  std::vector<Obs> obs;     // ascending sid (std::map order in the reference)
  // first / last observing state id, kept beside the node so that the per-frame walks over every track can skip a
  // track without touching its observation array (touch() after every change of obs)
  long long first_sid = 0x7fffffffffffffffLL, last_sid = -1;
  void touch() {
    first_sid = obs.empty() ? 0x7fffffffffffffffLL : obs.front().sid;
    last_sid = obs.empty() ? -1 : obs.back().sid;
  }
  // hybrid mode (feature.hpp:243-264): the idp record itself lives on the device (slot), these are its host twins
  bool in_state = false, ekf_feature = false;
  bool initialized = false; // host twin of "fgen[slot] == gen" (only maintained in hybrid mode)
  long long id_anchor = -1;
  double mpos[3] = {0, 0, 0}, minv = 0, mobs[2] = {0, 0};   // mirror: world position, inverse depth, obs_anchor
};

struct CloneMeta {
  long long id;
  double time;
  double dt;
};

struct CandInfo {     // host-side twin of a device candidate
  long long id;
  int kind;           // 0 lost, 1 tracked-long, 2 prune
};

struct FilterHost {
  std::map<long long, Track> map_server;              // ordered by id: the reference walks its std::map in this order
  std::unordered_map<long long, Track*> track_index;  // id -> node of map_server (node addresses are stable): the lookups
  Track* find_track(long long id) const {
    auto it = track_index.find(id);
    return it == track_index.end() ? nullptr : it->second;
  }
  Track& add_track(Track&& tr) {
    const long long id = tr.id;
    Track& t = map_server.emplace(id, std::move(tr)).first->second;
    track_index[id] = &t;
    return t;
  }
  void erase_track(long long id) {
    track_index.erase(id);
    map_server.erase(id);
  }
  std::vector<CloneMeta> clones;
  std::vector<int> free_slots;
  long long next_state_id = 0;
  long long next_gen = 1;
  long long state_id = 0;
  double imu_time = 0.0;
  double dt = 0.0;
  double tracking_rate = 0.0;
  bool first_features = false, gravity_set = false, has_init = false;
  double init_t = 0, init_q[4] = {0, 0, 0, 1}, init_p[3] = {0, 0, 0}, init_v[3] = {0, 0, 0},
         init_bg[3] = {0, 0, 0}, init_ba[3] = {0, 0, 0};
  double take_off_stamp = 0.0;
  bool active = false;        // took part in the current frame
  bool if_zupt = false;
  std::vector<double> coarse_feature_dis;   // checkZUPTFeat input, filled by addFeatureObservations (:1052-1058)
  double zupt_chi2 = 0.0, zupt_vnorm = 0.0;  // checkZUPTIMU diagnostics of the last frame
  std::vector<double> imu_mirror;      // IM_STRIDE
  std::vector<double> clone_mirror;    // Ncap * CL_STRIDE
  std::vector<double> cur_window_timestamps;
  OrcvioFrameStats stats{};
  std::vector<CandInfo> cinfo[2];      // phase 0 (lost) / 1 (prune)
  std::vector<int> cstatus[2];
  std::vector<double> cgamma[2];
  // hybrid MSCKF / EKF-SLAM mode (state_server.feature_states, grid_map, last_ZUPT_time)
  std::vector<long long> feature_states;
  std::vector<long long> ekf_watch;     // features of the state + rejected new ones: the tracks with a host mirror
  double last_zupt_time = 0.0;
  // per-frame log of the EKF branches (test / diagnostics surface: orcvio_get_hybrid_log)
  std::vector<long long> log_ekf_lost, log_ekf_ids, log_new_ids;
  std::vector<int> log_ekf_pass, log_new_ok;
  std::vector<double> log_ekf_gamma, log_new_gamma;
  std::vector<long long> log_reanchor;  // triples: feature id, old anchor state id, new anchor state id
  // object-update test hooks (include/orcvio/orcvio.h:101-119)
  int leg_dim_override = -1;
  int num_clone_override = -1;
  bool dcampose_fixed = false;
};

struct Blob {                 // one pinned host blob + device twin, carved into sections
  char* dev = nullptr;
  size_t dev_cap = 0;
  char* pinned = nullptr;     // sections are written in place: no pageable staging copy
  size_t pinned_cap = 0;
  size_t used = 0;
  size_t reserve(size_t bytes) {
    size_t off = (used + 255) & ~size_t(255);
    const size_t old_used = used;
    used = off + bytes;
    if (used > pinned_cap) {
      char* np = nullptr;
      const size_t ncap = used * 2 + 4096;
      if (getenv("ORCVIO_HOST_PROF") && atoi(getenv("ORCVIO_HOST_PROF")) == 3)
        fprintf(stderr, "[replay prof] growth: pinned blob -> %.1f MB\n", ncap / 1048576.0);
      if (cudaMallocHost(&np, ncap) != cudaSuccess) { used = old_used; return 0; }
      if (pinned) {
        if (old_used) std::memcpy(np, pinned, old_used);
        cudaFreeHost(pinned);
      }
      pinned = np;
      pinned_cap = ncap;
    }
    return off;
  }
  void reset() { used = 0; }
  void ensure_pinned(size_t bytes) {      // grow the pinned half ahead of time (contents are not preserved)
    if (bytes <= pinned_cap) return;
    char* np = nullptr;
    const size_t ncap = bytes * 2 + 4096;
    if (cudaMallocHost(&np, ncap) != cudaSuccess) return;
    if (pinned) cudaFreeHost(pinned);
    pinned = np;
    pinned_cap = ncap;
  }
};

struct PhaseTimes {
  double tri = 0, jac = 0, qr_tiles = 0, qr_chain = 0, update = 0, prop = 0, aug = 0, remove = 0;
  long long n_tri = 0, n_jac = 0, n_qr_tiles = 0, n_qr_chain = 0, n_update = 0, n_prop = 0;
};

class Batch {
 public:
  Batch(const Params& p, int n_filters);
  ~Batch();
  bool ok() const { return ok_; }
  const std::string& error() const { return err_; }

  void set_initial_state(int i, double t, const double* q, const double* p, const double* v,
                         const double* bg, const double* ba);
  int process(const double* t_img, const OrcvioFeature* feats, const int* feat_off,
              const OrcvioImu* imu, const int* imu_off, int* imu_used, int* published);
  int process_ptrs(const double* t_img, const OrcvioFeature* const* feats, const int* n_feats,
                   const OrcvioImu* const* imu, const int* n_imu, int* imu_used, int* published);
  // state17_out / cov15_out (either may be NULL): the IMU state and the leading 15 x 15 block of P after every frame
  int replay(int n_frames, const double* t_img, const OrcvioFeature* const* feats, const int* feat_off,
             const OrcvioImu* const* imu, const int* n_imu, double imu_window, double* poses_out, int* ok_out,
             double* state17_out = nullptr, double* cov15_out = nullptr);
  int get_state(int i, OrcvioState* out);
  int get_cov(int i, double* P, int cap, int* D);
  int set_cov(int i, const double* P, int D);
  // getMSCKFMapPointPositions: world positions of the map-server features (NaN = not initialised)
  int get_map_points(int i, long long* ids, double* xyz, int cap);
  // state_server.feature_states in state order: id, anchor state id, inverse depth, obs_anchor (2), world position (3)
  int get_feature_states(int i, long long* ids, long long* anchors, double* inv_depth, double* obs_anchor, double* xyz,
                         int cap);
  FilterHost& filter(int i) { return f_[i]; }
  const Params& params() const { return p_; }
  long long feature_updates() const { return feature_updates_; }
  long long kernel_launches() const { return launches_; }
  double gpu_ms() const { return gpu_ms_; }
  void set_profiling(bool on) { profiling_ = on; }
  const PhaseTimes& phase_times() const { return pt_; }

  struct PhaseWork;
  // Stage-level entry on a frozen window (orcvio_triangulate / orcvio_measurement_jacobians /
  // orcvio_snapshot_update): loads the window into filter 0 and runs tri -> jac -> compression + update.
  struct SnapshotIO {
    const double* clone_R = nullptr; const double* clone_p = nullptr;   // body poses (or camera poses)
    bool poses_are_camera = false;
    int n_clones = 0;
    const double* R_b2c = nullptr; const double* t_c_b = nullptr;
    const double* P_in = nullptr;
    const double* positions_in = nullptr;   // when given: skip triangulation, use these
    const int* feat_off = nullptr; const int* obs_clone = nullptr; const double* obs_z = nullptr;
    int n_feat = 0;
    int stages = 0;                         // bit0 tri, bit1 jac+gate, bit2 compression+update
    bool early_prior = false;               // start k_chol_prior as soon as P is uploaded (end-to-end call)
    int repeat = 1;
    double* P_lead9 = nullptr;               // leading 9 x 9 block of the posterior (what getPpose / getPvel read)
    double* P_out = nullptr; double* delta_x = nullptr; int* status = nullptr; double* gamma = nullptr;
    double* positions = nullptr; double* clone_out = nullptr; float* timings_us = nullptr; int* iters = nullptr; double* cost = nullptr;
    double* raw_Hx = nullptr; double* raw_He = nullptr; double* raw_Hf = nullptr; double* raw_r = nullptr;
  };
  int run_snapshot(const SnapshotIO& io);
  // persistent three-step form used by the orcvio_frame_* entry points
  int snapshot_prepare(const SnapshotIO& io);
  int snapshot_execute(bool download);
  int snapshot_execute_plain(bool download, bool prior_in_flight);
  int snapshot_fetch(const SnapshotIO& io);
  void snapshot_stage_times(float* us6);
  float last_syrk_us() const { return last_syrk_us_; }     // k_syrk / k_chol_prior of the last profiled run
  float last_prior_us() const { return last_prior_us_; }
  void sync() { cudaStreamSynchronize(stream_); }
  cudaStream_t stream() const { return stream_; }
  void override_tricfg(double translation_threshold, double cost_threshold, double init_final) {
    tricfg_.translation_threshold = translation_threshold;
    tricfg_.cost_threshold = cost_threshold;
    tricfg_.init_final_dist_threshold = init_final;
  }
  void override_noise(double sigma2, double chi2_p);
  void override_flags(int flags) { flags_ = flags; }

  // stage 3, filter side (objects.cu)
  int construct_object_jacobians(int fi, const double* jac_sensor, int rows, const double* timestamps, int n_ts,
                                 const double* Hf, int odim, const double* res, const int* zs_num,
                                 const double* cam_pose_se3, double* Hx_out, double* Hf_out, double* res_out,
                                 int* rows_out);
  int object_update(int fi, const double* Hx, const double* Hf, const double* res, int rows, int odim,
                    int* status_out, double* gamma_out);
  // legacy-state part of measurementUpdate_hybrid on a state with feature columns (objects.cu)
  int dense_update(const double* P_in, int D, const double* H, const double* r, int rows, double* dx_out,
                   double* P_out);
  // stage 6 stand-alone (objects.cu)
  int propagate_standalone(double* state16, const double* bg, const double* ba, const double* gyro_old,
                           const double* acc_old, const OrcvioImu* imu, int n, double* P, int D,
                           const double* noise4);

  int Ncap() const { return Ncap_; }
  int ldp() const { return ldp_; }

 private:
  friend struct CApi;
  bool ok_ = false;
  double* hDiag_ = nullptr;      // pinned: the 15 diagonal entries of the initial covariance
  std::string err_;
  Params p_;
  int B_ = 0, Ncap_ = 0, ldp_ = 0, Fcap_ = 0, ldr_ = 0, ldt_ = 0, dev_ = 0;
  int Emax_ = 0, nmax_ = 0;            // EKF-SLAM feature states (hybrid mode); window columns 6 Ncap + Emax
  bool hybrid_ = false;
  double* dFidp_ = nullptr;            // inverse-depth records by feature slot
  struct HybridBufs;
  struct HybridDeleter { void operator()(HybridBufs* p) const; };
  std::unique_ptr<HybridBufs, HybridDeleter> hyb_;
  int flags_ = 0;
  std::vector<FilterHost> f_;
  cudaStream_t stream_ = nullptr, stream2_ = nullptr;
  cudaEvent_t ev_fork_ = nullptr, ev_join_ = nullptr, ev_ls_ = nullptr, ev_block_ = nullptr;
  double *dAmat_ = nullptr, *dPart_ = nullptr;
  size_t amat_cap_ = 0, part_cap_ = 0;
  double* dLs_ = nullptr;
  int *dTileRows_ = nullptr, *dFilterRows_ = nullptr;
  unsigned int* dSyrkCnt_ = nullptr;   // split-K arrival counters of k_syrk
  int n_sm_ = 148, syrk_waves_ = 1, syrk_group_ = 8;
  float last_syrk_us_ = 0.f, last_prior_us_ = 0.f;
  size_t tilerows_cap_ = 0;
  cudaEvent_t ev_[16];
  // device state
  double *dP_ = nullptr, *dImu_ = nullptr, *dClones_ = nullptr, *dFpos_ = nullptr;
  long long* dFgen_ = nullptr;
  double *dT_ = nullptr, *dS_ = nullptr, *dYv_ = nullptr, *dDx_ = nullptr;
  double* dChi2_ = nullptr;
  // growable device scratch
  double *dHblk_ = nullptr, *dRblk_ = nullptr;
  size_t hblk_cap_ = 0, rblk_cap_ = 0;
  int* dStatus_ = nullptr;
  double* dGamma_ = nullptr;
  size_t cand_cap_ = 0;
  Blob blob_;
  Blob blob_early_;                    // feat_off + observation pools of the end-to-end call, uploaded ahead
  int* dTriDone_ = nullptr;            // per-candidate completion flags of k_triangulate (epoch-stamped)
  size_t tridone_cap_ = 0;
  int tri_epoch_ = 0;
  bool graph_capturing_ = false;
  int* dStatusF_ = nullptr;            // triangulation status by feature slot (early direct-mode pass)
  size_t statusf_cap_ = 0;
  bool tri_done_early_ = false, jac_done_early_ = false;
  cudaStream_t stream_up_ = nullptr;   // side stream of the work-list upload when kernels are already queued
  cudaEvent_t ev_up_ = nullptr, ev_p_ = nullptr;
  bool upload_on_side_stream_ = false;
  Blob blob_early2_;                   // per-feature offsets / size-class lists of the early Jacobian pass
  double* dGammaF_ = nullptr;          // gamma by feature slot (early direct-mode pass)
  const int *dir_feat_off_ = nullptr, *dir_rowoff_ = nullptr, *dir_hblkoff_ = nullptr, *dir_sblk_ = nullptr,
            *dir_eblk_ = nullptr;      // device views of the per-feature arrays of the direct-mode passes
  size_t gammaf_cap_ = 0;
  std::shared_ptr<class HostWorker> worker_;   // helper thread of the end-to-end frame call (batch.cu)
  // pinned download buffers
  int* hStatus_ = nullptr;
  double* hGamma_ = nullptr;
  size_t hcand_cap_ = 0;
  double *hImu_ = nullptr, *hClones_ = nullptr, *hDx_ = nullptr;
  TriCfg tricfg_{};
  long long feature_updates_ = 0, launches_ = 0;
  double gpu_ms_ = 0;
  bool profiling_ = false;
  PhaseTimes pt_;
  std::vector<double> chi2_host_;
  std::vector<double> chi2_zupt_host_;     // chi_squared_table_zupt (p = 0.95, :482-493)
  int* dZuptDec_ = nullptr; double* dZuptInfo_ = nullptr;
  double* dCovHist_ = nullptr;         // replay with covariance capture: n_filters x n_frames x 225
  size_t covhist_cap_ = 0;
  int* hZuptDec_ = nullptr; double* hZuptInfo_ = nullptr;

  void prereserve();
  void wait_stream();
  void upload_blob();
  void ensure_scratch(size_t n_cand, size_t hblk, size_t rblk);
  void run_phase(PhaseWork& w, int phase);
  void stage_phase(PhaseWork& w);
  void stage_pack(PhaseWork& w);
  void stage_upload(PhaseWork& w);
  void launch_phase(PhaseWork& w, bool download, bool prior_in_flight = false);
  UpdArgs upd_args(const FilterWork* dFw) const;
  HybArgs hyb_args(const PhaseWork& w) const;
  // host mirror (position, inverse depth, obs_anchor) of the EKF-SLAM features of every filter: queued on the stream
  void hybrid_queue_gather(std::vector<Track*>& out_tracks);
  void hybrid_apply_gather(const std::vector<Track*>& tracks);
  struct SnapState;
  struct SnapDeleter { void operator()(SnapState* p) const; };
  std::unique_ptr<SnapState, SnapDeleter> snap_;
  int* dIters_ = nullptr; double* dCost_ = nullptr; size_t iters_cap_ = 0;
  double *dRawHx_ = nullptr, *dRawHe_ = nullptr, *dRawHf_ = nullptr, *dRawR_ = nullptr; size_t raw_cap_ = 0;
  bool want_iters_ = false, want_raw_ = false, skip_tri_ = false, skip_update_ = false, skip_jac_ = false;
  void download_mirrors();
  void init_filter_device(int i);
};

void rotation_to_quat_xyzw(const double* R, double* q);

int object_residuals(const double* frames_wTc, int T, const double* wTo, const double* shape, const double* kps,
                     int K, const double* zs, const double* zb, int flags, double* fvec, double* fjac_cam,
                     double* fjac_obj, int* zs_num, double* cam_pose_se3, int* rows_out);

}  // namespace ob

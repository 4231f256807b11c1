// Host orchestration of a batch of filters.  See batch.h.
//
// Mirrors, function by function, the host-visible control flow of the reference:
//   processFeatures        src/orcvio.cpp:500-661
//   batchImuProcessing     :664-724   (sample selection on the host, arithmetic in k_propagate)
//   addFeatureObservations :1016-1068
//   stateAugmentation      :930-1013  (bookkeeping here, covariance in k_augment)
//   removeLostFeatures     :2196-2579 (classification here; triangulation, Jacobians, gate,
//                                      compression and update on the GPU)
//   findRedundantImuStates :2582-2626
//   pruneImuStateBuffer    :2629-2959
#include "batch.h"
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <cstdio>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace ob {

#define CK(call)                                                                                  \
  do {                                                                                            \
    cudaError_t e__ = (call);                                                                     \
    if (e__ != cudaSuccess) {                                                                     \
      std::fprintf(stderr, "[orcvio_b200] CUDA error %s at %s:%d\n", cudaGetErrorString(e__),     \
                   __FILE__, __LINE__);                                                           \
      err_ = cudaGetErrorString(e__);                                                             \
      ok_ = false;                                                                                \
    }                                                                                             \
  } while (0)

struct Batch::PhaseWork {
  std::vector<Cand> cands;
  std::vector<int> obs_clone;
  std::vector<double> obs_z;
  std::vector<Tile> tiles;
  std::vector<FilterWork> fw;
  std::vector<int> small_list, large_list;
  size_t hblk_total = 0, rows_total = 0;
  int max_tile_rows = 0;
  size_t arows_total = 0;        // rows of the stacked A matrix
  int syrk_units = 1;            // grid of k_syrk: widest split-K plan over the filters
  int own_wmax_blk = 1;
  int wmax_blk = 1;
  int maxN = 0;
  // hybrid mode: the dense rows of the EKF-SLAM features (hybrid_kernel.cu)
  std::vector<HybWork> hw;
  std::vector<HybFeat> hfeats;
  std::vector<HybNew> hnews;
  int maxE = 0, max_dense = 0, hyb_phase = -1;   // hyb_phase: 0 lost-feature update, 1 prune update, -1 off
  size_t dense_total = 0;
  const HybWork* dHw = nullptr; const HybFeat* dHfeats = nullptr; const HybNew* dHnews = nullptr;
  std::vector<int> cand_begin;   // per filter, size B + 1
  bool any_active = false;
  std::vector<int> extra_ints;   // uploaded alongside (clone removal indices)
  const int* d_extra = nullptr;
  // device views of the uploaded work lists (valid after stage_phase)
  const Cand* dC = nullptr; const int* dOc = nullptr; const double* dOz = nullptr;
  const Tile* dTiles = nullptr; const FilterWork* dFw = nullptr;
  const int* dSmall = nullptr; const int* dLarge = nullptr;
  // observation pools referenced in place (snapshot entry points): copied straight into the pinned blob
  const int* ext_obs_clone = nullptr; const double* ext_obs_z = nullptr; size_t ext_nobs = 0;
  // observation pools already on the device (end-to-end call: uploaded ahead for the early triangulation)
  const int* pre_dOc = nullptr; const double* pre_dOz = nullptr;
  bool obs_preuploaded = false;
  bool cands_stay_on_host = false;   // direct mode: the kernels read per-feature arrays, the records are not uploaded
  size_t off[8] = {0};           // blob section offsets (stage_pack -> stage_upload)
  size_t n_obs() const { return ext_obs_clone ? ext_nobs : obs_clone.size(); }
  void reset() {                 // keep the vectors' capacity across frames
    cands.clear(); obs_clone.clear(); obs_z.clear(); tiles.clear(); fw.clear();
    small_list.clear(); large_list.clear(); cand_begin.clear(); extra_ints.clear();
    hblk_total = rows_total = 0;
    max_tile_rows = 0; arows_total = 0; own_wmax_blk = 1; wmax_blk = 1; maxN = 0;
    hw.clear(); hfeats.clear(); hnews.clear(); maxE = 0; max_dense = 0; hyb_phase = -1; dense_total = 0;
    dHw = nullptr; dHfeats = nullptr; dHnews = nullptr;
    any_active = false; d_extra = nullptr;
    dC = nullptr; dOc = nullptr; dOz = nullptr; dTiles = nullptr; dFw = nullptr; dSmall = dLarge = nullptr;
    ext_obs_clone = nullptr; ext_obs_z = nullptr; ext_nobs = 0;
    pre_dOc = nullptr; pre_dOz = nullptr; obs_preuploaded = false; cands_stay_on_host = false;
  }
};

// Device / pinned buffers of the hybrid MSCKF / EKF-SLAM mode (allocated only when max_features_in_one_grid > 0).
struct Batch::HybridBufs {
  double* dSpecPos = nullptr;          // scratch position table of the speculative initializeInvParamPosition pass
  long long* dSpecGen = nullptr;
  double* dFinal = nullptr; size_t final_cap = 0;          // 3 per speculative candidate (anchor-frame solution)
  int* dSpecStatus = nullptr; int* hSpecStatus = nullptr; size_t spec_cap = 0;
  double* dHd = nullptr; size_t hd_cap = 0;                // dense rows, ldh = ldr
  double *dH1 = nullptr, *dh2 = nullptr, *dr1 = nullptr, *dScratch = nullptr;
  int *dEkfPass = nullptr, *dNewOk = nullptr, *dNNew = nullptr;
  double* dEkfGamma = nullptr;
  int* hEkfPass = nullptr; double* hEkfGamma = nullptr;    // pinned
  double *dGather = nullptr, *hGather = nullptr; size_t gather_cap = 0;
  // upload arena: sections are only appended between two synchronisations of the stream (reset after a sync), so a
  // queued copy never sees its pinned source rewritten; fixed capacity, so device pointers stay valid
  char *pin = nullptr, *dev = nullptr; size_t cap = 0, used = 0;
  template <class T>
  const T* put(const T* src, size_t n, cudaStream_t s, bool* ok) {
    const size_t off = (used + 255) & ~size_t(255), bytes = sizeof(T) * std::max<size_t>(n, 1);
    if (off + bytes > cap) { *ok = false; return nullptr; }
    if (n) std::memcpy(pin + off, src, sizeof(T) * n);
    if (n && cudaMemcpyAsync(dev + off, pin + off, sizeof(T) * n, cudaMemcpyHostToDevice, s) != cudaSuccess) *ok = false;
    used = off + bytes;
    return reinterpret_cast<const T*>(dev + off);
  }
};

void Batch::HybridDeleter::operator()(HybridBufs* h) const {
  if (!h) return;
  cudaFree(h->dSpecPos); cudaFree(h->dSpecGen); cudaFree(h->dFinal); cudaFree(h->dSpecStatus);
  if (h->hSpecStatus) cudaFreeHost(h->hSpecStatus);
  cudaFree(h->dHd); cudaFree(h->dH1); cudaFree(h->dh2); cudaFree(h->dr1); cudaFree(h->dScratch);
  cudaFree(h->dEkfPass); cudaFree(h->dNewOk); cudaFree(h->dNNew); cudaFree(h->dEkfGamma);
  if (h->hEkfPass) cudaFreeHost(h->hEkfPass);
  if (h->hEkfGamma) cudaFreeHost(h->hEkfGamma);
  cudaFree(h->dGather);
  if (h->hGather) cudaFreeHost(h->hGather);
  cudaFree(h->dev);
  if (h->pin) cudaFreeHost(h->pin);
  delete h;
}

Batch::Batch(const Params& p, int n) : p_(p), B_(n) {
  ok_ = true;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    err_ = "no CUDA device: orcvio_b200 has no CPU fallback";
    std::fprintf(stderr, "[orcvio_b200] %s\n", err_.c_str());
    ok_ = false;
    return;
  }
  cudaGetDevice(&dev_);               // the device of the creating thread; worker threads re-select it on entry
  Ncap_ = p_.sw_size + 1;
  if (Ncap_ > ORCVIO_MAX_OBS) {
    err_ = "sw_size too large (max 31)";
    ok_ = false;
    return;
  }
  Emax_ = p_.max_features * p_.grid_rows * p_.grid_cols;     // 0: pure MSCKF
  hybrid_ = Emax_ > 0;
  nmax_ = 6 * Ncap_ + Emax_;
  ldp_ = ((ORCVIO_LEG + nmax_ + 7) / 8) * 8;
  ldr_ = ((nmax_ + 1 + 7) / 8) * 8;
  ldt_ = ldp_;
  Fcap_ = 4096;
  flags_ = (p_.use_larvio_flag ? FL_LARVIO : 0) | (p_.use_left_perturbation_flag ? FL_LEFT : 0) |
           (p_.discard_large_update_flag ? FL_DISCARD_LARGE : 0);
  tricfg_.translation_threshold = p_.feature_translation_threshold;
  tricfg_.huber_epsilon = 0.01;
  tricfg_.estimation_precision = 5e-7;
  tricfg_.initial_damping = 1e-3;
  tricfg_.outer_max = 10;
  tricfg_.inner_max = 10;
  tricfg_.cost_threshold = p_.feature_cost_threshold;
  tricfg_.init_final_dist_threshold = p_.init_final_dist_threshold;
  f_.resize(B_);
  for (auto& F : f_) {
    F.imu_mirror.assign(IM_STRIDE, 0.0);
    F.clone_mirror.assign((size_t)Ncap_ * CL_STRIDE, 0.0);
    F.free_slots.reserve(Fcap_);
    for (int s = Fcap_ - 1; s >= 0; --s) F.free_slots.push_back(s);
  }
  CK(cudaStreamCreate(&stream_));
  {
    // the prior factor is ONE big CTA (a whole SM's shared memory and registers) competing with the thousands
    // of small CTAs of the feature kernels: highest priority, so that the block scheduler places it first
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    CK(cudaStreamCreateWithPriority(&stream2_, cudaStreamDefault, hi));
    CK(cudaStreamCreateWithFlags(&stream_up_, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&ev_up_, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ev_p_, cudaEventDisableTiming));
  }
  CK(cudaEventCreateWithFlags(&ev_fork_, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&ev_join_, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&ev_ls_, cudaEventDisableTiming));
  if (env_int("ORCVIO_BLOCKING_SYNC", 0)) CK(cudaEventCreateWithFlags(&ev_block_, cudaEventDisableTiming | cudaEventBlockingSync));
  for (auto& e : ev_) CK(cudaEventCreate(&e));
  const size_t nB = (size_t)B_;
  CK(cudaMalloc(&dP_, nB * ldp_ * ldp_ * sizeof(double)));
  CK(cudaMemset(dP_, 0, nB * ldp_ * ldp_ * sizeof(double)));
  CK(cudaMalloc(&dImu_, nB * IM_STRIDE * sizeof(double)));
  CK(cudaMemset(dImu_, 0, nB * IM_STRIDE * sizeof(double)));
  CK(cudaMalloc(&dClones_, nB * Ncap_ * CL_STRIDE * sizeof(double)));
  CK(cudaMemset(dClones_, 0, nB * Ncap_ * CL_STRIDE * sizeof(double)));
  CK(cudaMalloc(&dFpos_, nB * Fcap_ * FP_STRIDE * sizeof(double)));
  CK(cudaMemset(dFpos_, 0, nB * Fcap_ * FP_STRIDE * sizeof(double)));
  CK(cudaMalloc(&dFgen_, nB * Fcap_ * sizeof(long long)));
  CK(cudaMemset(dFgen_, 0xFF, nB * Fcap_ * sizeof(long long)));
  const int ncap = nmax_;
  if (hybrid_) {
    CK(cudaMalloc(&dFidp_, nB * Fcap_ * FI_STRIDE * sizeof(double)));
    CK(cudaMemset(dFidp_, 0, nB * Fcap_ * FI_STRIDE * sizeof(double)));
    hyb_.reset(new HybridBufs());
    HybridBufs& h = *hyb_;
    CK(cudaMalloc(&h.dSpecPos, nB * Fcap_ * FP_STRIDE * sizeof(double)));
    CK(cudaMemset(h.dSpecPos, 0, nB * Fcap_ * FP_STRIDE * sizeof(double)));
    CK(cudaMalloc(&h.dSpecGen, nB * Fcap_ * sizeof(long long)));
    CK(cudaMemset(h.dSpecGen, 0xFF, nB * Fcap_ * sizeof(long long)));
    const size_t ne = nB * Emax_;
    CK(cudaMalloc(&h.dH1, ne * ldr_ * sizeof(double)));
    CK(cudaMalloc(&h.dh2, ne * sizeof(double)));
    CK(cudaMalloc(&h.dr1, ne * sizeof(double)));
    CK(cudaMalloc(&h.dScratch, nB * 64 * ldr_ * sizeof(double)));
    CK(cudaMalloc(&h.dEkfPass, ne * sizeof(int)));
    CK(cudaMalloc(&h.dEkfGamma, ne * sizeof(double)));
    CK(cudaMalloc(&h.dNewOk, ne * sizeof(int)));
    CK(cudaMalloc(&h.dNNew, nB * sizeof(int)));
    CK(cudaMemset(h.dNNew, 0, nB * sizeof(int)));
    CK(cudaMallocHost(&h.hEkfPass, ne * sizeof(int)));
    CK(cudaMallocHost(&h.hEkfGamma, ne * sizeof(double)));
    h.gather_cap = 2 * ne + 64;
    CK(cudaMalloc(&h.dGather, h.gather_cap * 6 * sizeof(double)));
    CK(cudaMallocHost(&h.hGather, h.gather_cap * 6 * sizeof(double)));
    h.cap = (size_t)(2 << 20) + nB * (size_t)(64 << 10);
    CK(cudaMalloc(&h.dev, h.cap));
    CK(cudaMallocHost(&h.pin, h.cap));
  }
  CK(cudaMalloc(&dS_, nB * (size_t)(ncap + 1) * ldr_ * sizeof(double)));
  CK(cudaMalloc(&dYv_, nB * ldr_ * sizeof(double)));
  CK(cudaMalloc(&dT_, nB * (size_t)ncap * ldt_ * sizeof(double)));
  CK(cudaMalloc(&dDx_, nB * ldp_ * sizeof(double)));
  CK(cudaMemset(dDx_, 0, nB * ldp_ * sizeof(double)));
  CK(cudaMalloc(&dLs_, nB * ORCVIO_LEG * ORCVIO_LEG * sizeof(double)));
  CK(cudaMalloc(&dFilterRows_, nB * sizeof(int)));
  CK(cudaMemset(dFilterRows_, 0, nB * sizeof(int)));
  CK(cudaMalloc(&dSyrkCnt_, nB * SY_MAXP * (SY_MAXG + 1) * sizeof(unsigned int)));
  CK(cudaMemset(dSyrkCnt_, 0, nB * SY_MAXP * (SY_MAXG + 1) * sizeof(unsigned int)));
  {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&n_sm_, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n_sm_ < 1) n_sm_ = 148;
    if (const char* e = std::getenv("ORCVIO_SYRK_WAVES")) syrk_waves_ = std::max(1, std::atoi(e));
    syrk_group_ = std::max(1, env_int("ORCVIO_SYRK_GROUP", 8));
  }
  chi2_host_.assign(500, 0.0);
  for (int i = 1; i < 500; ++i) chi2_host_[i] = chi2_quantile(p_.chi_square_threshold_feat, i);
  CK(cudaMalloc(&dChi2_, 500 * sizeof(double)));
  CK(cudaMemcpy(dChi2_, chi2_host_.data(), 500 * sizeof(double), cudaMemcpyHostToDevice));
  if (p_.if_ZUPT_valid) {
    chi2_zupt_host_.assign(500, 0.0);
    if (!p_.if_use_feature_zupt_flag)
      for (int i = 1; i < 500; ++i) chi2_zupt_host_[i] = chi2_quantile(0.95, i);
    CK(cudaMalloc(&dZuptDec_, nB * sizeof(int)));
    CK(cudaMalloc(&dZuptInfo_, nB * 2 * sizeof(double)));
    CK(cudaMallocHost(&hZuptDec_, nB * sizeof(int)));
    CK(cudaMallocHost(&hZuptInfo_, nB * 2 * sizeof(double)));
    std::memset(hZuptDec_, 0, nB * sizeof(int));
  }
  CK(cudaMallocHost(&hImu_, nB * IM_STRIDE * sizeof(double)));
  CK(cudaMallocHost(&hClones_, nB * Ncap_ * CL_STRIDE * sizeof(double)));
  CK(cudaMallocHost(&hDx_, nB * ldp_ * sizeof(double)));
  std::memset(hImu_, 0, nB * IM_STRIDE * sizeof(double));
  if (B_ > 1 || env_int("ORCVIO_PRERESERVE", 0)) prereserve();
}

// Multi-trajectory batches: size the growable buffers for a typical frame up front.  Growing them later works (x 2
// policy) but every growth is a cudaFree / cudaMallocHost, i.e. a device-wide synchronisation -- with several batches
// replaying from as many host threads those stalls hit every thread at once.
// End of a phase of process(): the host needs the downloaded results.  A single filter spins (lowest latency); the
// batches of a multi-trajectory replay block on an event instead, so that a thread waiting for its kernels leaves its
// core to the bookkeeping of another batch.
void Batch::wait_stream() {
  if (B_ > 1 && ev_block_) {
    CK(cudaEventRecord(ev_block_, stream_));
    CK(cudaEventSynchronize(ev_block_));
  } else {
    CK(cudaStreamSynchronize(stream_));
  }
}

void Batch::prereserve() {
  const size_t nB = (size_t)B_;
  const size_t cands = nB * 192, rows = cands * 9, obs = cands * 6;
  ensure_scratch(cands, rows * 36, rows);
  const size_t tiles = nB * 48;
  if (tiles > tilerows_cap_) {
    tilerows_cap_ = tiles;
    CK(cudaMalloc(&dTileRows_, tilerows_cap_ * sizeof(int)));
  }
  const size_t need_a = (rows + 64 * nB + 16) * (size_t)ldr_;
  if (need_a > amat_cap_) {
    amat_cap_ = need_a;
    CK(cudaMalloc(&dAmat_, amat_cap_ * sizeof(double)));
  }
  // split-K partial tiles: up to ~18 work units per filter were seen on EuRoC-shaped frames (6 tile pairs x chunks of
  // >= 128 rows); 32 covers ~2500 stacked rows per filter without a growth in the middle of a replay
  const size_t need_p = nB * 32 * 4096;
  if (need_p > part_cap_) {
    part_cap_ = need_p;
    CK(cudaMalloc(&dPart_, part_cap_ * sizeof(double)));
  }
  const size_t blob_bytes = cands * sizeof(Cand) + obs * (sizeof(int) + 2 * sizeof(double)) + tiles * sizeof(Tile) +
                            nB * (sizeof(FilterWork) + 64) + cands * 2 * sizeof(int) + (size_t)(64 << 10);
  blob_.ensure_pinned(blob_bytes);
  if (blob_bytes > blob_.dev_cap) {
    blob_.dev_cap = blob_bytes;
    CK(cudaMalloc(&blob_.dev, blob_.dev_cap));
  }
  if (hybrid_) {
    HybridBufs& hb = *hyb_;
    hb.hd_cap = nB * (size_t)(2 * Emax_ + 16 * 9) * ldr_;
    CK(cudaMalloc(&hb.dHd, hb.hd_cap * sizeof(double)));
    hb.spec_cap = nB * 64;
    CK(cudaMalloc(&hb.dFinal, hb.spec_cap * 3 * sizeof(double)));
    CK(cudaMalloc(&hb.dSpecStatus, hb.spec_cap * sizeof(int)));
    CK(cudaMallocHost(&hb.hSpecStatus, hb.spec_cap * sizeof(int)));
  }
}

Batch::~Batch() {
  cudaDeviceSynchronize();
  cudaFree(dP_); cudaFree(dImu_); cudaFree(dClones_); cudaFree(dFpos_); cudaFree(dFgen_);
  cudaFree(dS_); cudaFree(dYv_); cudaFree(dT_); cudaFree(dDx_); cudaFree(dChi2_);
  cudaFree(dAmat_); cudaFree(dPart_);
  cudaFree(dStatusF_); cudaFree(dGammaF_); cudaFree(dFidp_); cudaFree(dTriDone_);
  if (blob_early2_.dev) cudaFree(blob_early2_.dev);
  if (blob_early2_.pinned) cudaFreeHost(blob_early2_.pinned);
  if (blob_early_.dev) cudaFree(blob_early_.dev);
  if (blob_early_.pinned) cudaFreeHost(blob_early_.pinned);
  cudaFree(dLs_); cudaFree(dTileRows_); cudaFree(dFilterRows_); cudaFree(dSyrkCnt_);
  if (dZuptDec_) cudaFree(dZuptDec_);
  if (dCovHist_) cudaFree(dCovHist_);
  if (dZuptInfo_) cudaFree(dZuptInfo_);
  if (hZuptDec_) cudaFreeHost(hZuptDec_);
  if (hZuptInfo_) cudaFreeHost(hZuptInfo_);
  cudaFree(dHblk_); cudaFree(dRblk_); cudaFree(dStatus_); cudaFree(dGamma_);
  if (blob_.dev) cudaFree(blob_.dev);
  if (blob_.pinned) cudaFreeHost(blob_.pinned);
  cudaFreeHost(hImu_); cudaFreeHost(hClones_); cudaFreeHost(hDx_);
  if (hDiag_) cudaFreeHost(hDiag_);
  if (hStatus_) cudaFreeHost(hStatus_);
  if (hGamma_) cudaFreeHost(hGamma_);
  for (auto& e : ev_) cudaEventDestroy(e);
  if (ev_fork_) cudaEventDestroy(ev_fork_);
  if (ev_join_) cudaEventDestroy(ev_join_);
  if (ev_ls_) cudaEventDestroy(ev_ls_);
  if (ev_block_) cudaEventDestroy(ev_block_);
  if (stream2_) cudaStreamDestroy(stream2_);
  if (stream_up_) cudaStreamDestroy(stream_up_);
  if (ev_up_) cudaEventDestroy(ev_up_);
  if (ev_p_) cudaEventDestroy(ev_p_);
  if (stream_) cudaStreamDestroy(stream_);
}

void Batch::set_initial_state(int i, double t, const double* q, const double* p, const double* v,
                              const double* bg, const double* ba) {
  FilterHost& F = f_[i];
  F.has_init = true;
  F.init_t = t;
  for (int k = 0; k < 4; ++k) F.init_q[k] = q[k];
  for (int k = 0; k < 3; ++k) {
    F.init_p[k] = p[k];
    F.init_v[k] = v[k];
    F.init_bg[k] = bg ? bg[k] : 0.0;
    F.init_ba[k] = ba ? ba[k] : 0.0;
  }
}

// Write the initial IMU record and covariance of filter i (reference :514-523, :201-225).
void Batch::init_filter_device(int i) {
  FilterHost& F = f_[i];
  double* im = hImu_ + (size_t)i * IM_STRIDE;
  std::memset(im, 0, IM_STRIDE * sizeof(double));
  quat_xyzw_to_R(F.init_q, im + IM_R);
  for (int k = 0; k < 3; ++k) {
    im[IM_V + k] = F.init_v[k];
    im[IM_P + k] = F.init_p[k];
    im[IM_BG + k] = F.init_bg[k];
    im[IM_BA + k] = F.init_ba[k];
    im[IM_TCB + k] = p_.t_cam0_imu[k];
  }
  for (int k = 0; k < 9; ++k) im[IM_RBC + k] = p_.R_imu_cam0[k];
  im[IM_TD] = p_.td;
  im[IM_TIME] = F.init_t;
  // Initial covariance: 15 diagonal entries, the rest zero.  Stream-ordered (a memset + one strided copy of the pinned
  // diagonal) -- a synchronous cudaMemcpy here runs on the legacy default stream, i.e. it waits for and blocks the
  // streams of EVERY batch of the process: with 16-32 replay threads initialising 64 filters each that was thousands of
  // device-wide serialisation points and first frames of up to 1.5 s (ORCVIO_HOST_PROF=3).
  if (!hDiag_) {
    CK(cudaMallocHost(&hDiag_, 16 * sizeof(double)));
    const double v[5] = {p_.cov_orientation, p_.cov_velocity, p_.cov_position, p_.cov_gyro_bias, p_.cov_acc_bias};
    for (int k = 0; k < 15; ++k) hDiag_[k] = v[k / 3];
    hDiag_[15] = 0.0;
  }
  double* dPi = dP_ + (size_t)i * ldp_ * ldp_;
  CK(cudaMemsetAsync(dPi, 0, (size_t)ldp_ * ldp_ * sizeof(double), stream_));
  CK(cudaMemcpy2DAsync(dPi, (size_t)(ldp_ + 1) * sizeof(double), hDiag_, sizeof(double), sizeof(double), 15,
                       cudaMemcpyHostToDevice, stream_));
}

// ORCVIO_HOST_PROF=3: every growth of a device / pinned buffer after construction (a device-wide synchronisation that
// stalls all the batches of the process) is reported
static void note_growth(const char* what, size_t bytes) {
  static const bool on = env_int("ORCVIO_HOST_PROF", 0) == 3;
  if (on) std::fprintf(stderr, "[replay prof] growth: %s -> %.1f MB\n", what, bytes / 1048576.0);
}

void Batch::ensure_scratch(size_t n_cand, size_t hblk, size_t rblk) {
  auto grow = [&](double*& ptr, size_t& cap, size_t need) {
    if (need <= cap) return;
    if (ptr) cudaFree(ptr);
    cap = need * 2 + 1024;
    note_growth("hblk / rblk", cap * sizeof(double));
    CK(cudaMalloc(&ptr, cap * sizeof(double)));
  };
  grow(dHblk_, hblk_cap_, hblk);
  grow(dRblk_, rblk_cap_, rblk);
  if (n_cand > cand_cap_) {
    if (dStatus_) cudaFree(dStatus_);
    if (dGamma_) cudaFree(dGamma_);
    cand_cap_ = n_cand * 2 + 1024;
    note_growth("candidate status", cand_cap_ * 12);
    CK(cudaMalloc(&dStatus_, cand_cap_ * sizeof(int)));
    CK(cudaMalloc(&dGamma_, cand_cap_ * sizeof(double)));
  }
  if (n_cand > hcand_cap_) {
    if (hStatus_) cudaFreeHost(hStatus_);
    if (hGamma_) cudaFreeHost(hGamma_);
    hcand_cap_ = n_cand * 2 + 1024;
    note_growth("candidate status (pinned)", hcand_cap_ * 12);
    CK(cudaMallocHost(&hStatus_, hcand_cap_ * sizeof(int)));
    CK(cudaMallocHost(&hGamma_, hcand_cap_ * sizeof(double)));
  }
}

void Batch::upload_blob() {
  if (blob_.used == 0) return;
  if (blob_.used > blob_.dev_cap) {
    if (blob_.dev) cudaFree(blob_.dev);
    blob_.dev_cap = blob_.used * 2 + 4096;
    note_growth("work-list blob", blob_.dev_cap);
    CK(cudaMalloc(&blob_.dev, blob_.dev_cap));
  }
  if (upload_on_side_stream_) {
    // kernels of this frame are already queued on stream_ (early triangulation / Jacobian pass): a copy on the
    // same stream would wait for them, so the blob goes up on its own stream and stream_ joins it afterwards
    CK(cudaMemcpyAsync(blob_.dev, blob_.pinned, blob_.used, cudaMemcpyHostToDevice, stream_up_));
    CK(cudaEventRecord(ev_up_, stream_up_));
    CK(cudaStreamWaitEvent(stream_, ev_up_, 0));
  } else {
    CK(cudaMemcpyAsync(blob_.dev, blob_.pinned, blob_.used, cudaMemcpyHostToDevice, stream_));
  }
}

void Batch::download_mirrors() {
  CK(cudaMemcpyAsync(hImu_, dImu_, (size_t)B_ * IM_STRIDE * sizeof(double), cudaMemcpyDeviceToHost, stream_));
  CK(cudaMemcpyAsync(hClones_, dClones_, (size_t)B_ * Ncap_ * CL_STRIDE * sizeof(double),
                     cudaMemcpyDeviceToHost, stream_));
}

// ---------------------------------------------------------------------------------------
// Build tiles for the candidates [c0, c1) of one filter (already sorted by s_blk).
static void build_tiles(Batch::PhaseWork& w, int fi, int c0, int c1);

struct CandBuild {
  Cand c;
  long long id;
  int kind;
};

void Batch::run_phase(PhaseWork& w, int phase) {
  stage_phase(w);
  launch_phase(w, true);
  (void)phase;
}

// Pack the work lists of one phase into the pinned blob and upload them (one H2D copy).
// Host half of the staging: carve the pinned blob and copy the work lists into it (no CUDA call as long as the
// pinned capacity suffices -- the end-to-end call reserves it up front and runs this on its helper thread).
void Batch::stage_pack(PhaseWork& w) {
  const int nC = (int)w.cands.size();
  blob_.reset();
  const bool up_c = !w.cands_stay_on_host;
  const size_t o_c = blob_.reserve(sizeof(Cand) * (up_c ? std::max(nC, 1) : 1));
  const size_t n_obs = w.obs_preuploaded ? 0 : w.n_obs();
  const size_t o_oc = blob_.reserve(sizeof(int) * std::max<size_t>(n_obs, 1));
  const size_t o_oz = blob_.reserve(sizeof(double) * std::max<size_t>(2 * n_obs, 1));
  const size_t o_t = blob_.reserve(sizeof(Tile) * std::max<size_t>(w.tiles.size(), 1));
  const size_t o_f = blob_.reserve(sizeof(FilterWork) * B_);
  const size_t o_s = blob_.reserve(sizeof(int) * std::max<size_t>(w.small_list.size(), 1));
  const size_t o_l = blob_.reserve(sizeof(int) * std::max<size_t>(w.large_list.size(), 1));
  const size_t o_x = blob_.reserve(sizeof(int) * std::max<size_t>(w.extra_ints.size(), 1));
  char* h = blob_.pinned;
  if (!w.extra_ints.empty()) std::memcpy(h + o_x, w.extra_ints.data(), sizeof(int) * w.extra_ints.size());
  if (nC && up_c) std::memcpy(h + o_c, w.cands.data(), sizeof(Cand) * nC);
  if (n_obs) {
    std::memcpy(h + o_oc, w.ext_obs_clone ? w.ext_obs_clone : w.obs_clone.data(), sizeof(int) * n_obs);
    std::memcpy(h + o_oz, w.ext_obs_z ? w.ext_obs_z : w.obs_z.data(), sizeof(double) * 2 * n_obs);
  }
  if (!w.tiles.empty()) std::memcpy(h + o_t, w.tiles.data(), sizeof(Tile) * w.tiles.size());
  std::memcpy(h + o_f, w.fw.data(), sizeof(FilterWork) * B_);
  if (!w.small_list.empty()) std::memcpy(h + o_s, w.small_list.data(), sizeof(int) * w.small_list.size());
  if (!w.large_list.empty()) std::memcpy(h + o_l, w.large_list.data(), sizeof(int) * w.large_list.size());
  w.off[0] = o_c; w.off[1] = o_oc; w.off[2] = o_oz; w.off[3] = o_t; w.off[4] = o_f; w.off[5] = o_s; w.off[6] = o_l;
  w.off[7] = o_x;
}

// Device half: grow the scratch buffers, upload the blob, publish the device views of the lists.
void Batch::stage_upload(PhaseWork& w) {
  const int nC = (int)w.cands.size();
  const size_t o_c = w.off[0], o_oc = w.off[1], o_oz = w.off[2], o_t = w.off[3], o_f = w.off[4], o_s = w.off[5],
               o_l = w.off[6], o_x = w.off[7];
  ensure_scratch(std::max(nC, 1), std::max<size_t>(w.hblk_total, 1), std::max<size_t>(w.rows_total, 1));
  // scratch of the update, grown outside any timed region
  if (w.tiles.size() > tilerows_cap_) {
    if (dTileRows_) cudaFree(dTileRows_);
    tilerows_cap_ = w.tiles.size() * 2 + 64;
    note_growth("tile rows", tilerows_cap_ * sizeof(int));
    CK(cudaMalloc(&dTileRows_, tilerows_cap_ * sizeof(int)));
  }
  int units = 1;
  for (const FilterWork& f : w.fw) units = std::max(units, syrk_plan(f, n_sm_ * syrk_waves_).total);
  w.syrk_units = units;
  const size_t need_a = (w.arows_total + 16) * (size_t)ldr_;
  if (need_a > amat_cap_) {
    if (dAmat_) cudaFree(dAmat_);
    amat_cap_ = need_a * 2;
    note_growth("A", amat_cap_ * sizeof(double));
    CK(cudaMalloc(&dAmat_, amat_cap_ * sizeof(double)));
  }
  const size_t need_p = (size_t)B_ * units * 4096;
  if (need_p > part_cap_) {
    if (dPart_) cudaFree(dPart_);
    part_cap_ = need_p * 2;
    note_growth("split-K partials", part_cap_ * sizeof(double));
    CK(cudaMalloc(&dPart_, part_cap_ * sizeof(double)));
  }
  if (hybrid_ && w.hyb_phase >= 0) {
    HybridBufs& hb = *hyb_;
    const size_t need_h = (w.dense_total + 8) * (size_t)ldr_;
    if (need_h > hb.hd_cap) {
      if (hb.dHd) cudaFree(hb.dHd);
      hb.hd_cap = need_h * 2;
      note_growth("hybrid dense rows", hb.hd_cap * sizeof(double));
      CK(cudaMalloc(&hb.dHd, hb.hd_cap * sizeof(double)));
    }
    bool okp = true;
    w.dHw = hb.put(w.hw.data(), w.hw.size(), stream_, &okp);
    w.dHfeats = hb.put(w.hfeats.data(), w.hfeats.size(), stream_, &okp);
    w.dHnews = hb.put(w.hnews.data(), w.hnews.size(), stream_, &okp);
    if (!okp) { ok_ = false; err_ = "hybrid upload arena exhausted"; }
  }
  upload_blob();
  char* d = blob_.dev;
  w.dC = (const Cand*)(d + o_c);
  w.dOc = w.obs_preuploaded ? w.pre_dOc : (const int*)(d + o_oc);
  w.dOz = w.obs_preuploaded ? w.pre_dOz : (const double*)(d + o_oz);
  w.dTiles = (const Tile*)(d + o_t);
  w.dFw = (const FilterWork*)(d + o_f);
  w.dSmall = (const int*)(d + o_s);
  w.dLarge = (const int*)(d + o_l);
  w.d_extra = (const int*)(d + o_x);
}

void Batch::stage_phase(PhaseWork& w) {
  stage_pack(w);
  stage_upload(w);
}

UpdArgs Batch::upd_args(const FilterWork* dFw) const {
  UpdArgs ua{};
  ua.fw = dFw; ua.n_filters = B_;
  ua.P = dP_; ua.p_stride = (size_t)ldp_ * ldp_; ua.ldp = ldp_;
  ua.r_stride = (size_t)(nmax_ + 1) * ldr_; ua.ldr = ldr_;
  ua.T = dT_; ua.S = dS_; ua.t_stride = (size_t)nmax_ * ldt_; ua.ldt = ldt_;
  ua.yv = dYv_;
  ua.imu = dImu_; ua.clones = dClones_; ua.clone_stride = (size_t)Ncap_ * CL_STRIDE;
  ua.dx = dDx_; ua.lddx = ldp_;
  ua.flags = flags_; ua.sigma2 = p_.feature_observation_noise;
  return ua;
}

HybArgs Batch::hyb_args(const PhaseWork& w) const {
  const HybridBufs& hb = *hyb_;
  HybArgs ha{};
  ha.hw = w.dHw; ha.n_filters = B_; ha.feats = w.dHfeats; ha.news = w.dHnews;
  ha.clones = dClones_; ha.clone_stride = (size_t)Ncap_ * CL_STRIDE; ha.imu = dImu_;
  ha.fpos = dFpos_; ha.fidp = dFidp_; ha.fcap = Fcap_;
  ha.P = dP_; ha.p_stride = (size_t)ldp_ * ldp_; ha.ldp = ldp_;
  ha.obs_clone = w.dOc; ha.obs_z = w.dOz;
  ha.status = dStatus_;
  ha.sigma2 = p_.feature_observation_noise; ha.chi2_dof2 = chi2_host_[2];
  ha.Hd = hb.dHd; ha.ldh = ldr_;
  ha.H1 = hb.dH1; ha.h2 = hb.dh2; ha.r1 = hb.dr1; ha.new_cap = Emax_;
  ha.scratch = hb.dScratch;
  ha.ekf_pass = hb.dEkfPass; ha.ekf_gamma = hb.dEkfGamma; ha.new_ok = hb.dNewOk; ha.n_new = hb.dNNew;
  ha.dx = dDx_; ha.lddx = ldp_;
  return ha;
}

// Kernel chain of one phase on already staged work lists: triangulate -> Jacobian/nullspace/gate
// -> whitened-form compression + EKF update; optionally queues the D2H copy of the per-candidate results.
void Batch::launch_phase(PhaseWork& w, bool download, bool prior_in_flight) {
  const int nC = (int)w.cands.size();
  const Cand* dC = w.dC; const int* dOc = w.dOc; const double* dOz = w.dOz;
  const Tile* dTiles = w.dTiles; const FilterWork* dFw = w.dFw;
  const int* dSmall = w.dSmall; const int* dLarge = w.dLarge;
  int nl = 0;
  cudaEvent_t* e = ev_;
  if (profiling_) CK(cudaEventRecord(e[0], stream_));
  const bool do_update = w.any_active && !skip_update_;
  if (do_update && !prior_in_flight) {
    // the prior factor depends on P alone: start it BEFORE the feature kernels are queued, otherwise its one
    // big CTA waits for an empty SM behind the first waves of k_triangulate
    CK(cudaEventRecord(ev_fork_, stream_));
    InfoBufs ib{};
    ib.Ls = dLs_; ib.ls_done = ev_ls_;
    launch_info_prior(upd_args(dFw), ib, w.maxN, stream2_, ev_fork_, ev_join_, profiling_ ? e[9] : nullptr,
                      profiling_ ? e[10] : nullptr, w.maxE);
    nl += 2;                               // k_chol_prior + k_imu_factor
    prior_in_flight = true;
  }
  const bool hyb_on = hybrid_ && w.hyb_phase >= 0 && do_update;
  HybArgs ha{};
  if (hyb_on) ha = hyb_args(w);
  if (want_iters_ && (size_t)nC > iters_cap_) {
    if (dIters_) cudaFree(dIters_);
    if (dCost_) cudaFree(dCost_);
    iters_cap_ = (size_t)nC * 2 + 64;
    CK(cudaMalloc(&dIters_, iters_cap_ * 2 * sizeof(int)));
    CK(cudaMalloc(&dCost_, iters_cap_ * sizeof(double)));
  }
  if (want_raw_ && w.n_obs() > raw_cap_) {
    for (double** p : {&dRawHx_, &dRawHe_, &dRawHf_, &dRawR_})
      if (*p) cudaFree(*p);
    raw_cap_ = w.n_obs() * 2 + 64;
    CK(cudaMalloc(&dRawHx_, raw_cap_ * 12 * sizeof(double)));
    CK(cudaMalloc(&dRawHe_, raw_cap_ * 12 * sizeof(double)));
    CK(cudaMalloc(&dRawHf_, raw_cap_ * 6 * sizeof(double)));
    CK(cudaMalloc(&dRawR_, raw_cap_ * 2 * sizeof(double)));
  }
  // k_jac_gate follows k_triangulate candidate by candidate (completion flags + programmatic launch) instead of
  // waiting for the slowest LM chain of the whole grid; ORCVIO_TRI_OVERLAP=0 restores the grid-wide dependency
  static const int overlap_env = env_int("ORCVIO_TRI_OVERLAP", 1);
  const bool tri_here = nC > 0 && !skip_tri_ && !tri_done_early_;
  // (measured: the slowest LM chain + its own Jacobian pass bound the overlapped pair at ~93 us whatever the count, so it
  // only pays when the Jacobian kernel alone needs more than one wave: 4096 features 107 -> 96 us, 2000 features 82 -> 93 us)
  static const int overlap_min = env_int("ORCVIO_TRI_OVERLAP_MIN", 2400);
  const bool overlap = overlap_env && tri_here && !skip_jac_ && !jac_done_early_ && !want_iters_ && !want_raw_ &&
                       nC >= overlap_min;
  if (overlap) {
    if ((size_t)nC > tridone_cap_) {
      if (dTriDone_) cudaFree(dTriDone_);
      tridone_cap_ = (size_t)nC * 2 + 1024;
      CK(cudaMalloc(&dTriDone_, tridone_cap_ * sizeof(int)));
      CK(cudaMemsetAsync(dTriDone_, 0, tridone_cap_ * sizeof(int), stream_));
    }
    ++tri_epoch_;
    // (inside a graph the epoch is a baked-in constant: the flags are cleared by a node of the graph instead)
    if (graph_capturing_) CK(cudaMemsetAsync(dTriDone_, 0, (size_t)nC * sizeof(int), stream_));
  }
  if (tri_here) {
    TriArgs ta{};
    ta.done = overlap ? dTriDone_ : nullptr; ta.epoch = tri_epoch_;
    ta.cand = dC; ta.n_cand = nC;
    ta.clones = dClones_; ta.clone_stride = (size_t)Ncap_ * CL_STRIDE;
    ta.fpos = dFpos_; ta.fgen = dFgen_; ta.fcap = Fcap_;
    ta.obs_clone = dOc; ta.obs_z = dOz;
    ta.cfg = tricfg_;
    ta.status = dStatus_;
    ta.iters = want_iters_ ? dIters_ : nullptr;
    ta.cost = want_iters_ ? dCost_ : nullptr;
    launch_triangulate(ta, stream_);
    ++nl;
  }
  if (profiling_ && !overlap) CK(cudaEventRecord(e[1], stream_));   // (an event between the two would serialise them)
  if (nC > 0 && !skip_jac_ && !jac_done_early_) {
    JacArgs ja{};
    ja.tri_done = overlap ? dTriDone_ : nullptr; ja.tri_epoch = tri_epoch_;
    ja.cand = dC;
    ja.clones = dClones_; ja.clone_stride = (size_t)Ncap_ * CL_STRIDE;
    ja.imu = dImu_; ja.fpos = dFpos_; ja.fcap = Fcap_;
    ja.P = dP_; ja.p_stride = (size_t)ldp_ * ldp_; ja.ldp = ldp_;
    ja.obs_clone = dOc; ja.obs_z = dOz;
    ja.flags = flags_; ja.sigma2 = p_.feature_observation_noise; ja.chi2 = dChi2_;
    ja.status = dStatus_; ja.gamma = dGamma_;
    ja.hblk = dHblk_; ja.rblk = dRblk_;
    if (want_raw_) { ja.raw_Hx = dRawHx_; ja.raw_He = dRawHe_; ja.raw_Hf = dRawHf_; ja.raw_r = dRawR_; }
    ja.tri_status_f = tri_done_early_ ? dStatusF_ : nullptr;
    JacArgs js = ja, jl = ja;
    js.cand_list = dSmall; js.n_list = (int)w.small_list.size();
    jl.cand_list = dLarge; jl.n_list = (int)w.large_list.size();
    launch_jac_gate(js, jl, stream_);
    nl += (js.n_list > 0) + (jl.n_list > 0);
  }
  if (profiling_ && overlap) CK(cudaEventRecord(e[1], stream_));    // stage "tri" = both kernels, stage "jac" = 0
  if (hyb_on && w.hyb_phase == 0) {     // dense rows of the features of the state / of the new features (gated)
    launch_hybrid_rows(ha, stream_);
    ++nl;
  }
  if (profiling_) CK(cudaEventRecord(e[2], stream_));
  if (do_update) {
    AformArgs qa{};
    qa.cand = dC; qa.status = dStatus_;
    qa.status_f = jac_done_early_ ? dStatusF_ : nullptr;
    if (jac_done_early_ && w.cands_stay_on_host) {
      qa.order_f = w.d_extra;
      qa.feat_off = dir_feat_off_; qa.rowoff_f = dir_rowoff_; qa.hblkoff_f = dir_hblkoff_;
      qa.sblk_f = dir_sblk_; qa.eblk_f = dir_eblk_;
    }
    qa.hblk = dHblk_; qa.rblk = dRblk_;
    qa.tiles = dTiles;
    qa.fw = dFw;
    InfoBufs ib{};
    ib.Ls = dLs_; ib.Amat = dAmat_; ib.part = dPart_; ib.ls_done = ev_ls_;
    ib.max_units = w.syrk_units; ib.cta_budget = n_sm_ * syrk_waves_; ib.group = syrk_group_; ib.syrk_cnt = dSyrkCnt_;
    ib.tile_rows = dTileRows_; ib.filter_rows = dFilterRows_;
    launch_info_update(qa, upd_args(dFw), ib, (int)w.tiles.size(), w.max_tile_rows, w.wmax_blk, w.maxN, stream_,
                       stream2_, ev_fork_, ev_join_, profiling_ ? e[3] : nullptr, profiling_ ? e[4] : nullptr, &nl,
                       prior_in_flight, profiling_ ? e[8] : nullptr, profiling_ ? e[9] : nullptr,
                       profiling_ ? e[10] : nullptr, w.maxE, hyb_on ? &ha : nullptr, w.max_dense);
    if (hyb_on) {
      // feature increments (+ delayed initialisation of this frame's new features), src/orcvio.cpp:1843-1941
      if (w.hyb_phase == 0) { launch_hybrid_post(ha, stream_); ++nl; }
      else if (w.maxE > 0) { launch_hybrid_feature_increment(ha, stream_); ++nl; }
    }
    if (profiling_) CK(cudaEventRecord(e[5], stream_));
  }
  launches_ += nl;
  tri_done_early_ = false;
  if (launch_error_count() > 0) { ok_ = false; err_ = "kernel launch failed"; }
  if (nC > 0 && download) {
    CK(cudaMemcpyAsync(hStatus_, jac_done_early_ ? dStatusF_ : dStatus_, sizeof(int) * nC, cudaMemcpyDeviceToHost, stream_));
    CK(cudaMemcpyAsync(hGamma_, jac_done_early_ ? dGammaF_ : dGamma_, sizeof(double) * nC, cudaMemcpyDeviceToHost, stream_));
  }
  jac_done_early_ = false;
}

// One persistent helper thread for host-side list building (sleeps on a condition variable between frames).
class HostWorker {
 public:
  HostWorker() : th_([this] { loop(); }) {}
  ~HostWorker() {
    { std::lock_guard<std::mutex> g(m_); quit_ = true; }
    cv_.notify_one();
    th_.join();
  }
  void run(std::function<void()> f) {
    { std::lock_guard<std::mutex> g(m_); job_ = std::move(f); has_job_ = true; }
    cv_.notify_one();
  }
 private:
  void loop() {
    for (;;) {
      std::function<void()> f;
      {
        std::unique_lock<std::mutex> g(m_);
        cv_.wait(g, [this] { return has_job_ || quit_; });
        if (quit_) return;
        f = std::move(job_);
        has_job_ = false;
      }
      f();
    }
  }
  std::mutex m_;
  std::condition_variable cv_;
  std::function<void()> job_;
  bool has_job_ = false, quit_ = false;
  std::thread th_;
};

// ORCVIO_HOST_PROF=1: wall-clock checkpoints of the end-to-end host path (mean over calls, printed every 64 calls)
struct HostProf {
  static constexpr int K = 12;
  double acc[K] = {0};
  const char* name[K] = {nullptr};
  int n = 0, calls = 0;
  std::chrono::steady_clock::time_point t;
  bool on = env_int("ORCVIO_HOST_PROF", 0) != 0;
  void start() { if (on) { t = std::chrono::steady_clock::now(); n = 0; } }
  void mark(const char* what) {
    if (!on || n >= K) return;
    const auto now = std::chrono::steady_clock::now();
    acc[n] += std::chrono::duration<double, std::micro>(now - t).count();
    name[n++] = what;
    t = now;
  }
  void done() {
    if (!on || ++calls % 64) return;
    std::fprintf(stderr, "[host prof]");
    for (int i = 0; i < n; ++i) { std::fprintf(stderr, " %s %.1f", name[i], acc[i] / 64); acc[i] = 0; }
    std::fprintf(stderr, "\n");
  }
};
static HostProf g_hp;

static void build_tiles(Batch::PhaseWork& w, int fi, int c0, int c1) {
  FilterWork& fw = w.fw[fi];
  fw.tile_begin = (int)w.tiles.size();
  fw.arow0 = (int)w.arows_total;
  int i = c0;
  while (i < c1) {
    Tile t{};
    t.filter = fi;
    t.cand_begin = i;
    t.c0_blk = w.cands[i].s_blk;
    t.c1_blk = w.cands[i].e_blk + 1;
    t.rows = std::max(2 * w.cands[i].jac_m - 3, 0);        // a one-observation track has no projected row
    int j = i + 1;
    while (j < c1) {
      const Cand& c = w.cands[j];
      const int nc1 = std::max(t.c1_blk, c.e_blk + 1);
      const int wblk = nc1 - t.c0_blk;
      const int own = c.e_blk - c.s_blk + 1;
      if (wblk > std::max(6, own) && c.s_blk != t.c0_blk) break;   // keep k_aform's 36-column chunk
      const int rows = t.rows + std::max(2 * c.jac_m - 3, 0);
      if (rows > AFORM_TILE_ROWS) break;
      if (j - i + 1 > QR_THREADS) break;
      t.c1_blk = nc1;
      t.rows = rows;
      ++j;
    }
    t.cand_end = j;
    t.arow = (int)w.arows_total;
    w.arows_total += (size_t)t.rows;
    w.max_tile_rows = std::max(w.max_tile_rows, t.rows);
    w.wmax_blk = std::max(w.wmax_blk, t.c1_blk - t.c0_blk);
    fw.wmax_blk = std::max(fw.wmax_blk, t.c1_blk - t.c0_blk);
    w.tiles.push_back(t);
    i = j;
  }
  fw.tile_end = (int)w.tiles.size();
  fw.arows = (int)w.arows_total - fw.arow0;
  // staircase of A = [r' | H' L]: a tile with window [c0, c1) fills the columns 0 .. 6 c1 of its rows
  for (int J = 0; J < SY_MAXT; ++J) fw.jrow0[J] = fw.arows;
  for (int t = fw.tile_begin; t < fw.tile_end; ++t)
    for (int J = 0; J < SY_MAXT; ++J)
      if (6 * w.tiles[t].c1_blk >= SY_TILE * J) fw.jrow0[J] = std::min(fw.jrow0[J], w.tiles[t].arow - fw.arow0);
}

// Append one filter's candidates (sorted by first clone, then id) to the phase work list.
static void append_candidates(Batch::PhaseWork& w, int fi, std::vector<CandBuild>& cb,
                              std::vector<CandInfo>& info_out, bool tri_only = false) {
  std::stable_sort(cb.begin(), cb.end(), [](const CandBuild& a, const CandBuild& b) {
    if (a.c.s_blk != b.c.s_blk) return a.c.s_blk < b.c.s_blk;
    return a.id < b.id;
  });
  const int c0 = (int)w.cands.size();
  for (auto& x : cb) {
    Cand c = x.c;
    c.filter = fi;
    const int r = tri_only ? 0 : 2 * c.jac_m - 3;
    c.row_off = (int)w.rows_total;
    c.hblk_off = (int)w.hblk_total;
    w.rows_total += (size_t)std::max(r, 0);
    w.hblk_total += (size_t)std::max(r, 0) * 6 * (c.e_blk - c.s_blk + 1);
    const int idx = (int)w.cands.size();
    if (!tri_only) {
      w.own_wmax_blk = std::max(w.own_wmax_blk, c.e_blk - c.s_blk + 1);
      if (c.jac_m <= 8) w.small_list.push_back(idx);
      else w.large_list.push_back(idx);
    }
    w.cands.push_back(c);
    info_out.push_back(CandInfo{x.id, x.kind});
  }
  if (!tri_only) build_tiles(w, fi, c0, (int)w.cands.size());
}

int Batch::process(const double* t_img, const OrcvioFeature* feats, const int* feat_off,
                   const OrcvioImu* imu, const int* imu_off, int* imu_used, int* published) {
  std::vector<const OrcvioFeature*> fp(B_);
  std::vector<const OrcvioImu*> ip(B_);
  std::vector<int> nf(B_), ni(B_);
  for (int fi = 0; fi < B_; ++fi) {
    fp[fi] = feats + feat_off[fi];
    nf[fi] = feat_off[fi + 1] - feat_off[fi];
    ip[fi] = imu + imu_off[fi];
    ni[fi] = imu_off[fi + 1] - imu_off[fi];
  }
  return process_ptrs(t_img, fp.data(), nf.data(), ip.data(), ni.data(), imu_used, published);
}

// rotationToQuaternion, include/orcvio/utils/math_utils.hpp:188-227 (Hamilton, x y z w, w >= 0)
void rotation_to_quat_xyzw(const double* R, double* q) {
  const double tr = R[0] + R[4] + R[8];
  const double score[4] = {R[0], R[4], R[8], tr};
  int best = 0;
  for (int i = 1; i < 4; ++i)
    if (score[i] > score[best]) best = i;
  if (best == 0) {
    q[0] = std::sqrt(1 + 2 * R[0] - tr) / 2.0;
    q[1] = (R[1] + R[3]) / (4 * q[0]); q[2] = (R[2] + R[6]) / (4 * q[0]); q[3] = (R[7] - R[5]) / (4 * q[0]);
  } else if (best == 1) {
    q[1] = std::sqrt(1 + 2 * R[4] - tr) / 2.0;
    q[0] = (R[1] + R[3]) / (4 * q[1]); q[2] = (R[5] + R[7]) / (4 * q[1]); q[3] = (R[2] - R[6]) / (4 * q[1]);
  } else if (best == 2) {
    q[2] = std::sqrt(1 + 2 * R[8] - tr) / 2.0;
    q[0] = (R[2] + R[6]) / (4 * q[2]); q[1] = (R[5] + R[7]) / (4 * q[2]); q[3] = (R[3] - R[1]) / (4 * q[2]);
  } else {
    q[3] = std::sqrt(1 + tr) / 2.0;
    q[0] = (R[7] - R[5]) / (4 * q[3]); q[1] = (R[2] - R[6]) / (4 * q[3]); q[2] = (R[3] - R[1]) / (4 * q[3]);
  }
  if (q[3] < 0)
    for (int i = 0; i < 4; ++i) q[i] = -q[i];
  const double n = std::sqrt((q[0] * q[0] + q[1] * q[1]) + (q[2] * q[2] + q[3] * q[3]));
  for (int i = 0; i < 4; ++i) q[i] /= n;
}

// ORCVIO_HOST_PROF=2: wall clock of the sections of processFeatures' host side, summed over calls and printed every
// 2000 filter-frames (diagnostic of the multi-trajectory replay, which is bound by this bookkeeping)
struct SecProf {
  static constexpr int K = 12;
  double acc[K] = {0}, cur[K] = {0}, worst[K] = {0};
  double worst_sum = 0.0;
  long long calls = 0, filters = 0;
  std::chrono::steady_clock::time_point t;
  const int mode = env_int("ORCVIO_HOST_PROF", 0);
  const bool on = mode == 2 || mode == 3;
  static const char* name(int i) {
    static const char* nm[K] = {"capacity", "imu+addObs", "prop_launch", "prop_wait", "lost_scan", "spec_tri", "lost_build",
                                "phaseA_launch", "phaseA_wait", "prune_build", "phaseB_launch", "phaseB_wait+post"};
    return nm[i];
  }
  void start() {
    if (!on) return;
    t = std::chrono::steady_clock::now();
    for (double& c : cur) c = 0.0;
  }
  void mark(int k) {
    if (!on) return;
    const auto now = std::chrono::steady_clock::now();
    const double us = std::chrono::duration<double, std::micro>(now - t).count();
    acc[k] += us;
    cur[k] += us;
    t = now;
  }
  void done(int B) {
    if (!on) return;
    double sum = 0.0;
    for (double c : cur) sum += c;
    if (sum > worst_sum) {                     // the slowest call of this thread so far: where did it spend its time
      worst_sum = sum;
      for (int i = 0; i < K; ++i) worst[i] = cur[i];
    }
    ++calls;
    filters += B;
    if (mode != 2 || filters < 2000) return;
    std::fprintf(stderr, "[host prof] us per filter-frame:");
    for (int i = 0; i < K; ++i) { std::fprintf(stderr, " %s %.2f", name(i), acc[i] / filters); acc[i] = 0; }
    std::fprintf(stderr, "  (%lld calls)\n", calls);
    calls = filters = 0;
  }
  void report_worst() {
    if (mode != 3) return;
    std::fprintf(stderr, "[replay prof] slowest call %.1f ms:", worst_sum / 1e3);
    for (int i = 0; i < K; ++i)
      if (worst[i] > 0.02 * worst_sum) std::fprintf(stderr, " %s %.1f ms", name(i), worst[i] / 1e3);
    std::fprintf(stderr, "\n");
    worst_sum = 0.0;
  }
};
static thread_local SecProf g_sp;

// Whole-sequence replay (Monte-Carlo / multi-sequence batches, SURVEY 8e): every filter's IMU stream and frames are
// handed over once; the lock-step loop over the frames runs here, so a replay costs the caller one call (the callers
// drive several batches from as many host threads).  poses_out: n_filters x n_frames x 7, the IMU pose after every
// frame (position, quaternion x y z w: one line of the reference's state_est_geo_feat.txt log, src/orcvio.cpp:643-645);
// ok_out[i] = 0 when some frame of filter i was not published.
//
// state17_out (n_filters x n_frames x 17: IM_TIME, p, q xyzw, v, b_g, b_a) comes from the host mirror like poses_out.
// cov15_out (n_filters x n_frames x 225) is captured on the device: after frame f, k_capture_imu_cov copies the leading
// 15 x 15 block of every filter's P into dCovHist_[i, f], and the history comes down once at the end.  The capture is
// queued on stream_ behind the whole frame.  Every kernel that writes P runs on stream_ (propagation, augmentation,
// ZUPT, k_compact_cov, k_reanchor, the update chain -- k_pinfo -- with the hybrid post kernels, k_remove;
// the initial covariance is a memset + copy on stream_), and the side stream stream2_ only reads P (k_chol_prior,
// k_imu_factor) and is joined to stream_ (ev_join_, ev_ls_) before the update writes it.  The next frame's P writers
// are queued on stream_ after the capture, and its side-stream work forks from stream_ after it (ev_fork_): nothing
// overwrites P before the capture has read it.
int Batch::replay(int n_frames, const double* t_img, const OrcvioFeature* const* feats, const int* feat_off,
                  const OrcvioImu* const* imu, const int* n_imu, double imu_window, double* poses_out, int* ok_out,
                  double* state17_out, double* cov15_out) {
  if (cov15_out && n_frames > 0) {
    const size_t need = (size_t)B_ * n_frames * 225;
    if (need > covhist_cap_) {                           // grown ahead of the loop, never inside it
      cudaSetDevice(dev_);
      if (dCovHist_) cudaFree(dCovHist_);
      dCovHist_ = nullptr;
      covhist_cap_ = 0;
      note_growth("covariance history", need * sizeof(double));
      if (cudaMalloc(&dCovHist_, need * sizeof(double)) != cudaSuccess) {
        dCovHist_ = nullptr;
        return ORCVIO_ERR_CUDA;
      }
      covhist_cap_ = need;
    }
  }
  std::vector<const OrcvioFeature*> fp(B_);
  std::vector<const OrcvioImu*> ip(B_);
  std::vector<int> nf(B_), ni(B_), cursor(B_, 0), used(B_), pub(B_);
  std::vector<double> tt(B_);
  for (int i = 0; i < B_; ++i) ok_out[i] = 1;
  // ORCVIO_HOST_PROF=3: wall clock of every frame of this batch (stalls of a replay thread show up as outliers)
  static const bool frame_prof = env_int("ORCVIO_HOST_PROF", 0) == 3;
  std::vector<double> frame_ms;
  for (int f = 0; f < n_frames; ++f) {
    for (int i = 0; i < B_; ++i) {
      const int* fo = feat_off + (size_t)i * (n_frames + 1);
      tt[i] = t_img[(size_t)i * n_frames + f];
      fp[i] = feats[i] + fo[f];
      nf[i] = fo[f + 1] - fo[f];
      // the samples up to the image stamp (+ a margin): what a driver would have queued by now; the filter consumes a
      // prefix of them (batchImuProcessing :664-724) and the rest is offered again with the next frame
      int k1 = cursor[i];
      while (k1 < n_imu[i] && imu[i][k1].t <= tt[i] + imu_window) ++k1;
      ip[i] = imu[i] + cursor[i];
      ni[i] = k1 - cursor[i];
    }
    const auto tf0 = std::chrono::steady_clock::now();
    const int rc = process_ptrs(tt.data(), fp.data(), nf.data(), ip.data(), ni.data(), used.data(), pub.data());
    if (rc != ORCVIO_OK) return rc;
    if (frame_prof) frame_ms.push_back(std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tf0).count());
    for (int i = 0; i < B_; ++i) {
      cursor[i] += used[i];
      if (!pub[i]) ok_out[i] = 0;
      const double* im = f_[i].imu_mirror.data();
      double* o = poses_out + ((size_t)i * n_frames + f) * 7;
      for (int k = 0; k < 3; ++k) o[k] = im[IM_P + k];
      rotation_to_quat_xyzw(im + IM_R, o + 3);
      if (state17_out) {
        double* s = state17_out + ((size_t)i * n_frames + f) * 17;
        s[0] = im[IM_TIME];
        for (int k = 0; k < 7; ++k) s[1 + k] = o[k];
        for (int k = 0; k < 3; ++k) {
          s[8 + k] = im[IM_V + k];
          s[11 + k] = im[IM_BG + k];
          s[14 + k] = im[IM_BA + k];
        }
      }
    }
    if (cov15_out) {
      launch_capture_imu_cov(dP_, (size_t)ldp_ * ldp_, ldp_, B_, dCovHist_, n_frames, f, stream_);
      ++launches_;
    }
  }
  if (cov15_out && n_frames > 0) {
    CK(cudaMemcpyAsync(cov15_out, dCovHist_, (size_t)B_ * n_frames * 225 * sizeof(double), cudaMemcpyDeviceToHost,
                       stream_));
    CK(cudaStreamSynchronize(stream_));
    if (launch_error_count() > 0) { ok_ = false; err_ = "kernel launch failed"; }
    if (!ok_) return ORCVIO_ERR_CUDA;
  }
  if (frame_prof && !frame_ms.empty()) {
    std::vector<double> v = frame_ms;
    std::sort(v.begin(), v.end());
    double sum = 0.0;
    for (double x : v) sum += x;
    int slow = 0;
    for (double x : v) slow += x > 3.0 * v[v.size() / 2];
    std::fprintf(stderr, "[replay prof] %d filters x %zu frames: total %.1f ms, per frame min %.2f median %.2f p90 %.2f max %.2f ms, "
                 "%d frames above 3 x median; first 5:", B_, v.size(), sum, v.front(), v[v.size() / 2], v[v.size() * 9 / 10],
                 v.back(), slow);
    for (size_t i = 0; i < std::min<size_t>(5, frame_ms.size()); ++i) std::fprintf(stderr, " %.2f", frame_ms[i]);
    std::fprintf(stderr, "\n");
    g_sp.report_worst();
  }
  return ORCVIO_OK;
}


int Batch::process_ptrs(const double* t_img, const OrcvioFeature* const* featp, const int* nfeat,
                        const OrcvioImu* const* imup, const int* nimu_v, int* imu_used, int* published) {
  if (!ok_) return ORCVIO_ERR_CUDA;
  g_sp.start();
  cudaSetDevice(dev_);                // the current device is per host thread (replays run on worker threads)
  const int L = ORCVIO_LEG;
  // Capacity is checked before anything is touched: a frame either runs on every filter or leaves all of them as
  // they were (a failure in the middle of the per-filter loop would leave host bookkeeping and device state apart).
  if (!p_.prediction_only_flag)
    for (int fi = 0; fi < B_; ++fi) {
      const FilterHost& F = f_[fi];
      const OrcvioFeature* ft = featp[fi];
      const int nf = nfeat[fi];
      if ((size_t)nf <= F.free_slots.size()) continue;     // even if every feature is new there is room
      size_t fresh = 0;
      for (int k = 0; k < nf; ++k) fresh += F.find_track((long long)ft[k].id) ? 0 : 1;
      if (fresh > F.free_slots.size()) {
        std::fprintf(stderr, "[orcvio_b200] feature table full (capacity %d live tracks per filter, filter %d needs %zu more)\n",
                     Fcap_, fi, fresh - F.free_slots.size());
        return ORCVIO_ERR_CAPACITY;
      }
    }
  g_sp.mark(0);
  // ---------------------------------------------------------------- A: propagation inputs
  std::vector<PropSample> samples;
  std::vector<int> samp_off(B_ + 1, 0), Dvec(B_, 0), Nvec(B_, 0), Evec(B_, 0);
  bool need_imu_upload = false;
  for (int fi = 0; fi < B_; ++fi) {
    FilterHost& F = f_[fi];
    F.active = false;
    F.stats = OrcvioFrameStats{};
    F.stats.removed_ids[0] = F.stats.removed_ids[1] = -1;
    F.cinfo[0].clear(); F.cinfo[1].clear();
    F.cstatus[0].clear(); F.cstatus[1].clear();
    F.cgamma[0].clear(); F.cgamma[1].clear();
    F.log_ekf_lost.clear(); F.log_ekf_ids.clear(); F.log_new_ids.clear(); F.log_ekf_pass.clear();
    F.log_new_ok.clear(); F.log_ekf_gamma.clear(); F.log_new_gamma.clear(); F.log_reanchor.clear();
    published[fi] = 0;
    imu_used[fi] = 0;
    samp_off[fi + 1] = (int)samples.size();
    const OrcvioImu* im = imup[fi];
    const int nimu = nimu_v[fi];
    const double ti = t_img[fi];
    if (!F.first_features) {   // :504-510
      if (nimu > 0 && (im[0].t - ti - p_.td <= 0.0)) F.first_features = true;
      else continue;
    }
    int prefix = 0;
    if (!F.gravity_set) {      // :513-563, initial_use_gt branch only
      if (!F.has_init) continue;
      int useful = 0;
      for (int k = 0; k < nimu; ++k) {
        if (im[k].t > F.init_t) break;
        ++useful;
      }
      if (useful >= nimu) --useful;
      if (useful < 0) continue;
      init_filter_device(fi);
      double* hm = hImu_ + (size_t)fi * IM_STRIDE;
      for (int k = 0; k < 3; ++k) {
        hm[IM_GOLD + k] = im[useful].gyro[k];
        hm[IM_AOLD + k] = im[useful].acc[k];
      }
      CK(cudaMemcpyAsync(dImu_ + (size_t)fi * IM_STRIDE, hm, IM_STRIDE * sizeof(double), cudaMemcpyHostToDevice, stream_));
      need_imu_upload = true;
      prefix = useful;
      F.gravity_set = true;
      F.imu_time = F.init_t;
      F.take_off_stamp = F.init_t;
      F.last_zupt_time = F.init_t;       // :556
    }
    // batchImuProcessing :664-724
    const double bound = ti + p_.td;
    int used = 0;
    double dt = 0.0;
    for (int k = prefix; k < nimu; ++k) {
      const double t = im[k].t;
      if (t <= F.imu_time) { ++used; continue; }
      if (t - bound > p_.imu_img_timeTh) break;
      PropSample s;
      s.t = t;
      for (int q = 0; q < 3; ++q) { s.w[q] = im[k].gyro[q]; s.a[q] = im[k].acc[q]; }
      samples.push_back(s);
      dt = t - bound;
      F.imu_time = t;
      ++used;
    }
    samp_off[fi + 1] = (int)samples.size();
    F.state_id = F.next_state_id++;
    F.dt = dt;
    imu_used[fi] = prefix + used;
    Nvec[fi] = (int)F.clones.size();
    Evec[fi] = (int)F.feature_states.size();
    Dvec[fi] = L + 6 * Nvec[fi] + Evec[fi];
    F.active = true;
    published[fi] = 1;

    // addFeatureObservations :1016-1068
    if (!p_.prediction_only_flag) {
      const OrcvioFeature* ft = featp[fi];
      const int nf = nfeat[fi];
      const long long sid = F.state_id;
      const int curr_feature_num = (int)F.map_server.size();
      int tracked = 0;
      for (int k = 0; k < nf; ++k) {
        const OrcvioFeature& m = ft[k];
        const long long id = (long long)m.id;
        Track* found = F.find_track(id);
        if (!found) {
          if (F.free_slots.empty()) {      // (cannot happen after the pre-pass; if it does the batch is unusable)
            std::fprintf(stderr, "[orcvio_b200] feature table full (capacity %d)\n", Fcap_);
            ok_ = false;
            err_ = "feature table overflow in the middle of a frame";
            return ORCVIO_ERR_CAPACITY;
          }
          Track tr;
          tr.id = id;
          tr.slot = F.free_slots.back();
          F.free_slots.pop_back();
          tr.gen = F.next_gen++;
          bool have_prev = false;
          double dt_prev = 0.0;
          if (!(m.u_init == -1 && m.v_init == -1)) {
            for (const auto& c : F.clones)
              if (c.id == sid - 1) { have_prev = true; dt_prev = c.dt; }
          }
          if (have_prev) {
            Obs o{};
            o.sid = sid - 1;
            o.z[0] = m.u_init + m.u_init_vel * dt_prev;
            o.z[1] = m.v_init + m.v_init_vel * dt_prev;
            o.vel[0] = m.u_init_vel; o.vel[1] = m.v_init_vel;
            tr.obs.push_back(o);
          }
          Obs o{};
          o.sid = sid;
          o.z[0] = m.u + m.u_vel * dt;
          o.z[1] = m.v + m.v_vel * dt;
          o.vel[0] = m.u_vel; o.vel[1] = m.v_vel;
          tr.obs.push_back(o);
          tr.touch();
          F.add_track(std::move(tr));
        } else {
          Obs o{};
          o.sid = sid;
          o.z[0] = m.u + m.u_vel * dt;
          o.z[1] = m.v + m.v_vel * dt;
          o.vel[0] = m.u_vel; o.vel[1] = m.v_vel;
          Track& tr = *found;
          if (!tr.obs.empty() && tr.obs.back().sid == sid) tr.obs.back() = o;
          else tr.obs.push_back(o);
          tr.touch();
          ++tracked;
          if (p_.if_ZUPT_valid && p_.if_use_feature_zupt_flag) {     // :1052-1058
            // (the observations are in ascending state-id order and end with this frame's: the previous frame's, if
            // there is one, is the one before it)
            if (tr.obs.size() >= 2 && tr.obs[tr.obs.size() - 2].sid == sid - 1) {
              const Obs& po = tr.obs[tr.obs.size() - 2];
              const double du = m.u - po.z[0], dv = m.v - po.z[1];
              F.coarse_feature_dis.push_back(std::sqrt(du * du + dv * dv));
            }
          }
        }
      }
      F.tracking_rate = (double)tracked / (double)curr_feature_num;   // 0/0 -> NaN like the reference
    }
    // stateAugmentation bookkeeping :937-961
    F.cur_window_timestamps.push_back(F.imu_time);
    F.clones.push_back(CloneMeta{F.state_id, F.imu_time, F.dt});
  }
  (void)need_imu_upload;
  g_sp.mark(1);

  // ---------------------------------------------------------------- B: propagate + augment
  {
    blob_.reset();
    const size_t o_s = blob_.reserve(sizeof(PropSample) * std::max<size_t>(samples.size(), 1));
    const size_t o_o = blob_.reserve(sizeof(int) * (B_ + 1));
    const size_t o_d = blob_.reserve(sizeof(int) * B_);
    const size_t o_n = blob_.reserve(sizeof(int) * B_);
    const size_t o_e = blob_.reserve(sizeof(int) * B_);
    char* h = blob_.pinned;
    std::memcpy(h + o_e, Evec.data(), sizeof(int) * B_);
    if (!samples.empty()) std::memcpy(h + o_s, samples.data(), sizeof(PropSample) * samples.size());
    std::memcpy(h + o_o, samp_off.data(), sizeof(int) * (B_ + 1));
    std::memcpy(h + o_d, Dvec.data(), sizeof(int) * B_);
    // augmentation only for active filters: N = -1 disables
    std::vector<int> Naug(B_);
    for (int fi = 0; fi < B_; ++fi) Naug[fi] = f_[fi].active ? Nvec[fi] : -1;
    std::memcpy(h + o_n, Naug.data(), sizeof(int) * B_);
    // ZUPT (:583-592): the feature test (checkZUPTFeat :3081-3125) is a host decision on the sorted
    // track displacements; the IMU test (checkZUPTIMU) needs P and runs inside k_zupt.
    size_t o_zm = 0, o_zn = 0, o_zc = 0;
    bool any_zupt = false;
    if (p_.if_ZUPT_valid) {
      std::vector<int> zmode(B_, 0), zN(B_, -1);
      std::vector<double> zchk(B_, 0.0);
      for (int fi = 0; fi < B_; ++fi) {
        FilterHost& F = f_[fi];
        F.if_zupt = false;
        if (!F.active) continue;
        zN[fi] = Nvec[fi] + 1;
        if (p_.if_use_feature_zupt_flag) {
          std::vector<double>& d = F.coarse_feature_dis;
          if (d.size() >= 20) {
            // (the reference sorts and reads element size - 9: the same order statistic without the full sort)
            std::nth_element(d.begin(), d.end() - 9, d.end());
            if (d[d.size() - 9] < p_.zupt_max_feature_dis) zmode[fi] = 1;
          }
          d.clear();
        } else {
          const int cnt = samp_off[fi + 1] - samp_off[fi];
          if (cnt >= 2) {
            zmode[fi] = 2;
            const int dof = 6 * (cnt - 1);
            zchk[fi] = dof < 500 ? chi2_zupt_host_[dof] : chi2_quantile(0.95, dof);
          }
        }
        any_zupt |= zmode[fi] != 0;
      }
      o_zm = blob_.reserve(sizeof(int) * B_);
      o_zn = blob_.reserve(sizeof(int) * B_);
      o_zc = blob_.reserve(sizeof(double) * B_);
      h = blob_.pinned;
      std::memcpy(h + o_zm, zmode.data(), sizeof(int) * B_);
      std::memcpy(h + o_zn, zN.data(), sizeof(int) * B_);
      std::memcpy(h + o_zc, zchk.data(), sizeof(double) * B_);
    }
    upload_blob();
    if (profiling_) CK(cudaEventRecord(ev_[6], stream_));
    PropArgs pa{};
    pa.P = dP_; pa.p_stride = (size_t)ldp_ * ldp_; pa.ldp = ldp_;
    pa.imu = dImu_;
    pa.samples = (const PropSample*)(blob_.dev + o_s);
    pa.samp_off = (const int*)(blob_.dev + o_o);
    pa.D = (const int*)(blob_.dev + o_d);
    pa.n_filters = B_; pa.flags = flags_;
    pa.qc[0] = p_.imu_gyro_noise; pa.qc[1] = p_.imu_acc_noise;
    pa.qc[2] = p_.imu_gyro_bias_noise; pa.qc[3] = p_.imu_acc_bias_noise;
    launch_propagate(pa, stream_);
    AugArgs aa{};
    aa.P = dP_; aa.p_stride = pa.p_stride; aa.ldp = ldp_;
    aa.imu = dImu_; aa.clones = dClones_; aa.clone_stride = (size_t)Ncap_ * CL_STRIDE;
    aa.N = (const int*)(blob_.dev + o_n); aa.n_filters = B_;
    aa.E = hybrid_ ? (const int*)(blob_.dev + o_e) : nullptr;
    launch_augment(aa, stream_);
    launches_ += 2;
    if (any_zupt) {
      ZuptArgs za{};
      za.P = dP_; za.p_stride = pa.p_stride; za.ldp = ldp_;
      za.imu = dImu_; za.clones = dClones_; za.clone_stride = aa.clone_stride;
      za.samples = pa.samples; za.samp_off = pa.samp_off;
      za.N = (const int*)(blob_.dev + o_zn);
      za.mode = (const int*)(blob_.dev + o_zm);
      za.chi2_check = (const double*)(blob_.dev + o_zc);
      za.decision = dZuptDec_; za.info = dZuptInfo_;
      za.dx = dDx_; za.lddx = ldp_;
      za.n_filters = B_; za.flags = flags_;
      za.noise_v = p_.zupt_noise_v; za.noise_p = p_.zupt_noise_p; za.noise_q = p_.zupt_noise_q;
      launch_zupt(za, stream_);
      ++launches_;
      CK(cudaMemcpyAsync(hZuptDec_, dZuptDec_, sizeof(int) * B_, cudaMemcpyDeviceToHost, stream_));
      CK(cudaMemcpyAsync(hZuptInfo_, dZuptInfo_, sizeof(double) * 2 * B_, cudaMemcpyDeviceToHost, stream_));
    }
    if (profiling_) {
      CK(cudaEventRecord(ev_[7], stream_));
    }
    // the blob is reused by the next phase: wait for the upload + kernels reading it
    g_sp.mark(2);
    wait_stream();
    g_sp.mark(3);
    if (profiling_) {
      float ms = 0;
      cudaEventElapsedTime(&ms, ev_[6], ev_[7]);
      pt_.prop += ms; pt_.n_prop++;
    }
    if (any_zupt) {
      for (int fi = 0; fi < B_; ++fi) {
        FilterHost& F = f_[fi];
        if (!F.active) continue;
        F.if_zupt = hZuptDec_[fi] != 0;
        F.zupt_chi2 = hZuptInfo_[2 * fi];
        F.zupt_vnorm = hZuptInfo_[2 * fi + 1];
        F.stats.zupt = F.if_zupt ? 1 : 0;
        F.stats.zupt_chi2 = F.zupt_chi2;
        F.stats.zupt_vnorm = F.zupt_vnorm;
        if (F.if_zupt) {
          F.last_zupt_time = F.imu_time;                 // :3451
          // checkZUPTFeat :3104-3115 / checkZUPTIMU :3304-3315: a stationary frame drops every EKF-SLAM feature; the
          // update itself only touched the leading 22 + 6N block, the feature rows / columns are simply abandoned
          for (long long id : F.feature_states) {
            Track& tr = *F.find_track(id);
            tr.in_state = tr.ekf_feature = tr.initialized = false;
            tr.gen = F.next_gen++;                       // the device slot no longer counts as initialised
          }
          F.feature_states.clear();
        }
      }
    }
  }

  // ---------------------------------------------------------------- C: removeLostFeatures
  PhaseWork wA;
  wA.fw.assign(B_, FilterWork{});
  wA.cand_begin.assign(B_ + 1, 0);
  if (hybrid_) { wA.hyb_phase = 0; wA.hw.assign(B_, HybWork{}); }
  // state id -> index in the window.  The window does not change between augmentation (above) and the end of the frame,
  // and its ids span a few dozen consecutive values: one small table per filter instead of a search per observation.
  std::vector<std::vector<short>> clone_lut(B_);
  for (int fi = 0; fi < B_; ++fi) {
    const FilterHost& F = f_[fi];
    if (!F.active || F.clones.empty()) continue;
    const long long base = F.clones.front().id, span = F.clones.back().id - base + 1;
    if (span > 4096) continue;                             // (never seen: falls back to the search)
    clone_lut[fi].assign((size_t)span, (short)-1);
    for (int k = 0; k < (int)F.clones.size(); ++k) clone_lut[fi][(size_t)(F.clones[k].id - base)] = (short)k;
  }
  const FilterHost* f_base = f_.data();
  auto clone_index_of = [&clone_lut, f_base](const FilterHost& F, long long sid) {
    const std::vector<short>& lut = clone_lut[&F - f_base];
    if (!lut.empty()) {
      const long long off = sid - F.clones.front().id;
      return (off >= 0 && off < (long long)lut.size()) ? (int)lut[(size_t)off] : -1;
    }
    for (int k = (int)F.clones.size() - 1; k >= 0; --k)
      if (F.clones[k].id == sid) return k;
    return -1;
  };
  // one candidate record + its observations in the pools of w (lost / tracked-long feature of removeLostFeatures)
  auto make_cand = [&](PhaseWork& w, const FilterHost& F, const Track& tr, bool tracked_now, int kind, int flags) {
    CandBuild x{};
    x.id = tr.id;
    x.kind = kind;
    Cand& c = x.c;
    c.slot = tr.slot;
    c.gen = tr.gen;
    c.flags = flags;
    c.jac_off = c.tri_off = (int)w.obs_clone.size();
    int s_blk = 1 << 30, e_blk = -1, cnt = 0;
    for (const Obs& o : tr.obs) {
      const int ci = clone_index_of(F, o.sid);
      if (ci < 0) continue;
      w.obs_clone.push_back(ci);
      w.obs_z.push_back(o.z[0]);
      w.obs_z.push_back(o.z[1]);
      s_blk = std::min(s_blk, ci);
      e_blk = std::max(e_blk, ci);
      ++cnt;
    }
    c.jac_m = cnt;
    c.tri_m = tracked_now ? cnt - 1 : cnt;   // initializePosition skips the current frame (:414)
    c.s_blk = s_blk;
    c.e_blk = e_blk;
    c.cm_first_clone = w.obs_clone[c.jac_off];
    c.cm_last_clone = w.obs_clone[c.jac_off + (tracked_now ? cnt - 2 : cnt - 1)];
    c.cm_zu = w.obs_z[2 * (size_t)c.jac_off];
    c.cm_zv = w.obs_z[2 * (size_t)c.jac_off + 1];
    return x;
  };
  std::vector<std::vector<CandBuild>> cbs(B_);
  // hybrid mode (:2283-2323): tracked-long features whose grid cell had room when the walk started.  Whether such a
  // feature becomes an EKF-SLAM feature depends on the triangulation outcome of the ones before it (cells fill up in
  // id order), so initializeInvParamPosition runs speculatively for all of them into a scratch table; the host then
  // replays the reference's sequential decision and commits the ones that took the branch.
  struct PossRec { Track* tr; int code; int spec; long long spec_gen; };
  std::vector<std::vector<PossRec>> poss(B_);
  std::vector<std::map<int, int>> cells(B_);
  std::vector<std::vector<Track*>> news(B_);
  PhaseWork wS;
  HybridBufs* hb = hyb_.get();
  bool hyb_ok = true;
  if (hybrid_) {
    hb->used = 0;                          // the stream is idle (synchronised at the end of section B)
    std::vector<int> newidx, Dold(B_, 0);
    bool any_compact = false;
    for (int fi = 0; fi < B_; ++fi) {
      FilterHost& F = f_[fi];
      if (!F.active || F.feature_states.empty()) continue;
      // features of the state: tracked now -> a 2-row update; lost -> dropped (:2210-2232, rmLostFeaturesCov :3776-3828)
      const int base = L + 6 * (int)F.clones.size(), E0 = (int)F.feature_states.size();
      std::vector<long long> kept;
      std::vector<int> map_e(E0, -1);
      for (int i = 0; i < E0; ++i) {
        Track& tr = *F.find_track(F.feature_states[i]);
        if (!tr.obs.empty() && tr.obs.back().sid == F.state_id) {
          map_e[i] = (int)kept.size();
          kept.push_back(tr.id);
        } else {
          const long long lost_id = tr.id;
          F.log_ekf_lost.push_back(lost_id);
          F.free_slots.push_back(tr.slot);
          F.erase_track(lost_id);
        }
      }
      if ((int)kept.size() != E0) {
        if (newidx.empty()) newidx.assign((size_t)B_ * ldp_, -1);
        int* ni = newidx.data() + (size_t)fi * ldp_;
        for (int j = 0; j < base; ++j) ni[j] = j;
        for (int i = 0; i < E0; ++i) ni[base + i] = map_e[i] < 0 ? -1 : base + map_e[i];
        Dold[fi] = base + E0;
        any_compact = true;
        F.feature_states = kept;
      }
    }
    if (any_compact) {
      const int* d_ni = hb->put(newidx.data(), newidx.size(), stream_, &hyb_ok);
      const int* d_do = hb->put(Dold.data(), Dold.size(), stream_, &hyb_ok);
      if (hyb_ok) { launch_compact_cov(dP_, (size_t)ldp_ * ldp_, ldp_, d_ni, d_do, B_, stream_); ++launches_; }
    }
  }
  auto grid_code = [&](const Track& tr) {   // :2286-2289 / :3841-3845 (the casts truncate toward zero)
    const double* z = tr.obs.back().z;
    const int row = (int)((z[1] - p_.y_min) / p_.grid_height);
    const int col = (int)((z[0] - p_.x_min) / p_.grid_width);
    return row * p_.grid_cols + col;
  };
  for (int fi = 0; fi < B_; ++fi) {
    FilterHost& F = f_[fi];
    FilterWork& fw = wA.fw[fi];
    fw.N = (int)F.clones.size();
    fw.D = L + 6 * fw.N + (int)F.feature_states.size();
    fw.active = 0;
    if (!F.active) continue;
    wA.maxN = std::max(wA.maxN, fw.N);
    const long long cur = F.state_id;
    std::vector<CandBuild>& cb = cbs[fi];
    std::vector<long long> invalid;
    bool ekf_open = false;
    if (hybrid_) {
      for (long long id : F.feature_states) cells[fi][grid_code(*F.find_track(id))]++;   // updateGridMap :3831-3850
      ekf_open = (F.imu_time - F.last_zupt_time > 5) && (int)F.feature_states.size() < Emax_;
    }
    for (auto& kv : F.map_server) {
      Track& tr = kv.second;
      if (tr.in_state) continue;
      const int nobs = (int)tr.obs.size();
      const bool tracked_now = nobs > 0 && tr.last_sid == cur;
      if (!tracked_now) {
        if (nobs < p_.least_Obs_Num) { invalid.push_back(tr.id); continue; }
      } else {
        if (!(nobs >= p_.max_track_len)) continue;
        if (ekf_open) {
          const int code = grid_code(tr);
          auto it = cells[fi].find(code);
          if ((it == cells[fi].end() ? 0 : it->second) < p_.max_features) {
            PossRec pr{&tr, code, -1, 0};
            if (!tr.ekf_feature) {
              // is_initialized = false (:2296): a fresh serial, so the kernel starts from the two-view guess
              pr.spec_gen = F.next_gen++;
              Track probe = tr;
              probe.gen = pr.spec_gen;
              CandBuild x = make_cand(wS, F, probe, true, 1, 0);
              x.c.filter = fi;
              pr.spec = (int)wS.cands.size();
              wS.cands.push_back(x.c);
            }
            poss[fi].push_back(pr);
            continue;
          }
        }
      }
      cb.push_back(make_cand(wA, F, tr, tracked_now, tracked_now ? 1 : 0, 0));
    }
    for (long long id : invalid) {
      F.free_slots.push_back(F.find_track(id)->slot);
      F.erase_track(id);
    }
  }
  g_sp.mark(4);
  std::vector<CommitRec> commits;
  if (hybrid_ && !wS.cands.empty()) {
    const size_t nS = wS.cands.size();
    if (nS > hb->spec_cap) {
      cudaFree(hb->dFinal); cudaFree(hb->dSpecStatus);
      if (hb->hSpecStatus) cudaFreeHost(hb->hSpecStatus);
      hb->spec_cap = nS * 2 + 64;
      note_growth("speculative triangulation (device + pinned)", hb->spec_cap * 28);
      CK(cudaMalloc(&hb->dFinal, hb->spec_cap * 3 * sizeof(double)));
      CK(cudaMalloc(&hb->dSpecStatus, hb->spec_cap * sizeof(int)));
      CK(cudaMallocHost(&hb->hSpecStatus, hb->spec_cap * sizeof(int)));
    }
    TriArgs ta{};
    ta.cand = hb->put(wS.cands.data(), nS, stream_, &hyb_ok); ta.n_cand = (int)nS;
    ta.clones = dClones_; ta.clone_stride = (size_t)Ncap_ * CL_STRIDE;
    ta.fpos = hb->dSpecPos; ta.fgen = hb->dSpecGen; ta.fcap = Fcap_;
    ta.obs_clone = hb->put(wS.obs_clone.data(), wS.obs_clone.size(), stream_, &hyb_ok);
    ta.obs_z = hb->put(wS.obs_z.data(), wS.obs_z.size(), stream_, &hyb_ok);
    ta.cfg = tricfg_;
    ta.status = hb->dSpecStatus;
    ta.final_pos = hb->dFinal;
    if (hyb_ok) {
      launch_triangulate(ta, stream_);
      ++launches_;
      CK(cudaMemcpyAsync(hb->hSpecStatus, hb->dSpecStatus, nS * sizeof(int), cudaMemcpyDeviceToHost, stream_));
      wait_stream();
    }
  }
  g_sp.mark(5);
  for (int fi = 0; fi < B_; ++fi) {
    FilterHost& F = f_[fi];
    wA.cand_begin[fi] = (int)wA.cands.size();
    FilterWork& fw = wA.fw[fi];
    if (!F.active) continue;
    std::vector<CandBuild>& cb = cbs[fi];
    const int E = (int)F.feature_states.size();
    if (hybrid_) {
      // the reference's sequential grid decision (:2291-2323), now that every triangulation outcome is known
      int n_new = 0;
      for (PossRec& pr : poss[fi]) {
        Track& tr = *pr.tr;
        int& cell = cells[fi][pr.code];
        if (!(cell < p_.max_features && E + n_new < Emax_)) {       // no room any more: an MSCKF feature
          cb.push_back(make_cand(wA, F, tr, true, 1, 0));
          continue;
        }
        if (!tr.ekf_feature) {
          tr.gen = pr.spec_gen;                                      // is_initialized = false
          tr.initialized = false;
          if (!(hb->hSpecStatus[pr.spec] & ST_TRI_VALID)) continue;  // checkMotion / triangulation failed (:2297-2303)
          tr.ekf_feature = true;
          tr.initialized = true;
          for (int k = (int)tr.obs.size() - 1; k >= 0; --k)          // anchor = the last camera used (feature.hpp:536)
            if (tr.obs[k].sid != F.state_id && clone_index_of(F, tr.obs[k].sid) >= 0) { tr.id_anchor = tr.obs[k].sid; break; }
          commits.push_back(CommitRec{pr.spec, fi * Fcap_ + tr.slot, tr.gen});
        }
        news[fi].push_back(&tr);
        ++cell;
        ++n_new;
      }
    }
    F.stats.n_candidates_lost = (int)cb.size();
    if (cb.empty() && E == 0 && news[fi].empty()) continue;
    if (F.if_zupt) {
      // :2564-2569: under ZUPT the candidates are still initialised (and the failures erased) but
      // no Jacobian is stacked and no update runs
      append_candidates(wA, fi, cb, F.cinfo[0], true);
      continue;
    }
    fw.active = 1;
    wA.any_active = true;
    append_candidates(wA, fi, cb, F.cinfo[0]);
    if (hybrid_) {
      HybWork& hw = wA.hw[fi];
      hw.N = fw.N; hw.E = E; hw.active = 1;
      hw.feat_begin = (int)wA.hfeats.size();
      for (long long id : F.feature_states) {
        const Track& tr = *F.find_track(id);
        HybFeat hf{};
        hf.slot = tr.slot;
        hf.anchor = clone_index_of(F, tr.id_anchor);
        hf.zu = tr.obs.back().z[0];
        hf.zv = tr.obs.back().z[1];
        if (hf.anchor < 0) { hyb_ok = false; hf.anchor = 0; }
        wA.hfeats.push_back(hf);
      }
      hw.feat_end = (int)wA.hfeats.size();
      hw.new_begin = (int)wA.hnews.size();
      int nd = 2 * E;
      for (Track* trp : news[fi]) {
        // its MSCKF rows over every observation only decide the gate (:2365-2370); they are not stacked
        CandBuild x = make_cand(wA, F, *trp, true, 3, CAND_GATE_ONLY);
        Cand c = x.c;
        c.filter = fi;
        const int r = std::max(2 * c.jac_m - 3, 0);
        c.row_off = (int)wA.rows_total;
        c.hblk_off = (int)wA.hblk_total;
        wA.rows_total += (size_t)r;
        wA.hblk_total += (size_t)r * 6 * (c.e_blk - c.s_blk + 1);
        wA.own_wmax_blk = std::max(wA.own_wmax_blk, c.e_blk - c.s_blk + 1);
        const int idx = (int)wA.cands.size();
        (c.jac_m <= 8 ? wA.small_list : wA.large_list).push_back(idx);
        wA.cands.push_back(c);
        F.cinfo[0].push_back(CandInfo{x.id, 3});
        HybNew hn{};
        hn.slot = trp->slot;
        hn.anchor = clone_index_of(F, trp->id_anchor);
        hn.cand = idx;
        hn.obs_off = c.jac_off;
        hn.obs_m = c.jac_m;
        hn.row_off = nd - 2 * E;
        if (hn.anchor < 0) { hyb_ok = false; hn.anchor = 0; }
        nd += 2 * (c.jac_m - 1) - 1;
        wA.hnews.push_back(hn);
      }
      hw.new_end = (int)wA.hnews.size();
      hw.dense_off = (int)wA.dense_total;
      hw.n_dense = nd;
      hw.arow_dense = fw.arows;
      fw.dense_rows = nd;
      for (int J = 0; J < SY_MAXT; ++J) fw.jrow0[J] = std::min(fw.jrow0[J], fw.arows);
      fw.arows += nd;
      wA.arows_total += (size_t)nd;
      wA.dense_total += (size_t)nd;
      wA.max_dense = std::max(wA.max_dense, nd);
      wA.maxE = std::max(wA.maxE, E);
    }
  }
  wA.cand_begin[B_] = (int)wA.cands.size();
  if (hybrid_ && !commits.empty()) {
    const CommitRec* d_rec = hb->put(commits.data(), commits.size(), stream_, &hyb_ok);
    if (hyb_ok) {
      launch_hybrid_commit(d_rec, (int)commits.size(), hb->dFinal, hb->dSpecPos, dFpos_, dFgen_, dFidp_, stream_);
      ++launches_;
    }
  }
  if (!hyb_ok) { ok_ = false; err_ = "hybrid bookkeeping failed (upload arena / anchor outside the window)"; return ORCVIO_ERR_CUDA; }
  cudaEvent_t* e = ev_;
  g_sp.mark(6);
  run_phase(wA, 0);
  std::vector<Track*> gather_tracks;
  if (hybrid_) {
    for (int fi = 0; fi < B_; ++fi) {       // the features whose host mirror the prune phase may need
      FilterHost& F = f_[fi];
      F.ekf_watch.clear();
      if (!F.active) continue;
      F.ekf_watch = F.feature_states;
      for (Track* trp : news[fi]) F.ekf_watch.push_back(trp->id);
    }
    hybrid_queue_gather(gather_tracks);
    if (!wA.hfeats.empty()) {
      CK(cudaMemcpyAsync(hb->hEkfPass, hb->dEkfPass, wA.hfeats.size() * sizeof(int), cudaMemcpyDeviceToHost, stream_));
      CK(cudaMemcpyAsync(hb->hEkfGamma, hb->dEkfGamma, wA.hfeats.size() * sizeof(double), cudaMemcpyDeviceToHost, stream_));
    }
  }
  download_mirrors();
  g_sp.mark(7);
  wait_stream();
  g_sp.mark(8);
  if (hybrid_) {
    hybrid_apply_gather(gather_tracks);
    hb->used = 0;
  }
  auto account = [&](bool had_update) {
    if (!profiling_) return;
    float ms = 0;
    cudaEventElapsedTime(&ms, e[0], e[1]); pt_.tri += ms; pt_.n_tri++;
    cudaEventElapsedTime(&ms, e[1], e[2]); pt_.jac += ms; pt_.n_jac++;
    if (had_update) {
      cudaEventElapsedTime(&ms, e[2], e[3]); pt_.qr_tiles += ms; pt_.n_qr_tiles++;
      cudaEventElapsedTime(&ms, e[3], e[4]); pt_.qr_chain += ms; pt_.n_qr_chain++;
      cudaEventElapsedTime(&ms, e[4], e[5]); pt_.update += ms; pt_.n_update++;
    }
  };
  account(wA.any_active);

  // ---------------------------------------------------------------- E: post-process A, prune
  PhaseWork wB;
  wB.fw.assign(B_, FilterWork{});
  wB.cand_begin.assign(B_ + 1, 0);
  if (hybrid_) { wB.hyb_phase = 1; wB.hw.assign(B_, HybWork{}); }
  std::vector<int> rm_idx(2 * (size_t)B_, -1), Nbefore(B_, 0), Ebefore(B_, 0);
  std::vector<ReanchorRec> reanchor;
  std::vector<int> reanchor_off(B_ + 1, 0);
  // pruneImuStateBuffer :2665-2773: an EKF-SLAM feature (of the state, or initialised and waiting outside it) whose anchor
  // clone is about to leave the window moves to a new anchor (getNewAnchorId :3892-3950) before anything else happens
  auto reanchor_tracks = [&](int fi, FilterHost& F, const long long* rm_ids, int n_rm) {
    if (F.ekf_watch.empty()) return;
    std::vector<long long> ids = F.ekf_watch;
    std::sort(ids.begin(), ids.end());
    auto removed = [&](long long sid) {
      for (int q = 0; q < n_rm; ++q) if (rm_ids[q] == sid) return true;
      return false;
    };
    for (long long id : ids) {
      Track* trp = F.find_track(id);
      if (!trp) continue;
      Track& tr = *trp;
      if (!tr.ekf_feature || !tr.initialized || !removed(tr.id_anchor)) continue;
      bool anchor_observed = false;
      for (const Obs& o : tr.obs) anchor_observed |= (o.sid == tr.id_anchor);
      if (!anchor_observed) continue;                   // `involved` holds only clones the feature was seen from
      // getNewAnchorId: the observing clone (the two newest and the removed ones excluded) whose stored observation is
      // closest to the reprojection of the feature; the newest clone when there is none
      const int n = (int)F.clones.size();
      long long new_id = F.clones.back().id;
      if (n > 2) {
        double min_dis = 99999.0;
        long long best = -1;
        for (int k = 0; k < n - 2; ++k) {
          const long long sid = F.clones[k].id;
          if (removed(sid)) continue;
          const Obs* ob = nullptr;
          for (const Obs& o : tr.obs) if (o.sid == sid) ob = &o;
          if (!ob) continue;
          const double* c = F.clone_mirror.data() + (size_t)k * CL_STRIDE;
          const double d[3] = {tr.mpos[0] - c[CL_PC], tr.mpos[1] - c[CL_PC + 1], tr.mpos[2] - c[CL_PC + 2]};
          double pn[3];
          m3_inv_vec(c + CL_RC, d, pn);
          const double du = pn[0] / pn[2] - ob->z[0], dv = pn[1] / pn[2] - ob->z[1];
          const double dis = std::sqrt(du * du + dv * dv);
          if (min_dis > dis) { min_dis = dis; best = sid; }
        }
        if (best >= 0) new_id = best;
      }
      ReanchorRec rc{};
      rc.filter = fi;
      rc.slot = tr.slot;
      rc.col = -1;
      if (tr.in_state)
        for (int i = 0; i < (int)F.feature_states.size(); ++i)
          if (F.feature_states[i] == id) rc.col = i;
      rc.old_idx = clone_index_of(F, tr.id_anchor);
      rc.new_idx = clone_index_of(F, new_id);
      if (!tr.in_state) {
        // :2762-2764: obs_anchor <- the stored observation in the new anchor (operator[] default-constructs it)
        const Obs* ob = nullptr;
        for (const Obs& o : tr.obs) if (o.sid == new_id) ob = &o;
        if (!ob) {
          Obs z{};
          z.sid = new_id;
          auto pos = std::lower_bound(tr.obs.begin(), tr.obs.end(), new_id,
                                      [](const Obs& o, long long sid) { return o.sid < sid; });
          ob = &*tr.obs.insert(pos, z);
          tr.touch();
        }
        rc.zu = ob->z[0];
        rc.zv = ob->z[1];
      } else {
        F.log_reanchor.push_back(id);
        F.log_reanchor.push_back(tr.id_anchor);
        F.log_reanchor.push_back(new_id);
      }
      tr.id_anchor = new_id;
      reanchor.push_back(rc);
    }
  };
  for (int fi = 0; fi < B_; ++fi) {
    FilterHost& F = f_[fi];
    wB.cand_begin[fi] = (int)wB.cands.size();
    reanchor_off[fi] = (int)reanchor.size();
    FilterWork& fw = wB.fw[fi];
    fw.N = (int)F.clones.size();
    fw.D = L + 6 * fw.N + (int)F.feature_states.size();
    fw.active = 0;
    Nbefore[fi] = fw.N;
    if (!F.active) { Ebefore[fi] = (int)F.feature_states.size(); continue; }
    std::memcpy(F.imu_mirror.data(), hImu_ + (size_t)fi * IM_STRIDE, IM_STRIDE * sizeof(double));
    std::memcpy(F.clone_mirror.data(), hClones_ + (size_t)fi * Ncap_ * CL_STRIDE,
                (size_t)Ncap_ * CL_STRIDE * sizeof(double));
    // results of phase A
    const int c0 = wA.cand_begin[fi], c1 = wA.cand_begin[fi + 1];
    for (int c = c0; c < c1; ++c) {
      const int st = hStatus_[c];
      const CandInfo& ci = F.cinfo[0][c - c0];
      F.cstatus[0].push_back(st);
      F.cgamma[0].push_back(hGamma_[c]);
      if (ci.kind == 3) {
        // candidate EKF-SLAM feature: in the state iff its MSCKF rows passed the gate (:2371-2411); a rejected one
        // keeps its inverse-depth record and waits outside the state
        const bool pass = (st & ST_GATE_PASS) != 0;
        F.log_new_ids.push_back(ci.id);
        F.log_new_ok.push_back(pass ? 1 : 0);
        F.log_new_gamma.push_back(hGamma_[c]);
        if (pass) {
          F.find_track(ci.id)->in_state = true;
          F.feature_states.push_back(ci.id);
          ++feature_updates_;
        }
        continue;
      }
      if (!(st & ST_TRI_VALID)) F.stats.n_tri_invalid_lost++;
      if (st & ST_GATE_PASS) { F.stats.n_gate_pass_lost++; ++feature_updates_; }
      // lost features are always erased (:2572-2576); tracked-long ones only when they were
      // initialised and therefore used (:2310-2319)
      if (ci.kind == 0 || (st & ST_TRI_VALID)) {
        if (Track* gone = F.find_track(ci.id)) {
          F.free_slots.push_back(gone->slot);
          F.erase_track(ci.id);
        }
      }
    }
    if (hybrid_ && wA.hw[fi].active) {
      const HybWork& hw = wA.hw[fi];
      for (int i = 0; i < hw.E; ++i) {
        F.log_ekf_ids.push_back(F.feature_states[i]);
        F.log_ekf_pass.push_back(hb->hEkfPass[hw.feat_begin + i]);
        F.log_ekf_gamma.push_back(hb->hEkfGamma[hw.feat_begin + i]);
        if (hb->hEkfPass[hw.feat_begin + i]) ++feature_updates_;
      }
    }
    fw.D = L + 6 * fw.N + (int)F.feature_states.size();
    Ebefore[fi] = (int)F.feature_states.size();
    wB.maxE = std::max(wB.maxE, Ebefore[fi]);
    auto fill_hw = [&]() {              // features of the state with their (possibly new) anchors
      if (!hybrid_) return;
      HybWork& hw = wB.hw[fi];
      hw.N = fw.N; hw.E = Ebefore[fi]; hw.active = fw.active;
      hw.feat_begin = (int)wB.hfeats.size();
      for (long long id : F.feature_states) {
        const Track& tr = *F.find_track(id);
        HybFeat hf{};
        hf.slot = tr.slot;
        hf.anchor = clone_index_of(F, tr.id_anchor);
        if (hf.anchor < 0) { hyb_ok = false; hf.anchor = 0; }
        wB.hfeats.push_back(hf);
      }
      hw.feat_end = (int)wB.hfeats.size();
      hw.new_begin = hw.new_end = 0;
    };
    // pruneImuStateBuffer :2629-2959
    if (F.if_zupt) {
      // :2633-2639: a stationary frame drops the previous clone (id - 1) and uses nothing
      const int n = (int)F.clones.size();
      if (n < 2) { fill_hw(); continue; }
      rm_idx[2 * fi] = n - 2;
      const long long rm_id = F.clones[n - 2].id;
      F.stats.n_removed_clones = 1;
      F.stats.removed_ids[0] = rm_id;
      if (hybrid_) reanchor_tracks(fi, F, &rm_id, 1);
      for (auto& kv : F.map_server) {
        Track& tr = kv.second;
        if (tr.first_sid > rm_id || tr.last_sid < rm_id) continue;     // (ascending ids: it cannot hold the clone)
        tr.obs.erase(std::remove_if(tr.obs.begin(), tr.obs.end(), [&](const Obs& o) { return o.sid == rm_id; }),
                     tr.obs.end());
        tr.touch();
      }
      fill_hw();
      continue;
    }
    if ((int)F.clones.size() < p_.sw_size) { fill_hw(); continue; }
    wB.maxN = std::max(wB.maxN, fw.N);
    // findRedundantImuStates :2582-2626
    const int n = (int)F.clones.size();
    int key_i = n - 4, st_i = key_i + 1, first_i = 0;
    const double* key = F.clone_mirror.data() + (size_t)key_i * CL_STRIDE;
    int rm[2];
    for (int r = 0; r < 2; ++r) {
      const double* c = F.clone_mirror.data() + (size_t)st_i * CL_STRIDE;
      const double dx = c[CL_PC] - key[CL_PC], dy = c[CL_PC + 1] - key[CL_PC + 1], dz = c[CL_PC + 2] - key[CL_PC + 2];
      const double distance = std::sqrt((dx * dx + dy * dy) + dz * dz);
      double Rr[9];
      m3_Tmul(c + CL_RC, key + CL_RC, Rr);      // rotation = R_cam^T ; rotation * key_rotation
      const double angle = angle_axis_angle(Rr);
      if (angle < p_.rotation_threshold && distance < p_.translation_threshold &&
          F.tracking_rate > p_.tracking_rate_threshold) {
        rm[r] = st_i;
        ++st_i;
      } else {
        rm[r] = first_i;
        ++first_i;
        st_i -= 2;
      }
    }
    if (rm[0] > rm[1]) std::swap(rm[0], rm[1]);
    rm_idx[2 * fi] = rm[0];
    rm_idx[2 * fi + 1] = rm[1];
    const long long rm_id0 = F.clones[rm[0]].id, rm_id1 = F.clones[rm[1]].id;
    F.stats.n_removed_clones = 2;
    F.stats.removed_ids[0] = rm_id0;
    F.stats.removed_ids[1] = rm_id1;
    const long long cur = F.state_id;
    if (hybrid_) {
      const long long rms[2] = {rm_id0, rm_id1};
      reanchor_tracks(fi, F, rms, 2);
    }
    std::vector<CandBuild> cb;
    auto clone_index = [&](long long sid) { return clone_index_of(F, sid); };
    for (auto& kv : F.map_server) {
      Track& tr = kv.second;
      if (tr.first_sid > rm_id1 || tr.last_sid < rm_id0) continue;     // (rm_id0 < rm_id1: neither clone observed it)
      int inv0 = -1, inv1 = -1;
      for (int k = 0; k < (int)tr.obs.size(); ++k) {
        if (tr.obs[k].sid == rm_id0) inv0 = k;
        if (tr.obs[k].sid == rm_id1) inv1 = k;
      }
      if (inv0 < 0 && inv1 < 0) continue;
      // (:2776: EKF-SLAM features never contribute MSCKF rows here)
      if (inv0 >= 0 && inv1 >= 0 && !tr.in_state && !tr.ekf_feature) {
        const int nobs = (int)tr.obs.size();
        const bool tracked = tr.obs.back().sid == cur;
        CandBuild x{};
        x.id = tr.id;
        x.kind = 2;
        Cand& c = x.c;
        c.slot = tr.slot;
        c.gen = tr.gen;
        c.flags = 0;
        c.tri_off = (int)wB.obs_clone.size();
        for (const Obs& o : tr.obs) {            // initializePosition_AssignAnchor: all obs
          wB.obs_clone.push_back(clone_index(o.sid));
          wB.obs_z.push_back(o.z[0]);
          wB.obs_z.push_back(o.z[1]);
        }
        c.tri_m = nobs;
        c.jac_off = (int)wB.obs_clone.size();
        const int ks[2] = {inv0, inv1};
        for (int q = 0; q < 2; ++q) {
          wB.obs_clone.push_back(clone_index(tr.obs[ks[q]].sid));
          wB.obs_z.push_back(tr.obs[ks[q]].z[0]);
          wB.obs_z.push_back(tr.obs[ks[q]].z[1]);
        }
        c.jac_m = 2;
        c.s_blk = rm[0];
        c.e_blk = rm[1];
        c.cm_first_clone = wB.obs_clone[c.tri_off];
        c.cm_last_clone = wB.obs_clone[c.tri_off + (tracked ? nobs - 2 : nobs - 1)];
        c.cm_zu = tr.obs[0].z[0];
        c.cm_zv = tr.obs[0].z[1];
        cb.push_back(x);
      }
      // erase the observations of the removed clones (:2842-2844)
      tr.obs.erase(std::remove_if(tr.obs.begin(), tr.obs.end(),
                                  [&](const Obs& o) { return o.sid == rm_id0 || o.sid == rm_id1; }),
                   tr.obs.end());
      tr.touch();
    }
    F.stats.n_candidates_prune = (int)cb.size();
    if (!cb.empty()) {
      fw.active = 1;
      wB.any_active = true;
      append_candidates(wB, fi, cb, F.cinfo[1]);
    }
    fill_hw();
  }
  wB.cand_begin[B_] = (int)wB.cands.size();
  reanchor_off[B_] = (int)reanchor.size();
  wB.extra_ints = rm_idx;
  wB.extra_ints.insert(wB.extra_ints.end(), Nbefore.begin(), Nbefore.end());
  wB.extra_ints.insert(wB.extra_ints.end(), Ebefore.begin(), Ebefore.end());
  if (!hyb_ok) { ok_ = false; err_ = "hybrid bookkeeping failed (anchor outside the window)"; return ORCVIO_ERR_CUDA; }
  g_sp.mark(9);
  stage_phase(wB);
  if (hybrid_ && !reanchor.empty()) {
    const ReanchorRec* d_rec = hb->put(reanchor.data(), reanchor.size(), stream_, &hyb_ok);
    const int* d_off = hb->put(reanchor_off.data(), reanchor_off.size(), stream_, &hyb_ok);
    if (hyb_ok) {
      launch_reanchor(d_rec, d_off, B_, wB.dHw, dClones_, (size_t)Ncap_ * CL_STRIDE, dImu_, dFpos_, dFidp_, Fcap_, dP_,
                      (size_t)ldp_ * ldp_, ldp_, stream_);
      ++launches_;
    }
  }
  launch_phase(wB, true);
  // remove the pruned clones from P / clone array (:2875-2956)
  bool any_rm = false;
  for (int v : rm_idx) any_rm |= (v >= 0);
  if (any_rm) {
    RemoveArgs ra{};
    ra.P = dP_; ra.p_stride = (size_t)ldp_ * ldp_; ra.ldp = ldp_;
    ra.clones = dClones_; ra.clone_stride = (size_t)Ncap_ * CL_STRIDE;
    ra.rm = wB.d_extra; ra.N = wB.d_extra + 2 * B_; ra.n_filters = B_;
    ra.E = hybrid_ ? wB.d_extra + 3 * B_ : nullptr;
    launch_remove(ra, stream_);
    ++launches_;
  }
  if (hybrid_) hybrid_queue_gather(gather_tracks);
  download_mirrors();
  g_sp.mark(10);
  wait_stream();
  if (hybrid_) {
    hybrid_apply_gather(gather_tracks);
    if (!hyb_ok) { ok_ = false; err_ = "hybrid upload arena exhausted"; }
  }
  account(wB.any_active);
  for (int fi = 0; fi < B_; ++fi) {
    FilterHost& F = f_[fi];
    if (!F.active) continue;
    const int c0 = wB.cand_begin[fi], c1 = wB.cand_begin[fi + 1];
    for (int c = c0; c < c1; ++c) {
      const int st = hStatus_[c];
      F.cstatus[1].push_back(st);
      F.cgamma[1].push_back(hGamma_[c]);
      if (!(st & ST_TRI_VALID)) F.stats.n_tri_invalid_prune++;
      if (st & ST_GATE_PASS) { F.stats.n_gate_pass_prune++; ++feature_updates_; }
    }
    if (rm_idx[2 * fi] >= 0) {
      const int a = rm_idx[2 * fi], b = rm_idx[2 * fi + 1];
      const double ta = F.clones[a].time, tb = b >= 0 ? F.clones[b].time : ta;
      F.cur_window_timestamps.erase(
          std::remove_if(F.cur_window_timestamps.begin(), F.cur_window_timestamps.end(),
                         [&](double t) { return t == ta || t == tb; }),
          F.cur_window_timestamps.end());
      if (b >= 0) F.clones.erase(F.clones.begin() + b);
      F.clones.erase(F.clones.begin() + a);
    }
    std::memcpy(F.imu_mirror.data(), hImu_ + (size_t)fi * IM_STRIDE, IM_STRIDE * sizeof(double));
    std::memcpy(F.clone_mirror.data(), hClones_ + (size_t)fi * Ncap_ * CL_STRIDE,
                (size_t)Ncap_ * CL_STRIDE * sizeof(double));
  }
  g_sp.mark(11);
  g_sp.done(B_);
  return ok_ ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

void Batch::hybrid_queue_gather(std::vector<Track*>& tracks) {
  tracks.clear();
  HybridBufs& hb = *hyb_;
  std::vector<int> filt, slots;
  for (int fi = 0; fi < B_; ++fi) {
    FilterHost& F = f_[fi];
    if (!F.active) continue;
    for (long long id : F.ekf_watch) {
      auto it = F.map_server.find(id);
      if (it == F.map_server.end()) continue;
      tracks.push_back(&it->second);
      filt.push_back(fi);
      slots.push_back(it->second.slot);
    }
  }
  const size_t n = tracks.size();
  if (n == 0) return;
  if (n > hb.gather_cap) {             // (the previous gather was consumed behind a synchronisation)
    cudaFree(hb.dGather);
    cudaFreeHost(hb.hGather);
    hb.gather_cap = n * 2;
    note_growth("hybrid gather (device + pinned)", hb.gather_cap * 6 * sizeof(double));
    CK(cudaMalloc(&hb.dGather, hb.gather_cap * 6 * sizeof(double)));
    CK(cudaMallocHost(&hb.hGather, hb.gather_cap * 6 * sizeof(double)));
  }
  bool okp = true;
  const int* d_f = hb.put(filt.data(), n, stream_, &okp);
  const int* d_s = hb.put(slots.data(), n, stream_, &okp);
  if (!okp) { ok_ = false; err_ = "hybrid upload arena exhausted"; tracks.clear(); return; }
  launch_hybrid_gather(d_f, d_s, (int)n, dFpos_, dFidp_, Fcap_, hb.dGather, stream_);
  ++launches_;
  CK(cudaMemcpyAsync(hb.hGather, hb.dGather, n * 6 * sizeof(double), cudaMemcpyDeviceToHost, stream_));
}

void Batch::hybrid_apply_gather(const std::vector<Track*>& tracks) {
  const double* g = hyb_->hGather;
  for (size_t k = 0; k < tracks.size(); ++k) {
    Track& tr = *tracks[k];
    for (int q = 0; q < 3; ++q) tr.mpos[q] = g[6 * k + q];
    tr.minv = g[6 * k + 3];
    tr.mobs[0] = g[6 * k + 4];
    tr.mobs[1] = g[6 * k + 5];
  }
}

int Batch::get_feature_states(int i, long long* ids, long long* anchors, double* inv_depth, double* obs_anchor,
                              double* xyz, int cap) {
  if (i < 0 || i >= B_) return ORCVIO_ERR_ARG;
  FilterHost& F = f_[i];
  int n = 0;
  for (long long id : F.feature_states) {
    if (n >= cap) break;
    const Track& tr = F.map_server.at(id);
    if (ids) ids[n] = id;
    if (anchors) anchors[n] = tr.id_anchor;
    if (inv_depth) inv_depth[n] = tr.minv;
    if (obs_anchor) { obs_anchor[2 * n] = tr.mobs[0]; obs_anchor[2 * n + 1] = tr.mobs[1]; }
    if (xyz) for (int q = 0; q < 3; ++q) xyz[3 * n + q] = tr.mpos[q];
    ++n;
  }
  return n;
}

int Batch::get_state(int i, OrcvioState* out) {
  if (i < 0 || i >= B_) return ORCVIO_ERR_ARG;
  FilterHost& F = f_[i];
  std::memset(out, 0, sizeof(*out));
  out->state_id = F.state_id;
  const double* im = F.imu_mirror.data();
  out->time = F.imu_time;
  for (int k = 0; k < 9; ++k) out->R[k] = im[IM_R + k];
  for (int k = 0; k < 3; ++k) {
    out->p[k] = im[IM_P + k];
    out->v[k] = im[IM_V + k];
    out->bg[k] = im[IM_BG + k];
    out->ba[k] = im[IM_BA + k];
  }
  out->n_clones = (int)F.clones.size();
  out->dim = ORCVIO_LEG + 6 * out->n_clones + (int)F.feature_states.size();
  out->n_map_features = (int)F.map_server.size();
  double c9[81];
  CK(cudaMemcpy2D(c9, 9 * sizeof(double), dP_ + (size_t)i * ldp_ * ldp_, ldp_ * sizeof(double),
                  9 * sizeof(double), 9, cudaMemcpyDeviceToHost));
  // getPpose :3000-3015: [[P_pp, P_po],[P_op, P_oo]]
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 3; ++b) {
      out->P_pose[6 * a + b] = c9[9 * (6 + a) + 6 + b];
      out->P_pose[6 * a + 3 + b] = c9[9 * (6 + a) + b];
      out->P_pose[6 * (3 + a) + b] = c9[9 * a + 6 + b];
      out->P_pose[6 * (3 + a) + 3 + b] = c9[9 * a + b];
      out->P_vel[3 * a + b] = c9[9 * (3 + a) + 3 + b];
    }
  return ORCVIO_OK;
}

int Batch::get_cov(int i, double* P, int cap, int* D) {
  if (i < 0 || i >= B_) return ORCVIO_ERR_ARG;
  const int d = ORCVIO_LEG + 6 * (int)f_[i].clones.size() + (int)f_[i].feature_states.size();
  if (D) *D = d;
  if (!P) return ORCVIO_OK;
  if (cap < d * d) return ORCVIO_ERR_ARG;
  // device is row-major with ld; P is symmetric so the column-major view is identical
  CK(cudaMemcpy2D(P, d * sizeof(double), dP_ + (size_t)i * ldp_ * ldp_, ldp_ * sizeof(double),
                  d * sizeof(double), d, cudaMemcpyDeviceToHost));
  return ORCVIO_OK;
}

int Batch::get_map_points(int i, long long* ids, double* xyz, int cap) {
  if (i < 0 || i >= B_) return ORCVIO_ERR_ARG;
  FilterHost& F = f_[i];
  std::vector<double> fp((size_t)Fcap_ * FP_STRIDE);
  std::vector<long long> fg(Fcap_);
  CK(cudaMemcpy(fp.data(), dFpos_ + (size_t)i * Fcap_ * FP_STRIDE, fp.size() * sizeof(double), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(fg.data(), dFgen_ + (size_t)i * Fcap_, fg.size() * sizeof(long long), cudaMemcpyDeviceToHost));
  int n = 0;
  for (auto& kv : F.map_server) {
    if (n >= cap) break;
    const Track& tr = kv.second;
    if (ids) ids[n] = tr.id;
    if (xyz) {
      const bool init = fg[tr.slot] == tr.gen;
      for (int k = 0; k < 3; ++k) xyz[3 * n + k] = init ? fp[(size_t)tr.slot * FP_STRIDE + k] : NAN;
    }
    ++n;
  }
  return n;
}

int Batch::set_cov(int i, const double* P, int D) {
  if (i < 0 || i >= B_ || D > ldp_ || !P) return ORCVIO_ERR_ARG;
  {
    // the update path only uses the window columns of H: that equals the reference as long as the extrinsic / time-offset
    // block of P (rows / columns 15..21) is zero (estimate_extrin = estimate_td = 0), so a covariance that breaks it is
    // refused instead of silently diverging; D must be the filter's current dimension (or the setStateCov override)
    const FilterHost& F = f_[i];
    const int d_now = ORCVIO_LEG + 6 * (int)F.clones.size() + (int)F.feature_states.size();
    const int d_ovr = (F.leg_dim_override >= 0 && F.num_clone_override >= 0) ? F.leg_dim_override + 6 * F.num_clone_override : -1;
    if (D != d_now && D != d_ovr) return ORCVIO_ERR_ARG;
    if (D == d_now && D != d_ovr)            // (the setStateCov hook re-defines the layout: LEG_DIM may be 15 there)
      for (int r = 15; r < ORCVIO_LEG; ++r)
        for (int c = 0; c < D; ++c)
          if (P[(size_t)r * D + c] != 0.0 || P[(size_t)c * D + r] != 0.0) return ORCVIO_ERR_ARG;
  }
  CK(cudaMemcpy2D(dP_ + (size_t)i * ldp_ * ldp_, ldp_ * sizeof(double), P, D * sizeof(double),
                  D * sizeof(double), D, cudaMemcpyHostToDevice));
  return ORCVIO_OK;
}


void Batch::override_noise(double sigma2, double chi2_p) {
  p_.feature_observation_noise = sigma2;
  if (chi2_p != p_.chi_square_threshold_feat) {
    p_.chi_square_threshold_feat = chi2_p;
    for (int i = 1; i < 500; ++i) chi2_host_[i] = chi2_quantile(chi2_p, i);
    CK(cudaMemcpy(dChi2_, chi2_host_.data(), 500 * sizeof(double), cudaMemcpyHostToDevice));
  }
}

// ---------------------------------------------------------------------------------------
// Frozen-window entry ("stack -> compress -> update" on one frame, SURVEY 8d).
// prepare: host staging of the window + work lists, one upload;  execute: restore the
// pristine window (D2D) and run the kernel chain;  fetch: results back to host buffers.
struct Batch::SnapState {
  PhaseWork w;
  std::vector<int> order;          // candidate order after sorting -> caller's feature index
  std::vector<int> sblk, eblk;     // first / last clone block per feature
  int N = 0, D = 0, n_feat = 0, nobs_total = 0;
  bool has_positions = false;
  double *dP0 = nullptr, *dCl0 = nullptr, *dIm0 = nullptr, *dPos0 = nullptr;   // pristine window
  long long* dGen0 = nullptr;
  size_t pos_cap = 0;
  double *hP0 = nullptr, *hCl0 = nullptr, *hIm0 = nullptr;                      // pinned staging
  double* hOut = nullptr;          // pinned download buffer (P, dx, clones)
  size_t hout_cap = 0;
  FilterWork* hFw = nullptr; FilterWork* dFw = nullptr;   // (N, D) record for the early prior launch
  bool prior_early = false;
  bool tri_early = false;          // k_triangulate (direct mode) already queued by snapshot_prepare
  std::vector<int> rowoff_f, hblkoff_f, small_f, large_f;   // per feature (caller's order): offsets, size classes
  bool jac_early = false;          // k_jac_gate (direct mode) already queued by snapshot_prepare
  bool by_feature = false;         // status / gamma of the last run are indexed by feature, not by candidate
  int list_err = 0;                // result of the (possibly threaded) work-list build
  std::atomic<int> scan_done{0}, lists_done{0};
  // CUDA graph of one resident-frame run (restore + kernel chain on both streams), replayed by snapshot_execute
  cudaGraphExec_t graph_exec = nullptr;
  int graph_launches = 0;          // kernels inside the graph
  int plain_runs = 0;              // uncaptured runs since the last prepare (the first ones grow the scratch buffers)
  void drop_graph() {
    if (graph_exec) cudaGraphExecDestroy(graph_exec);
    graph_exec = nullptr;
    plain_runs = 0;
  }
  ~SnapState() {
    drop_graph();
    cudaFree(dFw);
    if (hFw) cudaFreeHost(hFw);
    cudaFree(dP0); cudaFree(dCl0); cudaFree(dIm0); cudaFree(dPos0); cudaFree(dGen0);
    if (hP0) cudaFreeHost(hP0);
    if (hCl0) cudaFreeHost(hCl0);
    if (hIm0) cudaFreeHost(hIm0);
    if (hOut) cudaFreeHost(hOut);
  }
};

void Batch::SnapDeleter::operator()(SnapState* p) const { delete p; }

int Batch::snapshot_prepare(const SnapshotIO& io) {
  if (!ok_) return ORCVIO_ERR_NO_DEVICE;
  const int N = io.n_clones;
  if (N < 1 || N > Ncap_ || io.n_feat < 0) return ORCVIO_ERR_ARG;
  if (!snap_) {
    snap_.reset(new SnapState());
    SnapState& S = *snap_;
    CK(cudaMalloc(&S.dP0, (size_t)ldp_ * ldp_ * sizeof(double)));
    CK(cudaMalloc(&S.dCl0, (size_t)Ncap_ * CL_STRIDE * sizeof(double)));
    CK(cudaMalloc(&S.dIm0, IM_STRIDE * sizeof(double)));
    CK(cudaMallocHost(&S.hP0, (size_t)ldp_ * ldp_ * sizeof(double)));
    CK(cudaMallocHost(&S.hCl0, (size_t)Ncap_ * CL_STRIDE * sizeof(double)));
    CK(cudaMallocHost(&S.hIm0, IM_STRIDE * sizeof(double)));
    S.hout_cap = (size_t)ldp_ * ldp_ + ldp_ + (size_t)Ncap_ * CL_STRIDE;
    CK(cudaMallocHost(&S.hOut, S.hout_cap * sizeof(double)));
    CK(cudaMallocHost(&S.hFw, sizeof(FilterWork)));
    CK(cudaMalloc(&S.dFw, sizeof(FilterWork)));
  }
  SnapState& S = *snap_;
  S.drop_graph();                  // new work lists: the captured chain no longer matches
  g_hp.start();
  if (io.n_feat > Fcap_) {
    // grow the feature tables of this (single filter) batch
    CK(cudaStreamSynchronize(stream_));
    cudaFree(dFpos_); cudaFree(dFgen_);
    Fcap_ = io.n_feat + 1024;
    CK(cudaMalloc(&dFpos_, (size_t)B_ * Fcap_ * FP_STRIDE * sizeof(double)));
    CK(cudaMalloc(&dFgen_, (size_t)B_ * Fcap_ * sizeof(long long)));
  }
  const int D = ORCVIO_LEG + 6 * N;
  S.N = N; S.D = D; S.n_feat = io.n_feat;
  // the staging buffers may still be read by the previous call's async copies
  CK(cudaStreamSynchronize(stream_));
  g_hp.mark("sync");
  PhaseWork& w = S.w;
  w.reset();
  w.fw.assign(B_, FilterWork{});
  w.cand_begin.assign(B_ + 1, 0);
  FilterWork& fw = w.fw[0];
  fw.N = N; fw.D = D; fw.active = (io.stages & 4) ? 1 : 0;
  w.any_active = fw.active;
  w.maxN = N;
  // observations are referenced in place and copied once, straight into the pinned upload blob
  const int nF = io.n_feat;
  const int nobs_total = io.feat_off[nF];
  if (nobs_total < 0 || io.feat_off[0] != 0) return ORCVIO_ERR_ARG;
  S.nobs_total = nobs_total;
  w.ext_obs_clone = io.obs_clone; w.ext_obs_z = io.obs_z; w.ext_nobs = (size_t)nobs_total;
  // candidates sorted by first clone block, then feature index: a counting sort (what
  // append_candidates' stable sort produces, without the comparison sort)
  // The work lists (validation, counting sort, candidate records, tiles) are pure host work on the caller's
  // arrays: in the end-to-end call a helper thread builds them while this thread stages P, starts the prior
  // factor, uploads the observation pools and starts the early triangulation.
  const bool early_tri = io.early_prior && (io.stages & 1) && (io.stages & 2) && !io.positions_in && !io.iters &&
                         !io.cost && nF > 0;
  w.obs_preuploaded = early_tri;
  blob_.ensure_pinned(4096 + (size_t)std::max(nF, 1) * (sizeof(Cand) + sizeof(Tile) + 2 * sizeof(int)) +
                      sizeof(FilterWork) * B_ + (early_tri ? 0 : (size_t)nobs_total * 20));
  S.list_err = ORCVIO_OK;
  S.scan_done.store(0, std::memory_order_relaxed);
  S.lists_done.store(0, std::memory_order_relaxed);
  auto build_lists = [this, &S, &w, io, nF, N]() {
    int* err = &S.list_err;
    int bucket[ORCVIO_MAX_OBS + 2] = {0};
    auto scan = [&]() {
      S.sblk.resize(nF);
      S.eblk.resize(nF);
      S.rowoff_f.resize(nF);
      S.hblkoff_f.resize(nF);
      S.small_f.clear();
      S.large_f.clear();
      for (int f = 0; f < nF; ++f) {
        const int o0 = io.feat_off[f], m = io.feat_off[f + 1] - o0;
        if (m < 1 || m > ORCVIO_MAX_OBS) { *err = ORCVIO_ERR_ARG; return; }
        int s = 1 << 30, e = -1;
        for (int k = 0; k < m; ++k) {
          const int ci = io.obs_clone[o0 + k];
          if (ci < 0 || ci >= N) { *err = ORCVIO_ERR_ARG; return; }
          s = std::min(s, ci);
          e = std::max(e, ci);
        }
        S.sblk[f] = s; S.eblk[f] = e;
        ++bucket[s + 1];
        // rows / compact block of the feature, placed in the caller's feature order (any placement works: the
        // candidate records carry the offsets)
        const int r = std::max(2 * m - 3, 0), wb = e - s + 1;
        S.rowoff_f[f] = (int)w.rows_total;
        S.hblkoff_f[f] = (int)w.hblk_total;
        w.rows_total += (size_t)r;
        w.hblk_total += (size_t)r * 6 * wb;
        w.own_wmax_blk = std::max(w.own_wmax_blk, wb);
        if (m <= 8) S.small_f.push_back(f);
        else S.large_f.push_back(f);
      }
    };
    scan();
    S.scan_done.store(1, std::memory_order_release);
    if (*err == ORCVIO_OK) {
      for (int k = 1; k <= ORCVIO_MAX_OBS + 1; ++k) bucket[k] += bucket[k - 1];
      S.order.resize(nF);
      for (int f = 0; f < nF; ++f) S.order[bucket[S.sblk[f]]++] = f;
      w.cands.resize(nF);
      for (int pos = 0; pos < nF; ++pos) {
        const int f = S.order[pos];
        const int o0 = io.feat_off[f], m = io.feat_off[f + 1] - o0;
        Cand& c = w.cands[pos];
        c.filter = 0;
        c.slot = f;
        c.gen = f + 1;
        c.flags = CAND_FORCE_TRI;
        c.tri_off = c.jac_off = o0;
        c.tri_m = c.jac_m = m;
        c.s_blk = S.sblk[f]; c.e_blk = S.eblk[f];
        c.cm_first_clone = io.obs_clone[o0];
        c.cm_last_clone = io.obs_clone[o0 + m - 1];
        c.cm_zu = io.obs_z[2 * (size_t)o0];
        c.cm_zv = io.obs_z[2 * (size_t)o0 + 1];
        c.row_off = S.rowoff_f[f];
        c.hblk_off = S.hblkoff_f[f];
        if (m <= 8) w.small_list.push_back(pos);
        else w.large_list.push_back(pos);
      }
      build_tiles(w, 0, 0, nF);
    }
    S.lists_done.store(1, std::memory_order_release);
  };
  const bool threaded = io.early_prior && nF >= 512;
  if (threaded) {
    if (!worker_) worker_.reset(new HostWorker());
    worker_->run(build_lists);
  } else {
    build_lists();
  }
  auto wait_flag = [](std::atomic<int>& f) {
    while (!f.load(std::memory_order_acquire)) std::this_thread::yield();
  };
  // the caller's observation pools go up first, as they are (nothing has to be sorted for that): by the time the
  // inputs are validated and the prior factor is started, they are on the device and the early triangulation /
  // Jacobian pass can start at once
  size_t e_fo = 0, e_oc = 0, e_oz = 0;
  if (early_tri) {
    blob_early_.reset();
    e_fo = blob_early_.reserve(sizeof(int) * (size_t)(nF + 1));
    e_oc = blob_early_.reserve(sizeof(int) * (size_t)nobs_total);
    e_oz = blob_early_.reserve(sizeof(double) * 2 * (size_t)nobs_total);
    std::memcpy(blob_early_.pinned + e_fo, io.feat_off, sizeof(int) * (size_t)(nF + 1));
    std::memcpy(blob_early_.pinned + e_oc, io.obs_clone, sizeof(int) * (size_t)nobs_total);
    std::memcpy(blob_early_.pinned + e_oz, io.obs_z, sizeof(double) * 2 * (size_t)nobs_total);
    if (blob_early_.used > blob_early_.dev_cap) {
      if (blob_early_.dev) cudaFree(blob_early_.dev);
      blob_early_.dev_cap = blob_early_.used * 2 + 4096;
      CK(cudaMalloc(&blob_early_.dev, blob_early_.dev_cap));
    }
    if ((size_t)nF > statusf_cap_) {
      if (dStatusF_) cudaFree(dStatusF_);
      statusf_cap_ = (size_t)nF * 2 + 1024;
      CK(cudaMalloc(&dStatusF_, statusf_cap_ * sizeof(int)));
    }
    CK(cudaMemcpyAsync(blob_early_.dev, blob_early_.pinned, blob_early_.used, cudaMemcpyHostToDevice, stream_));
    g_hp.mark("obs_up");
  }
  // ---- host staging of the window
  double* cl = S.hCl0;
  double* im = S.hIm0;
  std::memset(cl, 0, (size_t)Ncap_ * CL_STRIDE * sizeof(double));
  std::memset(im, 0, IM_STRIDE * sizeof(double));
  double Rbc[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, tcb[3] = {0, 0, 0};
  if (io.R_b2c) std::memcpy(Rbc, io.R_b2c, sizeof(Rbc));
  if (io.t_c_b) std::memcpy(tcb, io.t_c_b, sizeof(tcb));
  for (int k = 0; k < 9; ++k) im[IM_RBC + k] = Rbc[k];
  for (int k = 0; k < 3; ++k) im[IM_TCB + k] = tcb[k];
  for (int c = 0; c < N; ++c) {
    double* r = cl + (size_t)c * CL_STRIDE;
    const double* R = io.clone_R + 9 * (size_t)c;
    const double* p = io.clone_p + 3 * (size_t)c;
    if (io.poses_are_camera) {
      // camera poses given directly (triangulation-only entry): body pose unused
      for (int k = 0; k < 9; ++k) { r[CL_RC + k] = R[k]; r[CL_R + k] = R[k]; }
      for (int k = 0; k < 3; ++k) { r[CL_PC + k] = p[k]; r[CL_P + k] = p[k]; }
    } else {
      for (int k = 0; k < 9; ++k) r[CL_R + k] = R[k];
      for (int k = 0; k < 3; ++k) r[CL_P + k] = p[k];
      double Rc[9], t[3];
      m3_mulT(R, Rbc, Rc);
      m3_vec(R, tcb, t);
      for (int k = 0; k < 9; ++k) r[CL_RC + k] = Rc[k];
      for (int k = 0; k < 3; ++k) r[CL_PC + k] = p[k] + t[k];
    }
  }
  // imu record: current state = newest clone (only used by the state increment)
  for (int k = 0; k < 9; ++k) im[IM_R + k] = cl[(size_t)(N - 1) * CL_STRIDE + CL_R + k];
  for (int k = 0; k < 3; ++k) im[IM_P + k] = cl[(size_t)(N - 1) * CL_STRIDE + CL_P + k];
  CK(cudaMemcpyAsync(S.dCl0, S.hCl0, (size_t)Ncap_ * CL_STRIDE * sizeof(double), cudaMemcpyHostToDevice, stream_));
  CK(cudaMemcpyAsync(S.dIm0, S.hIm0, IM_STRIDE * sizeof(double), cudaMemcpyHostToDevice, stream_));
  FilterHost& F = f_[0];
  F.clones.clear();
  for (int c = 0; c < N; ++c) F.clones.push_back(CloneMeta{c, (double)c, 0.0});

  if (!early_tri) {
    wait_flag(S.scan_done);
    if (S.list_err != ORCVIO_OK) {
      wait_flag(S.lists_done);
      return S.list_err;
    }
  }
  // Early triangulation (end-to-end call): the inputs are validated, so upload the caller's observation pools
  // as they are and start k_triangulate in direct mode now -- it runs (beside the prior factor) while the host
  // sorts the candidates, builds the tiles and uploads the work lists below.
  S.tri_early = false;
  if (early_tri) {
    // the window the kernels work on (snapshot_execute skips these restores for this run)
    CK(cudaMemcpyAsync(dClones_, S.dCl0, (size_t)Ncap_ * CL_STRIDE * sizeof(double), cudaMemcpyDeviceToDevice, stream_));
    CK(cudaMemcpyAsync(dImu_, S.dIm0, IM_STRIDE * sizeof(double), cudaMemcpyDeviceToDevice, stream_));
    CK(cudaMemsetAsync(dFgen_, 0xFF, (size_t)Fcap_ * sizeof(long long), stream_));
    w.pre_dOc = (const int*)(blob_early_.dev + e_oc);
    w.pre_dOz = (const double*)(blob_early_.dev + e_oz);
    TriArgs ta{};
    ta.cand = nullptr; ta.n_cand = nF;
    ta.clones = dClones_; ta.clone_stride = (size_t)Ncap_ * CL_STRIDE;
    ta.fpos = dFpos_; ta.fgen = dFgen_; ta.fcap = Fcap_;
    ta.obs_clone = w.pre_dOc; ta.obs_z = w.pre_dOz;
    ta.cfg = tricfg_;
    ta.status = dStatusF_;
    ta.feat_off = (const int*)(blob_early_.dev + e_fo);
    ta.direct_n_clones = N; ta.direct_n_obs = nobs_total;
    launch_triangulate(ta, stream_);
    ++launches_;
    S.tri_early = true;
    g_hp.mark("tri_early");
    // the kernel guards itself against malformed lists; the host check that turns them into an error code runs
    // while it is already working
    bool bad = false;
    for (int f = 0; f < nF && !bad; ++f) {
      const int o0 = io.feat_off[f], m = io.feat_off[f + 1] - o0;
      if (m < 1 || m > ORCVIO_MAX_OBS || o0 < 0 || o0 + m > nobs_total) { bad = true; break; }
      for (int k = 0; k < m; ++k) {
        const int ci = io.obs_clone[o0 + k];
        if (ci < 0 || ci >= N) { bad = true; break; }
      }
    }
    if (bad) {
      wait_flag(S.lists_done);
      CK(cudaStreamSynchronize(stream_));
      S.tri_early = false;
      return ORCVIO_ERR_ARG;
    }
    g_hp.mark("validate");
  }
  // P: the caller's matrix is column-major and symmetric, the device copy row-major with ld
  if (io.P_in) {
    for (int i = 0; i < D; ++i) {
      std::memcpy(S.hP0 + (size_t)i * ldp_, io.P_in + (size_t)i * D, D * sizeof(double));
      for (int j = D; j < ldp_; ++j) S.hP0[(size_t)i * ldp_ + j] = 0.0;
    }
    for (int i = D; i < ldp_; ++i) std::memset(S.hP0 + (size_t)i * ldp_, 0, ldp_ * sizeof(double));
  } else {
    std::memset(S.hP0, 0, (size_t)ldp_ * ldp_ * sizeof(double));
  }
  g_hp.mark("stageP");
  // when the early triangulation is already queued on stream_, P goes up on the side stream: the prior factor
  // (which forks off the P upload) must not wait for k_triangulate
  cudaStream_t sp = S.tri_early ? stream_up_ : stream_;
  CK(cudaMemcpyAsync(S.dP0, S.hP0, (size_t)ldp_ * ldp_ * sizeof(double), cudaMemcpyHostToDevice, sp));
  S.prior_early = false;
  if ((io.stages & 4) && io.early_prior) {
    // The prior factor needs only P: put P in place and start k_chol_prior on the second stream now, so it
    // runs while the host is still building and uploading this frame's work lists.
    S.hFw[0] = FilterWork{};
    S.hFw[0].N = N; S.hFw[0].D = D; S.hFw[0].active = 1;
    CK(cudaMemcpyAsync(S.dFw, S.hFw, sizeof(FilterWork), cudaMemcpyHostToDevice, sp));
    CK(cudaMemcpyAsync(dP_, S.dP0, (size_t)ldp_ * ldp_ * sizeof(double), cudaMemcpyDeviceToDevice, sp));
    CK(cudaEventRecord(ev_fork_, sp));
    InfoBufs ib{};
    ib.Ls = dLs_; ib.ls_done = ev_ls_;
    launch_info_prior(upd_args(S.dFw), ib, N, stream2_, ev_fork_, ev_join_);
    launches_ += 2;
    S.prior_early = true;
  }
  if (sp != stream_) {               // everything queued on stream_ from here on sees P (and dP_)
    CK(cudaEventRecord(ev_p_, sp));
    CK(cudaStreamWaitEvent(stream_, ev_p_, 0));
  }
  g_hp.mark("prior_launch");
  S.jac_early = false;
  if (S.tri_early) {
    wait_flag(S.scan_done);            // per-feature offsets and size classes (helper thread); inputs already validated
    g_hp.mark("scan_wait");
    // ... and the Jacobian / nullspace / gate pass right behind it, also in direct mode: the per-feature
    // offsets and size classes come out of the validation scan, so nothing of it waits for the sorted lists
    if (!io.raw_Hx) {
      ensure_scratch(std::max(nF, 1), std::max<size_t>(w.hblk_total, 1), std::max<size_t>(w.rows_total, 1));
      if ((size_t)nF > gammaf_cap_) {
        if (dGammaF_) cudaFree(dGammaF_);
        gammaf_cap_ = (size_t)nF * 2 + 1024;
        CK(cudaMalloc(&dGammaF_, gammaf_cap_ * sizeof(double)));
      }
      blob_early2_.reset();
      const size_t e_ro = blob_early2_.reserve(sizeof(int) * (size_t)nF);
      const size_t e_ho = blob_early2_.reserve(sizeof(int) * (size_t)nF);
      const size_t e_sb = blob_early2_.reserve(sizeof(int) * (size_t)nF);
      const size_t e_eb = blob_early2_.reserve(sizeof(int) * (size_t)nF);
      const size_t e_sm = blob_early2_.reserve(sizeof(int) * std::max<size_t>(S.small_f.size(), 1));
      const size_t e_lg = blob_early2_.reserve(sizeof(int) * std::max<size_t>(S.large_f.size(), 1));
      std::memcpy(blob_early2_.pinned + e_ro, S.rowoff_f.data(), sizeof(int) * (size_t)nF);
      std::memcpy(blob_early2_.pinned + e_ho, S.hblkoff_f.data(), sizeof(int) * (size_t)nF);
      std::memcpy(blob_early2_.pinned + e_sb, S.sblk.data(), sizeof(int) * (size_t)nF);
      std::memcpy(blob_early2_.pinned + e_eb, S.eblk.data(), sizeof(int) * (size_t)nF);
      if (!S.small_f.empty()) std::memcpy(blob_early2_.pinned + e_sm, S.small_f.data(), sizeof(int) * S.small_f.size());
      if (!S.large_f.empty()) std::memcpy(blob_early2_.pinned + e_lg, S.large_f.data(), sizeof(int) * S.large_f.size());
      if (blob_early2_.used > blob_early2_.dev_cap) {
        if (blob_early2_.dev) cudaFree(blob_early2_.dev);
        blob_early2_.dev_cap = blob_early2_.used * 2 + 4096;
        CK(cudaMalloc(&blob_early2_.dev, blob_early2_.dev_cap));
      }
      CK(cudaMemcpyAsync(blob_early2_.dev, blob_early2_.pinned, blob_early2_.used, cudaMemcpyHostToDevice, stream_));
      JacArgs ja{};
      ja.cand = nullptr;
      ja.clones = dClones_; ja.clone_stride = (size_t)Ncap_ * CL_STRIDE;
      ja.imu = dImu_; ja.fpos = dFpos_; ja.fcap = Fcap_;
      ja.P = dP_; ja.p_stride = (size_t)ldp_ * ldp_; ja.ldp = ldp_;
      ja.obs_clone = w.pre_dOc; ja.obs_z = w.pre_dOz;
      ja.flags = flags_; ja.sigma2 = p_.feature_observation_noise; ja.chi2 = dChi2_;
      ja.status = dStatusF_; ja.gamma = dGammaF_;
      ja.hblk = dHblk_; ja.rblk = dRblk_;
      ja.feat_off = (const int*)(blob_early_.dev + e_fo);
      ja.rowoff_f = (const int*)(blob_early2_.dev + e_ro);
      ja.hblkoff_f = (const int*)(blob_early2_.dev + e_ho);
      JacArgs js = ja, jl = ja;
      js.cand_list = (const int*)(blob_early2_.dev + e_sm); js.n_list = (int)S.small_f.size();
      jl.cand_list = (const int*)(blob_early2_.dev + e_lg); jl.n_list = (int)S.large_f.size();
      if (!S.prior_early) CK(cudaMemcpyAsync(dP_, S.dP0, (size_t)ldp_ * ldp_ * sizeof(double), cudaMemcpyDeviceToDevice, stream_));
      launch_jac_gate(js, jl, stream_);
      launches_ += (js.n_list > 0) + (jl.n_list > 0);
      S.jac_early = true;
      // the A-form kernel reads the same per-feature arrays (+ the sorted order): no candidate record is uploaded
      dir_feat_off_ = ja.feat_off; dir_rowoff_ = ja.rowoff_f; dir_hblkoff_ = ja.hblkoff_f;
      dir_sblk_ = (const int*)(blob_early2_.dev + e_sb);
      dir_eblk_ = (const int*)(blob_early2_.dev + e_eb);
      w.cands_stay_on_host = true;
    }
    g_hp.mark("jac_early");
  }
  wait_flag(S.lists_done);
  if (w.cands_stay_on_host) w.extra_ints.assign(S.order.begin(), S.order.end());
  g_hp.mark("lists_wait");
  const int nC = nF;

  S.has_positions = io.positions_in != nullptr;
  if (S.has_positions) {
    if ((size_t)Fcap_ > S.pos_cap) {
      cudaFree(S.dPos0); cudaFree(S.dGen0);
      S.pos_cap = Fcap_;
      CK(cudaMalloc(&S.dPos0, S.pos_cap * FP_STRIDE * sizeof(double)));
      CK(cudaMalloc(&S.dGen0, S.pos_cap * sizeof(long long)));
    }
    std::vector<double> pos_in((size_t)Fcap_ * FP_STRIDE, 0.0);
    for (int f = 0; f < io.n_feat; ++f)
      for (int k = 0; k < 3; ++k) pos_in[(size_t)f * FP_STRIDE + k] = io.positions_in[3 * (size_t)f + k];
    // mark every slot initialised with its own generation so the kernels use the given positions
    std::vector<long long> gens(Fcap_, -1);
    for (int f = 0; f < io.n_feat; ++f) gens[f] = f + 1;
    CK(cudaMemcpy(S.dPos0, pos_in.data(), pos_in.size() * sizeof(double), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(S.dGen0, gens.data(), gens.size() * sizeof(long long), cudaMemcpyHostToDevice));
  }
  want_iters_ = io.iters || io.cost;
  want_raw_ = io.raw_Hx != nullptr;
  skip_tri_ = !(io.stages & 1);
  skip_jac_ = !(io.stages & 2);
  skip_update_ = !(io.stages & 4);
  // (packing the blob on the helper thread as well was measured: the H2D copy of lines last written by
  // another core delays the GPU by ~60 us -- the copy into the pinned blob stays on this thread)
  upload_on_side_stream_ = S.tri_early;
  stage_phase(w);
  upload_on_side_stream_ = false;
  g_hp.mark("stage_blob");
  if (skip_tri_ && nC > 0) {
    std::vector<int> st(nC, ST_TRI_VALID);
    CK(cudaMemcpy(dStatus_, st.data(), sizeof(int) * nC, cudaMemcpyHostToDevice));
  }
  return ok_ ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

// Restore the pristine window and run the kernel chain once (asynchronous on stream_).
int Batch::snapshot_execute(bool download) {
  if (!snap_) return ORCVIO_ERR_ARG;
  SnapState& S = *snap_;
  const bool prior_in_flight = S.prior_early;      // P restored and k_chol_prior started by snapshot_prepare
  S.prior_early = false;
  // Repeated runs on a resident frame (orcvio_frame_run: the device-timed loop) replay ONE CUDA graph holding the
  // restore copies and the whole two-stream kernel chain: the per-kernel launch latencies leave the critical path.
  // The first two runs after a prepare go the ordinary way (they grow scratch buffers and set function attributes).
  static const int graph_env = env_int("ORCVIO_GRAPH", 1);
  const bool graphable = graph_env && !download && !profiling_ && !prior_in_flight && !S.tri_early && !S.jac_early &&
                         !want_iters_ && !want_raw_;
  if (graphable && S.graph_exec) {
    CK(cudaGraphLaunch(S.graph_exec, stream_));
    launches_ += S.graph_launches;
    S.by_feature = false;
    return ok_ ? ORCVIO_OK : ORCVIO_ERR_CUDA;
  }
  const bool capture = graphable && S.plain_runs >= 2;
  const long long launches_before = launches_;
  if (capture) {
    if (cudaStreamBeginCapture(stream_, cudaStreamCaptureModeRelaxed) != cudaSuccess) {
      cudaGetLastError();
      return snapshot_execute_plain(download, prior_in_flight);
    }
    graph_capturing_ = true;
  }
  const int rc = snapshot_execute_plain(download, prior_in_flight);
  if (capture) {
    graph_capturing_ = false;
    cudaGraph_t g = nullptr;
    if (cudaStreamEndCapture(stream_, &g) != cudaSuccess || !g) {
      cudaGetLastError();
      S.plain_runs = -1000000;         // give up on graphs for this frame
      return snapshot_execute_plain(download, false);
    }
    if (cudaGraphInstantiate(&S.graph_exec, g, 0) != cudaSuccess) {
      cudaGetLastError();
      S.graph_exec = nullptr;
      S.plain_runs = -1000000;
    }
    cudaGraphDestroy(g);
    S.graph_launches = (int)(launches_ - launches_before);
    launches_ = launches_before;       // nothing has run yet: the capture only recorded the chain
    if (S.graph_exec) {
      CK(cudaGraphLaunch(S.graph_exec, stream_));
      launches_ += S.graph_launches;
      return ok_ ? ORCVIO_OK : ORCVIO_ERR_CUDA;
    }
    return snapshot_execute_plain(download, false);
  }
  if (graphable) ++S.plain_runs;
  return rc;
}

int Batch::snapshot_execute_plain(bool download, bool prior_in_flight) {
  SnapState& S = *snap_;
  if (!prior_in_flight && !(S.tri_early && S.jac_early))
    CK(cudaMemcpyAsync(dP_, S.dP0, (size_t)ldp_ * ldp_ * sizeof(double), cudaMemcpyDeviceToDevice, stream_));
  tri_done_early_ = S.tri_early;                    // window restored and k_triangulate started by snapshot_prepare
  jac_done_early_ = S.tri_early && S.jac_early;
  S.by_feature = jac_done_early_;
  S.tri_early = false;
  S.jac_early = false;
  if (!tri_done_early_) {
    CK(cudaMemcpyAsync(dClones_, S.dCl0, (size_t)Ncap_ * CL_STRIDE * sizeof(double), cudaMemcpyDeviceToDevice, stream_));
    CK(cudaMemcpyAsync(dImu_, S.dIm0, IM_STRIDE * sizeof(double), cudaMemcpyDeviceToDevice, stream_));
    if (S.has_positions) {
      CK(cudaMemcpyAsync(dFpos_, S.dPos0, (size_t)Fcap_ * FP_STRIDE * sizeof(double), cudaMemcpyDeviceToDevice, stream_));
      CK(cudaMemcpyAsync(dFgen_, S.dGen0, (size_t)Fcap_ * sizeof(long long), cudaMemcpyDeviceToDevice, stream_));
    } else {
      CK(cudaMemsetAsync(dFgen_, 0xFF, (size_t)Fcap_ * sizeof(long long), stream_));
    }
  }
  launch_phase(S.w, download, prior_in_flight);
  g_hp.mark("launch");
  return ok_ ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

int Batch::snapshot_fetch(const SnapshotIO& io) {
  if (!snap_) return ORCVIO_ERR_ARG;
  SnapState& S = *snap_;
  const int N = S.N, D = S.D, nC = (int)S.w.cands.size();
  // queue every download on the stream, then one synchronisation
  double* hP = S.hOut;
  double* hDx = hP + (size_t)ldp_ * ldp_;
  double* hCl = hDx + ldp_;
  if (io.P_out) CK(cudaMemcpyAsync(hP, dP_, (size_t)D * ldp_ * sizeof(double), cudaMemcpyDeviceToHost, stream_));
  else if (io.P_lead9) CK(cudaMemcpyAsync(hP, dP_, (size_t)9 * ldp_ * sizeof(double), cudaMemcpyDeviceToHost, stream_));
  if (io.delta_x) CK(cudaMemcpyAsync(hDx, dDx_, ldp_ * sizeof(double), cudaMemcpyDeviceToHost, stream_));
  if (io.clone_out) CK(cudaMemcpyAsync(hCl, dClones_, (size_t)N * CL_STRIDE * sizeof(double), cudaMemcpyDeviceToHost, stream_));
  CK(cudaStreamSynchronize(stream_));
  g_hp.mark("gpu_wait");
  if (io.status || io.gamma)
    for (int c = 0; c < nC; ++c) {
      const int f = S.by_feature ? c : S.order[c];
      if (io.status) io.status[f] = hStatus_[c];
      if (io.gamma) io.gamma[f] = hGamma_[c];
    }
  if (io.iters || io.cost) {
    std::vector<int> it(2 * (size_t)nC);
    std::vector<double> cs(nC);
    CK(cudaMemcpy(it.data(), dIters_, it.size() * sizeof(int), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(cs.data(), dCost_, cs.size() * sizeof(double), cudaMemcpyDeviceToHost));
    for (int c = 0; c < nC; ++c) {
      if (io.iters) { io.iters[2 * S.order[c]] = it[2 * c]; io.iters[2 * S.order[c] + 1] = it[2 * c + 1]; }
      if (io.cost) io.cost[S.order[c]] = cs[c];
    }
  }
  if (io.positions) {
    std::vector<double> fp((size_t)S.n_feat * FP_STRIDE);
    CK(cudaMemcpy(fp.data(), dFpos_, fp.size() * sizeof(double), cudaMemcpyDeviceToHost));
    for (int f = 0; f < S.n_feat; ++f)
      for (int k = 0; k < 3; ++k) io.positions[3 * (size_t)f + k] = fp[(size_t)f * FP_STRIDE + k];
  }
  if (io.raw_Hx) {
    const size_t no = (size_t)S.nobs_total;
    CK(cudaMemcpy(io.raw_Hx, dRawHx_, no * 12 * sizeof(double), cudaMemcpyDeviceToHost));
    if (io.raw_He) CK(cudaMemcpy(io.raw_He, dRawHe_, no * 12 * sizeof(double), cudaMemcpyDeviceToHost));
    if (io.raw_Hf) CK(cudaMemcpy(io.raw_Hf, dRawHf_, no * 6 * sizeof(double), cudaMemcpyDeviceToHost));
    if (io.raw_r) CK(cudaMemcpy(io.raw_r, dRawR_, no * 2 * sizeof(double), cudaMemcpyDeviceToHost));
  }
  if (io.P_lead9)
    for (int i = 0; i < 9; ++i) std::memcpy(io.P_lead9 + 9 * i, hP + (size_t)i * ldp_, 9 * sizeof(double));
  if (io.P_out)   // the posterior is exactly symmetric: row-major with ld == column-major D x D
    for (int i = 0; i < D; ++i) std::memcpy(io.P_out + (size_t)i * D, hP + (size_t)i * ldp_, D * sizeof(double));
  if (io.delta_x) std::memcpy(io.delta_x, hDx, D * sizeof(double));
  if (io.clone_out)
    for (int c = 0; c < N; ++c) {
      for (int k = 0; k < 9; ++k) io.clone_out[12 * (size_t)c + k] = hCl[(size_t)c * CL_STRIDE + CL_R + k];
      for (int k = 0; k < 3; ++k) io.clone_out[12 * (size_t)c + 9 + k] = hCl[(size_t)c * CL_STRIDE + CL_P + k];
    }
  g_hp.mark("unpack");
  g_hp.done();
  return ok_ ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

// Per-stage device times (us) of the most recent snapshot_execute run with profiling on.
void Batch::snapshot_stage_times(float* us6) {
  float ms = 0;
  const bool upd = !skip_update_ && snap_ && snap_->w.any_active;
  for (int k = 0; k < 6; ++k) us6[k] = 0.f;
  cudaEventElapsedTime(&ms, ev_[0], ev_[1]); us6[0] = ms * 1000.f;
  cudaEventElapsedTime(&ms, ev_[1], ev_[2]); us6[1] = ms * 1000.f;
  if (upd) {
    cudaEventElapsedTime(&ms, ev_[2], ev_[3]); us6[2] = ms * 1000.f;
    cudaEventElapsedTime(&ms, ev_[3], ev_[4]); us6[3] = ms * 1000.f;
    cudaEventElapsedTime(&ms, ev_[4], ev_[5]); us6[4] = ms * 1000.f;
    cudaEventElapsedTime(&ms, ev_[0], ev_[5]); us6[5] = ms * 1000.f;
    cudaEventElapsedTime(&ms, ev_[3], ev_[8]); last_syrk_us_ = ms * 1000.f;
    if (cudaEventElapsedTime(&ms, ev_[9], ev_[10]) == cudaSuccess) last_prior_us_ = ms * 1000.f;
    else (void)cudaGetLastError();
  } else {
    cudaEventElapsedTime(&ms, ev_[0], ev_[2]); us6[5] = ms * 1000.f;
  }
}

int Batch::run_snapshot(const SnapshotIO& io) {
  int rc = snapshot_prepare(io);
  if (rc != ORCVIO_OK) return rc;
  const bool old_prof = profiling_;
  profiling_ = true;
  double acc[6] = {0, 0, 0, 0, 0, 0};
  const int reps = std::max(io.repeat, 1);
  for (int rep = 0; rep < reps; ++rep) {
    snapshot_execute(true);
    CK(cudaStreamSynchronize(stream_));
    float us[6];
    snapshot_stage_times(us);
    for (int k = 0; k < 6; ++k) acc[k] += us[k];
  }
  profiling_ = old_prof;
  if (io.timings_us)
    for (int k = 0; k < 6; ++k) io.timings_us[k] = (float)(acc[k] / reps);
  rc = snapshot_fetch(io);
  want_iters_ = want_raw_ = skip_tri_ = skip_jac_ = skip_update_ = false;
  return rc;
}

}  // namespace ob

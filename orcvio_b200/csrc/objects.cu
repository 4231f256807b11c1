// Host side of stage 3 (object residual update) and the stand-alone stage 6 entry.
//   Batch::construct_object_jacobians  OrcVIO::constructObjectResidualJacobians  src/orcvio.cpp:2017-2151
//   Batch::object_update               OrcVIO::removeLostObjects                  src/orcvio.cpp:2154-2193
//                                       (-> nullspace projection, gate with dof = rows, update)
//   object_residuals                    CameraLM / ObjectLM functor evaluation     (obj_kernel.cu)
//   Batch::propagate_standalone        OrcVIO::processModel over a sample list    src/orcvio.cpp:727-823
#include <cmath>
#include <cstdio>
#include <cstring>

#include "batch.h"

namespace ob {

#define CKO(call)                                                                                  \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess) {                                                                      \
      std::fprintf(stderr, "[orcvio_b200] CUDA error %s at %s:%d\n", cudaGetErrorString(e__),      \
                   __FILE__, __LINE__);                                                            \
      return ORCVIO_ERR_CUDA;                                                                      \
    }                                                                                              \
  } while (0)

namespace {

struct DevBuf {
  void* p = nullptr;
  ~DevBuf() { if (p) cudaFree(p); }
  template <class T> T* as() { return (T*)p; }
  cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 8); }
};

// Scratch of the calling thread for the per-object entries: ONE grow-only device block and ONE pinned host block,
// carved by bump pointers.  The entries are called once per object and frame; a cudaMalloc / cudaFree pair per buffer
// (about ten per call, each a device-wide synchronisation) and a blocking copy per argument were most of their time.
// A call stages its inputs in the pinned block, uploads them with one copy, runs, and brings its outputs back with one.
struct Scratch {
  char *dev = nullptr, *pin = nullptr;
  size_t dcap = 0, pcap = 0, dused = 0, pused = 0;
  int device = -1;
  ~Scratch() {}                                       // (thread exit: the context outlives us; nothing to do safely)
  bool begin(size_t dbytes, size_t pbytes) {
    int cur = 0;
    if (cudaGetDevice(&cur) != cudaSuccess) return false;
    if (cur != device) { dev = nullptr; pin = nullptr; dcap = pcap = 0; device = cur; }   // (another context's block)
    dbytes += 4096; pbytes += 4096;
    if (dbytes > dcap) {
      if (dev) cudaFree(dev);
      dcap = dbytes * 2;
      if (cudaMalloc(&dev, dcap) != cudaSuccess) { dev = nullptr; dcap = 0; return false; }
    }
    if (pbytes > pcap) {
      if (pin) cudaFreeHost(pin);
      pcap = pbytes * 2;
      if (cudaMallocHost(&pin, pcap) != cudaSuccess) { pin = nullptr; pcap = 0; return false; }
    }
    dused = pused = 0;
    return true;
  }
  template <class T> T* d(size_t n) {
    T* r = (T*)(dev + dused);
    dused += (n * sizeof(T) + 255) & ~(size_t)255;
    return r;
  }
  template <class T> T* h(size_t n) {
    T* r = (T*)(pin + pused);
    pused += (n * sizeof(T) + 255) & ~(size_t)255;
    return r;
  }
};
thread_local Scratch g_scr;
inline size_t al(size_t bytes) { return (bytes + 255) & ~(size_t)255; }

// Sophus::SE3d::exp([upsilon, omega]) (call site src/orcvio.cpp:2083): R (row-major 3x3), t
void se3_exp_host(const double* xi, double* R, double* t) {
  const double* ups = xi;
  const double* om = xi + 3;
  so3_exp(om, R);
  const double th = std::sqrt((om[0] * om[0] + om[1] * om[1]) + om[2] * om[2]);
  double V[9];
  if (th < 1e-10) {
    std::memcpy(V, R, sizeof(V));
  } else {
    double W[9], W2[9];
    m3_skew(om, W);
    m3_mul(W, W, W2);
    const double a = (1 - std::cos(th)) / (th * th), b = (th - std::sin(th)) / (th * th * th);
    for (int i = 0; i < 9; ++i) V[i] = ((i % 4 == 0) ? 1.0 : 0.0) + a * W[i] + b * W2[i];
  }
  m3_vec(V, ups, t);
}

// get_cam_wrt_imu_se3_jacobian, include/orcvio/utils/se3_ops.hpp:531-552 (row-major 6x6)
void cam_wrt_imu_jacobian(const double* R_b2c, const double* t_c_b, const double* R_w2c, const double* t_b_w,
                          bool left, double* J) {
  std::memset(J, 0, 36 * sizeof(double));
  if (left) {
    double S[9];
    m3_skew(t_b_w, S);
    for (int i = 0; i < 3; ++i) {
      for (int j = 0; j < 3; ++j) J[6 * i + j] = S[3 * i + j];
      J[6 * (3 + i) + i] = 1.0;
      J[6 * i + 3 + i] = 1.0;
    }
  } else {
    double S[9], RS[9];
    m3_skew(t_c_b, S);
    m3_mul(R_b2c, S, RS);
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) {
        J[6 * i + j] = -RS[3 * i + j];
        J[6 * (3 + i) + j] = R_b2c[3 * i + j];
        J[6 * i + 3 + j] = R_w2c[3 * i + j];
      }
  }
}

}  // namespace

int object_residuals(const double* frames_wTc, int T, const double* wTo, const double* shape, const double* kps,
                     int K, const double* zs, const double* zb, int flags, double* fvec, double* fjac_cam,
                     double* fjac_obj, int* zs_num, double* cam_pose_se3, int* rows_out) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    std::fprintf(stderr, "[orcvio_b200] no CUDA device: orcvio_b200 has no CPU fallback\n");
    return ORCVIO_ERR_NO_DEVICE;
  }
  if (T < 1 || K < 1 || K > 32) return ORCVIO_ERR_ARG;
  std::vector<int> off(T), num(T);
  int rows_kp = 0;
  for (int f = 0; f < T; ++f) {
    int k = 0;
    for (int q = 0; q < K; ++q) {
      const double a = zs[((size_t)f * K + q) * 2], b = zs[((size_t)f * K + q) * 2 + 1];
      if (std::isfinite(a) && std::isfinite(b)) ++k;          // filter_valid_indices, ObjectLM.cpp:190-198
    }
    off[f] = rows_kp;
    num[f] = k;
    rows_kp += 2 * k;
  }
  const int rows = rows_kp + 4 * T, odim = 9 + 3 * K;
  // inputs: [frames | wTo | shape | kps | zs | zb | off] in one upload; outputs [fvec | Jc | Jo | xi] in one download
  const size_t n_in = (size_t)16 * T + 16 + 3 + 3 * K + (size_t)2 * K * T + 4 * T;
  const size_t n_out = (size_t)rows * (1 + 6 + odim) + 6 * T;
  const size_t in_bytes = al(n_in * sizeof(double)) + al(sizeof(int) * T), out_bytes = al(n_out * sizeof(double));
  if (!g_scr.begin(in_bytes + out_bytes, in_bytes + out_bytes)) return ORCVIO_ERR_CUDA;
  double* hin = g_scr.h<double>(n_in);
  int* hoff = g_scr.h<int>(T);
  double* hout = g_scr.h<double>(n_out);
  double* din = g_scr.d<double>(n_in);
  int* doff = g_scr.d<int>(T);
  double* dout = g_scr.d<double>(n_out);
  double* q = hin;
  std::memcpy(q, frames_wTc, sizeof(double) * 16 * T); q += 16 * T;
  std::memcpy(q, wTo, sizeof(double) * 16); q += 16;
  std::memcpy(q, shape, sizeof(double) * 3); q += 3;
  std::memcpy(q, kps, sizeof(double) * 3 * K); q += 3 * K;
  std::memcpy(q, zs, sizeof(double) * 2 * K * T); q += (size_t)2 * K * T;
  std::memcpy(q, zb, sizeof(double) * 4 * T);
  std::memcpy(hoff, off.data(), sizeof(int) * T);
  // (hin and hoff are adjacent in both blocks: one copy)
  CKO(cudaMemcpyAsync(din, hin, in_bytes, cudaMemcpyHostToDevice, 0));
  const double *dT = din, *dW = dT + 16 * T, *dS = dW + 16, *dK = dS + 3, *dZs = dK + 3 * K, *dZb = dZs + (size_t)2 * K * T;
  double *dF = dout, *dJc = dF + rows, *dJo = dJc + (size_t)rows * 6, *dXi = dJo + (size_t)rows * odim;
  CKO(cudaMemsetAsync(dJc, 0, sizeof(double) * rows * (6 + odim), 0));
  launch_object_rows(dT, T, dW, dS, dK, K, dZs, dZb, flags, doff, rows_kp, rows, dF, dJc, dJo, dXi, 0);
  CKO(cudaMemcpyAsync(hout, dout, n_out * sizeof(double), cudaMemcpyDeviceToHost, 0));
  CKO(cudaStreamSynchronize(0));
  if (launch_error_count() > 0) return ORCVIO_ERR_CUDA;
  if (fvec) std::memcpy(fvec, hout, sizeof(double) * rows);
  if (fjac_cam) std::memcpy(fjac_cam, hout + rows, sizeof(double) * rows * 6);
  if (fjac_obj) std::memcpy(fjac_obj, hout + (size_t)rows * 7, sizeof(double) * rows * odim);
  if (cam_pose_se3) std::memcpy(cam_pose_se3, hout + (size_t)rows * (7 + odim), sizeof(double) * 6 * T);
  if (zs_num) std::memcpy(zs_num, num.data(), sizeof(int) * T);
  if (rows_out) *rows_out = rows;
  return ORCVIO_OK;
}

// Output matrices are column-major with leading dimension `rows` (the input row count).
int Batch::construct_object_jacobians(int fi, const double* jac_sensor, int rows, const double* timestamps, int n_ts,
                                      const double* Hf, int odim, const double* res, const int* zs_num,
                                      const double* cam_pose_se3, double* Hx_out, double* Hf_out, double* res_out,
                                      int* rows_out) {
  if (!ok_) return ORCVIO_ERR_NO_DEVICE;
  FilterHost& F = f_[fi];
  if (rows_out) *rows_out = 0;
  if (!p_.use_object_residual_update_cam_pose_flag) return 0;        // :2029-2031
  const int leg = F.leg_dim_override > 0 ? F.leg_dim_override : ORCVIO_LEG;
  const int ncl = F.num_clone_override > 0 ? F.num_clone_override : (int)F.clones.size();
  const int D = leg + 6 * ncl;
  int sum_zs = 0;
  for (int k = 0; k < n_ts; ++k) sum_zs += 2 * zs_num[k];
  if (sum_zs + 4 * n_ts != rows) return ORCVIO_ERR_ARG;
  const double* im = F.imu_mirror.data();
  const bool left = p_.use_left_perturbation_flag != 0;
  std::vector<int> map5;
  std::vector<double> jac;
  int row = 0, frow = 0, kept = 0;
  for (int k = 0; k < n_ts; ++k) {
    const int nz = 2 * zs_num[k];
    int pi = -1;
    for (size_t q = 0; q < F.cur_window_timestamps.size(); ++q)
      if (F.cur_window_timestamps[q] == timestamps[k]) { pi = (int)q; break; }     // exact ==, :2073
    if (pi >= 0 && pi < ncl) {
      double J[36];
      if (F.dcampose_fixed) {
        std::memset(J, 0, sizeof(J));
        for (int i = 0; i < 6; ++i) J[7 * i] = 1.0;
      } else {
        double R[9], t[3], Rw2c[9], tmp[3], tbw[3];
        se3_exp_host(cam_pose_se3 + 6 * k, R, t);                  // wTc
        for (int i = 0; i < 3; ++i)
          for (int j = 0; j < 3; ++j) Rw2c[3 * i + j] = R[3 * j + i];
        // t_b_w = R_c2w (-R_b2c t_c_b) + t_c_w   (:2087-2088)
        m3_vec(im + IM_RBC, im + IM_TCB, tmp);
        for (int i = 0; i < 3; ++i) tmp[i] = -tmp[i];
        m3_vec(R, tmp, tbw);
        for (int i = 0; i < 3; ++i) tbw[i] += t[i];
        cam_wrt_imu_jacobian(im + IM_RBC, im + IM_TCB, Rw2c, tbw, left, J);
      }
      const int m[5] = {frow, nz, sum_zs + 4 * k, row, pi};
      map5.insert(map5.end(), m, m + 5);
      jac.insert(jac.end(), J, J + 36);
      row += nz + 4;
      ++kept;
    }
    frow += nz;
  }
  if (rows_out) *rows_out = row;
  if (kept == 0) return 0;
  // inputs [jac_sensor | Hf | res | dcam/dimu | map5] in one upload, outputs [Hx | Hf | res] in one download
  const size_t n_in = (size_t)rows * (6 + odim + 1) + jac.size();
  const size_t n_out = (size_t)rows * (D + odim + 1);
  const size_t in_bytes = al(n_in * sizeof(double)) + al(sizeof(int) * map5.size()), out_bytes = al(n_out * sizeof(double));
  if (!g_scr.begin(in_bytes + out_bytes, in_bytes + out_bytes)) return ORCVIO_ERR_CUDA;
  double* hin = g_scr.h<double>(n_in);
  int* hmap = g_scr.h<int>(map5.size());
  double* hout = g_scr.h<double>(n_out);
  double* din = g_scr.d<double>(n_in);
  int* dmap = g_scr.d<int>(map5.size());
  double* dout = g_scr.d<double>(n_out);
  double* q = hin;
  std::memcpy(q, jac_sensor, sizeof(double) * rows * 6); q += (size_t)rows * 6;
  std::memcpy(q, Hf, sizeof(double) * rows * odim); q += (size_t)rows * odim;
  std::memcpy(q, res, sizeof(double) * rows); q += rows;
  std::memcpy(q, jac.data(), sizeof(double) * jac.size());
  std::memcpy(hmap, map5.data(), sizeof(int) * map5.size());
  CKO(cudaMemcpyAsync(din, hin, in_bytes, cudaMemcpyHostToDevice, stream_));
  CKO(cudaMemsetAsync(dout, 0, n_out * sizeof(double), stream_));
  const double *dJs = din, *dHf = dJs + (size_t)rows * 6, *dRes = dHf + (size_t)rows * odim, *dJac = dRes + rows;
  double *dHx = dout, *dHfo = dHx + (size_t)rows * D, *dReso = dHfo + (size_t)rows * odim;
  launch_object_construct(dJs, dHf, dRes, rows, odim, dmap, dJac, kept, leg, D, rows, dHx, dHfo, dReso, stream_);
  CKO(cudaMemcpyAsync(hout, dout, n_out * sizeof(double), cudaMemcpyDeviceToHost, stream_));
  CKO(cudaStreamSynchronize(stream_));
  ++launches_;
  if (Hx_out) std::memcpy(Hx_out, hout, sizeof(double) * rows * D);
  if (Hf_out) std::memcpy(Hf_out, hout + (size_t)rows * D, sizeof(double) * rows * odim);
  if (res_out) std::memcpy(res_out, hout + (size_t)rows * (D + odim), sizeof(double) * rows);
  return 1;
}

// status: 0 updated, 1 empty, 2 disabled, 3 nullspace fail, 4 gate fail, 5 nan
int Batch::object_update(int fi, const double* Hx, const double* Hf, const double* res, int rows, int odim,
                         int* status_out, double* gamma_out) {
  if (!ok_) return ORCVIO_ERR_NO_DEVICE;
  FilterHost& F = f_[fi];
  auto done = [&](int st, int rc) { if (status_out) *status_out = st; return rc; };
  if (gamma_out) *gamma_out = -1.0;
  if (rows == 0) return done(1, 0);                                               // :2159-2160
  if (!p_.use_object_residual_update_cam_pose_flag) return done(2, 0);            // :2156-2157
  if (rows <= odim) return done(3, 0);                                            // math_utils.hpp:290-297
  const int N = (int)F.clones.size(), n = 6 * N, D = ORCVIO_LEG + n;
  if (N < 1) return done(1, 0);
  const int ld = odim + n + 1;
  const size_t nM = (size_t)rows * ld;
  const size_t up_bytes = al(nM * sizeof(double)) + al(sizeof(FilterWork));
  if (!g_scr.begin(up_bytes, up_bytes + al((n + 1) * sizeof(double)))) return ORCVIO_ERR_CUDA;
  double* M = g_scr.h<double>(nM);
  FilterWork* hFw = g_scr.h<FilterWork>(1);
  double* hy = g_scr.h<double>(n + 1);
  double* dM = g_scr.d<double>(nM);
  FilterWork* dFw = g_scr.d<FilterWork>(1);
  for (int i = 0; i < rows; ++i) {
    double* r = M + (size_t)i * ld;
    for (int c = 0; c < odim; ++c) r[c] = Hf[(size_t)c * rows + i];
    for (int k = 0; k < n; ++k) r[odim + k] = Hx[(size_t)(ORCVIO_LEG + k) * rows + i];
    r[ld - 1] = res[i];
  }
  const int prow = rows - odim;
  FilterWork fw{};                                       // jrow0 = 0: a dense block has no staircase
  fw.N = N; fw.D = D; fw.active = 1; fw.arow0 = 0; fw.arows = prow;
  const int units = syrk_plan(fw, n_sm_ * syrk_waves_).total;
  const size_t need_a = ((size_t)prow + 16) * ldr_;
  if (need_a > amat_cap_) {
    if (dAmat_) cudaFree(dAmat_);
    amat_cap_ = need_a * 2;
    CKO(cudaMalloc(&dAmat_, amat_cap_ * sizeof(double)));
  }
  const size_t need_p = (size_t)units * 4096;
  if (need_p > part_cap_) {
    if (dPart_) cudaFree(dPart_);
    part_cap_ = need_p * 2;
    CKO(cudaMalloc(&dPart_, part_cap_ * sizeof(double)));
  }
  *hFw = fw;
  CKO(cudaMemcpyAsync(dM, M, up_bytes, cudaMemcpyHostToDevice, stream_));        // M and the work record: one copy
  launch_project_dense(dM, rows, ld, odim, ld, stream_);                          // nullspace_project_inplace_svd
  const size_t r_stride = (size_t)(nmax_ + 1) * ldr_;
  UpdArgs ua{};
  ua.fw = dFw; ua.n_filters = 1;
  ua.P = dP_ + (size_t)fi * ldp_ * ldp_; ua.p_stride = (size_t)ldp_ * ldp_; ua.ldp = ldp_;
  ua.r_stride = r_stride; ua.ldr = ldr_;
  ua.T = dT_ + (size_t)fi * nmax_ * ldt_; ua.S = dS_ + (size_t)fi * r_stride;
  ua.t_stride = (size_t)nmax_ * ldt_; ua.ldt = ldt_;
  ua.yv = dYv_ + (size_t)fi * ldr_;
  ua.imu = dImu_ + (size_t)fi * IM_STRIDE; ua.clones = dClones_ + (size_t)fi * Ncap_ * CL_STRIDE;
  ua.clone_stride = (size_t)Ncap_ * CL_STRIDE;
  ua.dx = dDx_ + (size_t)fi * ldp_; ua.lddx = ldp_;
  ua.flags = flags_; ua.sigma2 = p_.feature_observation_noise;
  InfoBufs ib{};
  ib.Ls = dLs_ + (size_t)fi * ORCVIO_LEG * ORCVIO_LEG; ib.Amat = dAmat_; ib.part = dPart_;
  ib.max_units = units; ib.cta_budget = n_sm_ * syrk_waves_; ib.group = syrk_group_; ib.syrk_cnt = dSyrkCnt_;
  ib.tile_rows = nullptr; ib.filter_rows = dFilterRows_ + fi;
  const double* Hp = dM + (size_t)odim * ld + odim;
  launch_info_dense_factor(ua, ib, Hp, ld, prow, n, stream_);
  launches_ += 5;
  CKO(cudaMemcpyAsync(hy, ua.yv, n * sizeof(double), cudaMemcpyDeviceToHost, stream_));
  CKO(cudaMemcpyAsync(hy + n, ua.S + (size_t)n * ldr_ + n, sizeof(double), cudaMemcpyDeviceToHost, stream_));
  CKO(cudaStreamSynchronize(stream_));
  if (launch_error_count() > 0) return ORCVIO_ERR_CUDA;
  const double corner = hy[n];
  double yy = 0.0;
  for (int k = 0; k < n; ++k) yy += hy[k] * hy[k];
  const double gamma = (corner - yy) / p_.feature_observation_noise;              // Woodbury, see info_kernel.cu
  if (gamma_out) *gamma_out = gamma;
  // gatingTestFeature with dof = rows (:2172-2175); dof >= 500 computes the quantile on the fly (:1962-1968)
  const double chi = (prow < 500) ? chi2_host_[prow] : chi2_quantile(p_.chi_square_threshold_feat, prow);
  if (!(gamma < chi)) return done(4, 0);
  for (int i = 0; i < rows; ++i) {                                                // check_nan :2178-2181
    if (std::isnan(res[i])) return done(5, 0);
    for (int k = 0; k < D; ++k)
      if (std::isnan(Hx[(size_t)k * rows + i])) return done(5, 0);
  }
  launch_info_dense_apply(ua, ib, n, stream_);
  launches_ += 1;
  download_mirrors();
  CKO(cudaStreamSynchronize(stream_));
  std::memcpy(F.imu_mirror.data(), hImu_ + (size_t)fi * IM_STRIDE, IM_STRIDE * sizeof(double));
  std::memcpy(F.clone_mirror.data(), hClones_ + (size_t)fi * Ncap_ * CL_STRIDE,
              (size_t)Ncap_ * CL_STRIDE * sizeof(double));
  return done(0, 1);
}

// Stage 6 stand-alone: propagate (state, P) over n IMU samples with the filter's kernel.
int Batch::propagate_standalone(double* state16, const double* bg, const double* ba, const double* gyro_old,
                                const double* acc_old, const OrcvioImu* imu, int n, double* P, int D,
                                const double* noise4) {
  if (!ok_) return ORCVIO_ERR_NO_DEVICE;
  if (D < ORCVIO_LEG || D > ldp_ || (D - ORCVIO_LEG) % 6 != 0 || n < 0) return ORCVIO_ERR_ARG;
  std::vector<double> im(IM_STRIDE, 0.0);
  for (int k = 0; k < 9; ++k) im[IM_R + k] = state16[k];
  for (int k = 0; k < 3; ++k) {
    im[IM_V + k] = state16[9 + k];
    im[IM_P + k] = state16[12 + k];
    im[IM_BG + k] = bg ? bg[k] : 0.0;
    im[IM_BA + k] = ba ? ba[k] : 0.0;
    im[IM_GOLD + k] = gyro_old ? gyro_old[k] : 0.0;
    im[IM_AOLD + k] = acc_old ? acc_old[k] : 0.0;
  }
  for (int k = 0; k < 9; ++k) im[IM_RBC + k] = (k % 4 == 0) ? 1.0 : 0.0;
  im[IM_TIME] = state16[15];
  CKO(cudaMemcpy(dImu_, im.data(), IM_STRIDE * sizeof(double), cudaMemcpyHostToDevice));
  CKO(cudaMemcpy2D(dP_, ldp_ * sizeof(double), P, D * sizeof(double), D * sizeof(double), D, cudaMemcpyHostToDevice));
  std::vector<PropSample> smp(std::max(n, 1));
  for (int k = 0; k < n; ++k) {
    smp[k].t = imu[k].t;
    for (int q = 0; q < 3; ++q) { smp[k].w[q] = imu[k].gyro[q]; smp[k].a[q] = imu[k].acc[q]; }
  }
  DevBuf dS, dOff, dD;
  int off[2] = {0, n};
  CKO(dS.alloc(sizeof(PropSample) * smp.size())); CKO(dOff.alloc(sizeof(off))); CKO(dD.alloc(sizeof(int)));
  CKO(cudaMemcpy(dS.p, smp.data(), sizeof(PropSample) * smp.size(), cudaMemcpyHostToDevice));
  CKO(cudaMemcpy(dOff.p, off, sizeof(off), cudaMemcpyHostToDevice));
  CKO(cudaMemcpy(dD.p, &D, sizeof(int), cudaMemcpyHostToDevice));
  PropArgs pa{};
  pa.P = dP_; pa.p_stride = (size_t)ldp_ * ldp_; pa.ldp = ldp_;
  pa.imu = dImu_;
  pa.samples = dS.as<PropSample>(); pa.samp_off = dOff.as<int>(); pa.D = dD.as<int>();
  pa.n_filters = 1; pa.flags = flags_;
  for (int k = 0; k < 4; ++k) pa.qc[k] = noise4[k];
  launch_propagate(pa, stream_);
  ++launches_;
  CKO(cudaStreamSynchronize(stream_));
  if (launch_error_count() > 0) return ORCVIO_ERR_CUDA;
  CKO(cudaMemcpy(im.data(), dImu_, IM_STRIDE * sizeof(double), cudaMemcpyDeviceToHost));
  CKO(cudaMemcpy2D(P, D * sizeof(double), dP_, ldp_ * sizeof(double), D * sizeof(double), D, cudaMemcpyDeviceToHost));
  for (int k = 0; k < 9; ++k) state16[k] = im[IM_R + k];
  for (int k = 0; k < 3; ++k) { state16[9 + k] = im[IM_V + k]; state16[12 + k] = im[IM_P + k]; }
  state16[15] = im[IM_TIME];
  return ORCVIO_OK;
}

// measurementUpdate_hybrid, legacy-state part (src/orcvio.cpp:1808-1820, 1884-1901), on a state with E inverse-depth
// feature states behind the clones (D = 22 + 6 N + E): the stacked H_o may touch every column behind the IMU block,
// so it goes through the dense whitened update (prior factor, A = H L, W = s^2 I + A^T A, P+ = s^2 Y^T Y + F_2 F_2^T)
// with n = D - 22 window columns.  Stage-level entry: P and H_o come from the caller, dx and P+ go back.
int Batch::dense_update(const double* P_in, int D, const double* H, const double* r, int rows, double* dx_out,
                        double* P_out) {
  if (!ok_) return ORCVIO_ERR_NO_DEVICE;
  const int n = D - ORCVIO_LEG;
  if (n < 1 || D > ldp_ || n > nmax_ || rows < 1) return ORCVIO_ERR_ARG;
  const int fi = 0;
  CKO(cudaMemsetAsync(dP_, 0, (size_t)ldp_ * ldp_ * sizeof(double), stream_));
  CKO(cudaMemcpy2DAsync(dP_, ldp_ * sizeof(double), P_in, D * sizeof(double), D * sizeof(double), D,
                        cudaMemcpyHostToDevice, stream_));
  const int ld = n + 1;
  std::vector<double> M((size_t)rows * ld);
  for (int i = 0; i < rows; ++i) {
    for (int k = 0; k < n; ++k) M[(size_t)i * ld + k] = H[(size_t)i * D + ORCVIO_LEG + k];
    M[(size_t)i * ld + n] = r[i];
  }
  DevBuf dM, dFw;
  CKO(dM.alloc(M.size() * sizeof(double)));
  CKO(cudaMemcpyAsync(dM.p, M.data(), M.size() * sizeof(double), cudaMemcpyHostToDevice, stream_));
  FilterWork fw{};
  fw.N = 0;                                              // no clone poses behind this entry: dx is returned, not applied
  fw.D = D; fw.active = 1; fw.arow0 = 0; fw.arows = rows;
  const int units = syrk_plan(fw, n_sm_ * syrk_waves_).total;
  const size_t need_a = ((size_t)rows + 16) * ldr_;
  if (need_a > amat_cap_) {
    if (dAmat_) cudaFree(dAmat_);
    amat_cap_ = need_a * 2;
    CKO(cudaMalloc(&dAmat_, amat_cap_ * sizeof(double)));
  }
  const size_t need_p = (size_t)units * 4096;
  if (need_p > part_cap_) {
    if (dPart_) cudaFree(dPart_);
    part_cap_ = need_p * 2;
    CKO(cudaMalloc(&dPart_, part_cap_ * sizeof(double)));
  }
  CKO(dFw.alloc(sizeof(FilterWork)));
  CKO(cudaMemcpyAsync(dFw.p, &fw, sizeof(fw), cudaMemcpyHostToDevice, stream_));
  const size_t r_stride = (size_t)(nmax_ + 1) * ldr_;
  UpdArgs ua{};
  ua.fw = dFw.as<FilterWork>(); ua.n_filters = 1;
  ua.P = dP_; ua.p_stride = (size_t)ldp_ * ldp_; ua.ldp = ldp_;
  ua.r_stride = r_stride; ua.ldr = ldr_;
  ua.T = dT_; ua.S = dS_; ua.t_stride = (size_t)nmax_ * ldt_; ua.ldt = ldt_;
  ua.yv = dYv_;
  ua.imu = dImu_; ua.clones = dClones_; ua.clone_stride = (size_t)Ncap_ * CL_STRIDE;
  ua.dx = dDx_; ua.lddx = ldp_;
  ua.flags = 0; ua.sigma2 = p_.feature_observation_noise;
  InfoBufs ib{};
  ib.Ls = dLs_; ib.Amat = dAmat_; ib.part = dPart_;
  ib.max_units = units; ib.cta_budget = n_sm_ * syrk_waves_; ib.group = syrk_group_; ib.syrk_cnt = dSyrkCnt_;
  ib.tile_rows = nullptr; ib.filter_rows = dFilterRows_ + fi;
  CKO(cudaMemsetAsync(dImu_, 0, IM_STRIDE * sizeof(double), stream_));
  launch_info_dense_factor(ua, ib, dM.as<double>(), ld, rows, n, stream_);
  launch_info_dense_apply(ua, ib, n, stream_);
  launches_ += 6;
  CKO(cudaMemcpyAsync(dx_out, dDx_, D * sizeof(double), cudaMemcpyDeviceToHost, stream_));
  CKO(cudaMemcpy2DAsync(P_out, D * sizeof(double), dP_, ldp_ * sizeof(double), D * sizeof(double), D,
                        cudaMemcpyDeviceToHost, stream_));
  CKO(cudaStreamSynchronize(stream_));
  return launch_error_count() > 0 ? ORCVIO_ERR_CUDA : ORCVIO_OK;
}

}  // namespace ob

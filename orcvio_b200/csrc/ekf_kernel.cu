// Hybrid EKF-SLAM feature rows, stage level (SURVEY 8a H1 / H2) -- the per-observation Jacobians of a
// 1-D inverse-depth feature anchored in a clone of the window, and the stacked, gated rows of the features
// that are already part of the state.
//
// Reference: OrcVIO::measurementJacobian_ekf_1didp (src/orcvio.cpp:1356-1478), featureJacobian_ekf
// (:1575-1651) and gatingTestFeature with dof 2 (:1953-1976), for feature_idp_dim == 1, use_schmidt == 0,
// if_FEJ == 0, estimate_td == 0 (every shipped yaml).  The filter-level integration of these rows (state
// augmentation with a feature block, delayed initialisation, anchor change) is not built yet: these entry
// points are the element-wise parity surface for H1 / H2, like orcvio_measurement_jacobians is for J1.
//
// Parallelisation: thread per observation (H1) / thread per feature (H2: 19 structurally non-zero columns,
// H P H^T from the corresponding 19 x 19 entries of P) -- a frame holds at most a few dozen such features.
#include <cstdio>
#include <vector>

#include "../../include/orcvio_b200.h"
#include "config.h"
#include "devmem.h"
#include "kernels.h"
#include "ekf_math.cuh"

namespace ob {

struct EkfArgs {
  const double* clones; const double* Rbc; const double* tcb;
  const int* anchor; const double* rho; const double* fan; const double* pos;   // per feature
  const int* obs_feat; const int* obs_clone; const double* obs_z; int n_obs;   // per observation
  double* Hf; double* Ha; double* Hx; double* He; double* r;
};

__global__ void __launch_bounds__(128) k_ekf_jac(EkfArgs a) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= a.n_obs) return;
  const int f = a.obs_feat[o], k = a.obs_clone[o], an = a.anchor[f];
  double Hf[2], Ha[12], Hx[12], He[12], r[2];
  ekf_jacobian_1didp(a.clones + (size_t)k * CL_STRIDE, a.clones + (size_t)an * CL_STRIDE, a.Rbc, a.tcb, a.fan[2 * f],
                     a.fan[2 * f + 1], a.rho[f], a.pos + 3 * (size_t)f, a.obs_z[2 * (size_t)o], a.obs_z[2 * (size_t)o + 1],
                     k == an, Hf, Ha, Hx, He, r);
  for (int i = 0; i < 2; ++i) { a.Hf[2 * (size_t)o + i] = Hf[i]; a.r[2 * (size_t)o + i] = r[i]; }
  for (int i = 0; i < 12; ++i) {
    a.Ha[12 * (size_t)o + i] = Ha[i];
    a.Hx[12 * (size_t)o + i] = Hx[i];
    a.He[12 * (size_t)o + i] = He[i];
  }
}

// featureJacobian_ekf + gate: feature f (state column L + 6N + f) observed by the newest clone N - 1.
struct EkfRowArgs {
  const double* clones; const double* Rbc; const double* tcb; int N; int n_feat;
  const int* anchor; const double* rho; const double* fan; const double* pos; const double* z;
  const double* P; int D;                 // column-major == row-major (symmetric)
  double sigma2, chi2;
  double* H; double* r; double* gamma; int* pass;
};

__global__ void __launch_bounds__(64) k_ekf_rows(EkfRowArgs a) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= a.n_feat) return;
  const int k = a.N - 1, an = a.anchor[f], D = a.D;
  double Hf[2], Ha[12], Hx[12], He[12], r[2];
  ekf_jacobian_1didp(a.clones + (size_t)k * CL_STRIDE, a.clones + (size_t)an * CL_STRIDE, a.Rbc, a.tcb, a.fan[2 * f],
                     a.fan[2 * f + 1], a.rho[f], a.pos + 3 * (size_t)f, a.z[2 * f], a.z[2 * f + 1], k == an, Hf, Ha, Hx,
                     He, r);
  double* H = a.H + (size_t)2 * f * D;
  for (int i = 0; i < 2 * D; ++i) H[i] = 0.0;
  const int cf = ORCVIO_LEG + 6 * a.N + f, ca = ORCVIO_LEG + 6 * an, ck = ORCVIO_LEG + 6 * k;
  for (int i = 0; i < 2; ++i) {
    H[(size_t)i * D + cf] = Hf[i];
    for (int j = 0; j < 6; ++j) H[(size_t)i * D + ca + j] = Ha[6 * i + j];
    for (int j = 0; j < 6; ++j) H[(size_t)i * D + ck + j] = Hx[6 * i + j];     // after H_a, like :1644-1645
    for (int j = 0; j < 6; ++j) H[(size_t)i * D + 15 + j] = He[6 * i + j];
  }
  a.r[2 * f] = r[0];
  a.r[2 * f + 1] = r[1];
  // S = H P H^T + sigma^2 I over the structurally non-zero columns
  int cols[19];
  int nc = 0;
  for (int j = 0; j < 6; ++j) cols[nc++] = 15 + j;
  for (int j = 0; j < 6; ++j) cols[nc++] = ca + j;
  if (ck != ca)
    for (int j = 0; j < 6; ++j) cols[nc++] = ck + j;
  cols[nc++] = cf;
  double s00 = 0.0, s01 = 0.0, s11 = 0.0;
  for (int x = 0; x < nc; ++x) {
    double t0 = 0.0, t1 = 0.0;
    for (int y = 0; y < nc; ++y) {
      const double p = a.P[(size_t)cols[x] * D + cols[y]];
      t0 += p * H[cols[y]];
      t1 += p * H[(size_t)D + cols[y]];
    }
    s00 += H[cols[x]] * t0;
    s01 += H[cols[x]] * t1;
    s11 += H[(size_t)D + cols[x]] * t1;
  }
  s00 += a.sigma2;
  s11 += a.sigma2;
  const double det = s00 * s11 - s01 * s01;
  const double g = (r[0] * (s11 * r[0] - s01 * r[1]) + r[1] * (s00 * r[1] - s01 * r[0])) / det;
  a.gamma[f] = g;
  a.pass[f] = g < a.chi2 ? 1 : 0;
}


// updateFeatureCov_1didp (src/orcvio.cpp:3611-3773): anchor change of one inverse-depth feature.  One CTA: the
// 1 x D Jacobian J (19 structurally non-zero entries) is built by thread 0, Pfleg = J P by all threads (one
// column each), then the feature's row / column of P is replaced (J P J^T on the diagonal).  P stays exactly
// symmetric (row and column are written from the same values), so the reference's (P + P^T)/2 is the identity.
struct ReanchorArgs {
  const double* clones; const double* Rbc; const double* tcb; int N;
  int feat_idx, old_idx, new_idx;
  double pw[3]; double rho_new;
  double* P; int D;
  double* J_out;                           // optional: the Jacobian row (D)
};

__global__ void __launch_bounds__(256) k_ekf_reanchor(ReanchorArgs a) {
  extern __shared__ double sm[];           // J (D), Pfleg (D)
  double* J = sm;
  double* Pf = sm + a.D;
  const int D = a.D, tid = threadIdx.x;
  for (int i = tid; i < D; i += blockDim.x) J[i] = 0.0;
  __syncthreads();
  const int c = ORCVIO_LEG + 6 * a.N + a.feat_idx;
  if (tid == 0)
    ekf_reanchor_jacobian(a.clones + (size_t)a.old_idx * CL_STRIDE, a.clones + (size_t)a.new_idx * CL_STRIDE, a.Rbc,
                          a.tcb, a.pw, a.rho_new, J + c, J + ORCVIO_LEG + 6 * a.old_idx, J + ORCVIO_LEG + 6 * a.new_idx,
                          J + 15);
  __syncthreads();
  if (a.J_out)
    for (int i = tid; i < D; i += blockDim.x) a.J_out[i] = J[i];
  // Pfleg[j] = sum_i J[i] P[i][j]: J is zero outside 15..20, the two clone blocks and the feature column
  const int co = ORCVIO_LEG + 6 * a.old_idx, cn = ORCVIO_LEG + 6 * a.new_idx;
  for (int j = tid; j < D; j += blockDim.x) {
    double s = 0.0;
    for (int i = 15; i < 21; ++i) s += J[i] * a.P[(size_t)i * D + j];
    for (int i = co; i < co + 6; ++i) s += J[i] * a.P[(size_t)i * D + j];
    if (cn != co)
      for (int i = cn; i < cn + 6; ++i) s += J[i] * a.P[(size_t)i * D + j];
    s += J[c] * a.P[(size_t)c * D + j];
    Pf[j] = s;
  }
  __syncthreads();
  __shared__ double s_pff;
  if (tid == 0) {
    double s = 0.0;
    for (int j = 0; j < D; ++j) s += Pf[j] * J[j];
    s_pff = s;
  }
  __syncthreads();
  for (int j = tid; j < D; j += blockDim.x) {
    const double v = (j == c) ? s_pff : Pf[j];
    a.P[(size_t)c * D + j] = v;
    a.P[(size_t)j * D + c] = v;
  }
}

// rmLostFeaturesCov (src/orcvio.cpp:3776-3828): drop one row / column of P (D x D -> (D-1) x (D-1)).
__global__ void k_ekf_drop_state(const double* Pin, int D, int col, double* Pout) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int Dn = D - 1;
  if (e >= Dn * Dn) return;
  const int i = e / Dn, j = e - i * Dn;
  Pout[e] = Pin[(size_t)(i + (i >= col)) * D + (j + (j >= col))];
}

// featureJacobian_ekf_new (:1481-1572) + the new-feature sparsification of removeLostFeatures (:2413-2443), one CTA
// per new feature.  The feature part of a new 1-D inverse-depth feature's rows is ONE column h with its own rows, so
// W = [V U] is block diagonal per feature and the sparsification is a single Householder reflection that maps h to
// beta e_0: row 0 of the reflected block is the initialisation row (H_1 | H_2 = beta, r_1), the other 2k - 1 rows
// have lost their feature part and join H_o.  (Any orthonormal basis gives the same update: SURVEY 0 #1.)
struct EkfNewArgs {
  const double* clones; const double* Rbc; const double* tcb; int N; int D;
  const int* anchor; const double* rho; const double* fan; const double* pos;
  const int* feat_off; const int* obs_clone; const double* obs_z;
  const int* row_off;                      // first nullspace row of every feature in Ho
  double* H1; double* h2; double* r1;      // initialisation rows: F x D, F, F
  double* Ho; double* ro;                  // nullspace rows: sum(2k - 1) x D, residuals
  double* scratch;                         // F x 64 x D: unreflected rows
};

__global__ void __launch_bounds__(128) k_ekf_new_rows(EkfNewArgs a) {
  __shared__ double hv[64], rv[64];
  __shared__ int orow[ORCVIO_MAX_OBS];
  __shared__ double s_tau, s_beta;
  __shared__ int s_k;
  const int f = blockIdx.x, tid = threadIdx.x, D = a.D;
  const int o0 = a.feat_off[f], m = a.feat_off[f + 1] - o0, an = a.anchor[f];
  if (tid == 0) {
    int k = 0;
    for (int i = 0; i < m; ++i)
      if (a.obs_clone[o0 + i] != an) orow[k++] = o0 + i;     // the anchor frame's own observation is not used
    s_k = k;
  }
  __syncthreads();
  const int k = s_k, rows = 2 * k;
  double* M = a.scratch + (size_t)f * 64 * D;
  for (int e = tid; e < rows * D; e += blockDim.x) M[e] = 0.0;
  __syncthreads();
  if (tid < k) {
    const int o = orow[tid], c = a.obs_clone[o];
    double Hf[2], Ha[12], Hx[12], He[12], r[2];
    ekf_jacobian_1didp(a.clones + (size_t)c * CL_STRIDE, a.clones + (size_t)an * CL_STRIDE, a.Rbc, a.tcb, a.fan[2 * f],
                       a.fan[2 * f + 1], a.rho[f], a.pos + 3 * (size_t)f, a.obs_z[2 * (size_t)o], a.obs_z[2 * (size_t)o + 1],
                       false, Hf, Ha, Hx, He, r);
    const int ca = ORCVIO_LEG + 6 * an, cc = ORCVIO_LEG + 6 * c;
    for (int i = 0; i < 2; ++i) {
      double* row = M + (size_t)(2 * tid + i) * D;
      for (int j = 0; j < 6; ++j) row[ca + j] = Ha[6 * i + j];
      for (int j = 0; j < 6; ++j) row[cc + j] = Hx[6 * i + j];
      for (int j = 0; j < 6; ++j) row[15 + j] = He[6 * i + j];
      hv[2 * tid + i] = Hf[i];
      rv[2 * tid + i] = r[i];
    }
  }
  __syncthreads();
  if (rows == 0) return;
  if (tid == 0) {            // Householder vector of h (LAPACK dlarfg convention): (I - tau v v^T) h = beta e_0, v_0 = 1
    double sig = 0.0;
    for (int i = 1; i < rows; ++i) sig += hv[i] * hv[i];
    const double alpha = hv[0];
    double beta = alpha, tau = 0.0;
    if (sig > 0.0) {
      const double nrm = sqrt(alpha * alpha + sig);
      beta = alpha >= 0.0 ? -nrm : nrm;
      tau = (beta - alpha) / beta;
      const double sc = 1.0 / (alpha - beta);
      for (int i = 1; i < rows; ++i) hv[i] *= sc;
    }
    hv[0] = 1.0;
    s_tau = tau;
    s_beta = beta;
  }
  __syncthreads();
  const double tau = s_tau;
  const int ro0 = a.row_off[f];
  for (int c = tid; c <= D; c += blockDim.x) {               // column D = the residual
    double dot = 0.0;
    for (int i = 0; i < rows; ++i) dot += hv[i] * (c < D ? M[(size_t)i * D + c] : rv[i]);
    dot *= tau;
    for (int i = 0; i < rows; ++i) {
      const double v = (c < D ? M[(size_t)i * D + c] : rv[i]) - dot * hv[i];
      if (i == 0) {
        if (c < D) a.H1[(size_t)f * D + c] = v;
        else a.r1[f] = v;
      } else {
        if (c < D) a.Ho[(size_t)(ro0 + i - 1) * D + c] = v;
        else a.ro[ro0 + i - 1] = v;
      }
    }
  }
  if (tid == 0) a.h2[f] = s_beta;
}

// The new-state part of measurementUpdate_hybrid (:1823-1832, 1903-1941; no Schmidt): HH = H_2^-1 H_1 (H_2 diagonal),
// dx_new = -HH dx_leg + H_2^-1 r_1, P_aug = [[P, -P HH^T], [-HH P, HH P HH^T + s^2 (H_2^T H_2)^-1]], symmetrised.
struct EkfInitArgs {
  const double* P; int D; int F;
  const double* dx_leg; const double* H1; const double* h2; const double* r1; double sigma2;
  double* nHHP;              // F x D scratch
  double* dx_new; double* Paug;
};

__global__ void __launch_bounds__(256) k_ekf_init_cross(EkfInitArgs a) {      // grid: F
  const int j = blockIdx.x, D = a.D, tid = threadIdx.x;
  extern __shared__ double hh[];               // HH row j
  const double ih = 1.0 / a.h2[j];
  for (int i = tid; i < D; i += blockDim.x) hh[i] = a.H1[(size_t)j * D + i] * ih;
  __syncthreads();
  for (int c = tid; c < D; c += blockDim.x) {
    double s = 0.0;
    for (int i = 0; i < D; ++i) s += hh[i] * a.P[(size_t)i * D + c];
    a.nHHP[(size_t)j * D + c] = -s;
  }
  if (tid == 0) {
    double s = 0.0;
    for (int i = 0; i < D; ++i) s += hh[i] * a.dx_leg[i];
    a.dx_new[j] = -s + a.r1[j] * ih;
  }
}

__global__ void __launch_bounds__(256) k_ekf_init_assemble(EkfInitArgs a) {
  const int D = a.D, F = a.F, Da = D + F;
  const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (size_t)Da * Da) return;
  const int i = (int)(e / Da), j = (int)(e - (size_t)i * Da);
  double v;
  if (i < D && j < D) {
    v = 0.5 * (a.P[(size_t)i * D + j] + a.P[(size_t)j * D + i]);
  } else if (i >= D && j < D) {
    v = a.nHHP[(size_t)(i - D) * D + j];
  } else if (i < D && j >= D) {
    v = a.nHHP[(size_t)(j - D) * D + i];
  } else {
    const int p = i - D, q = j - D;
    double s0 = 0.0, s1 = 0.0;              // (HH P HH^T)[p][q] and [q][p], then their mean
    const double ihq = 1.0 / a.h2[q], ihp = 1.0 / a.h2[p];
    for (int c = 0; c < D; ++c) {
      s0 -= a.nHHP[(size_t)p * D + c] * (a.H1[(size_t)q * D + c] * ihq);
      s1 -= a.nHHP[(size_t)q * D + c] * (a.H1[(size_t)p * D + c] * ihp);
    }
    v = 0.5 * (s0 + s1);
    if (p == q) v += a.sigma2 * ihp * ihp;
  }
  a.Paug[e] = v;
}

// stateAugmentation with a feature block behind the clones (src/orcvio.cpp:963-1010): the new clone's 6 x 6 block
// goes in at index c0 = 22 + 6 N, BEFORE the feature states, and equals J P J^T with J selecting theta (0..2) and
// p (6..8) of the IMU state -- so every entry of the new matrix is an entry of the old one: P'[i][j] = P[m(i)][m(j)].
__global__ void k_ekf_augment(const double* P, int D, int c0, double* Pn) {
  const int Dn = D + 6;
  const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (size_t)Dn * Dn) return;
  const int i = (int)(e / Dn), j = (int)(e - (size_t)i * Dn);
  auto m = [c0](int x) { return x < c0 ? x : (x < c0 + 6 ? (x - c0 < 3 ? x - c0 : x - c0 + 3) : x - 6); };
  const int mi = m(i), mj = m(j);
  Pn[e] = 0.5 * (P[(size_t)mi * D + mj] + P[(size_t)mj * D + mi]);
}

// pruneImuStateBuffer's covariance part for one clone (src/orcvio.cpp:2916-2940): drop its 6 rows / columns.
__global__ void k_ekf_drop_block(const double* Pin, int D, int c0, int w, double* Pout) {
  const int Dn = D - w;
  const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (size_t)Dn * Dn) return;
  const int i = (int)(e / Dn), j = (int)(e - (size_t)i * Dn);
  Pout[e] = Pin[(size_t)(i + (i >= c0 ? w : 0)) * D + (j + (j >= c0 ? w : 0))];
}

namespace {
// (at least one element, so that an empty array still has a device address)
template <class T>
bool make(DeviceBuf<T>& d, size_t n) { return d.alloc(std::max<size_t>(n, 1)); }
template <class T>
bool put(DeviceBuf<T>& d, const T* h, size_t n) {
  return make(d, n) && (n == 0 || cudaMemcpy(d.get(), h, n * sizeof(T), cudaMemcpyHostToDevice) == cudaSuccess);
}

std::vector<double> clone_records(const double* clone_R, const double* clone_p, int N) {
  std::vector<double> cl((size_t)N * CL_STRIDE, 0.0);
  for (int c = 0; c < N; ++c) {
    for (int k = 0; k < 9; ++k) cl[(size_t)c * CL_STRIDE + CL_R + k] = clone_R[9 * (size_t)c + k];
    for (int k = 0; k < 3; ++k) cl[(size_t)c * CL_STRIDE + CL_P + k] = clone_p[3 * (size_t)c + k];
  }
  return cl;
}
}  // namespace
}  // namespace ob

extern "C" int orcvio_ekf_measurement_jacobians(const double* clone_R, const double* clone_p, int n_clones,
                                                const double* R_b2c, const double* t_c_b, const int* anchor,
                                                const double* inv_depth, const double* f_an,
                                                const double* positions, const int* feat_off, const int* obs_clone,
                                                const double* obs_z, int n_feat, double* H_f, double* H_a,
                                                double* H_x, double* H_e, double* r) {
  using namespace ob;
  if (n_clones < 1 || n_feat < 0) return ORCVIO_ERR_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return ORCVIO_ERR_NO_DEVICE;
  const int n_obs = n_feat ? feat_off[n_feat] : 0;
  std::vector<int> obs_feat(n_obs);
  for (int f = 0; f < n_feat; ++f) {
    if (anchor[f] < 0 || anchor[f] >= n_clones || !(inv_depth[f] != 0.0)) return ORCVIO_ERR_ARG;
    for (int o = feat_off[f]; o < feat_off[f + 1]; ++o) {
      if (obs_clone[o] < 0 || obs_clone[o] >= n_clones) return ORCVIO_ERR_ARG;
      obs_feat[o] = f;
    }
  }
  if (n_obs == 0) return ORCVIO_OK;
  const std::vector<double> cl = clone_records(clone_R, clone_p, n_clones);
  DeviceBuf<double> dcl, dR, dt, drho, dfan, dpos, doz, dHf, dHa, dHx, dHe, dr;
  DeviceBuf<int> dan, dof, doc;
  bool ok = put(dcl, cl.data(), cl.size()) && put(dR, R_b2c, 9) && put(dt, t_c_b, 3) && put(dan, anchor, n_feat) &&
            put(drho, inv_depth, n_feat) && put(dfan, f_an, 2 * (size_t)n_feat) && put(dpos, positions, 3 * (size_t)n_feat) &&
            put(dof, obs_feat.data(), n_obs) && put(doc, obs_clone, n_obs) && put(doz, obs_z, 2 * (size_t)n_obs) &&
            make(dHf, 2 * (size_t)n_obs) && make(dHa, 12 * (size_t)n_obs) &&
            make(dHx, 12 * (size_t)n_obs) && make(dHe, 12 * (size_t)n_obs) && make(dr, 2 * (size_t)n_obs);
  if (!ok) return ORCVIO_ERR_CUDA;
  EkfArgs a{dcl.get(), dR.get(), dt.get(), dan.get(), drho.get(), dfan.get(),
            dpos.get(), dof.get(), doc.get(), doz.get(), n_obs, dHf.get(), dHa.get(),
            dHx.get(), dHe.get(), dr.get()};
  k_ekf_jac<<<(n_obs + 127) / 128, 128>>>(a);
  check_launch("k_ekf_jac");
  ok = cudaMemcpy(H_f, dHf.get(), 2 * (size_t)n_obs * 8, cudaMemcpyDeviceToHost) == cudaSuccess &&
       cudaMemcpy(H_a, dHa.get(), 12 * (size_t)n_obs * 8, cudaMemcpyDeviceToHost) == cudaSuccess &&
       cudaMemcpy(H_x, dHx.get(), 12 * (size_t)n_obs * 8, cudaMemcpyDeviceToHost) == cudaSuccess &&
       cudaMemcpy(H_e, dHe.get(), 12 * (size_t)n_obs * 8, cudaMemcpyDeviceToHost) == cudaSuccess &&
       cudaMemcpy(r, dr.get(), 2 * (size_t)n_obs * 8, cudaMemcpyDeviceToHost) == cudaSuccess;
  return ok ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

extern "C" int orcvio_ekf_feature_rows(const double* clone_R, const double* clone_p, int n_clones, const double* R_b2c,
                                       const double* t_c_b, const int* anchor, const double* inv_depth,
                                       const double* f_an, const double* positions, const double* z_cur, int n_feat,
                                       const double* P, int D, double noise_var, double chi2_p, double* H, double* r,
                                       double* gamma, int* pass) {
  using namespace ob;
  if (n_clones < 1 || n_feat < 0 || D != ORCVIO_LEG + 6 * n_clones + n_feat) return ORCVIO_ERR_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return ORCVIO_ERR_NO_DEVICE;
  for (int f = 0; f < n_feat; ++f)
    if (anchor[f] < 0 || anchor[f] >= n_clones || !(inv_depth[f] != 0.0)) return ORCVIO_ERR_ARG;
  if (n_feat == 0) return ORCVIO_OK;
  const std::vector<double> cl = clone_records(clone_R, clone_p, n_clones);
  DeviceBuf<double> dcl, dR, dt, drho, dfan, dpos, dz, dP, dH, dr, dg;
  DeviceBuf<int> dan, dp;
  bool ok = put(dcl, cl.data(), cl.size()) && put(dR, R_b2c, 9) && put(dt, t_c_b, 3) && put(dan, anchor, n_feat) &&
            put(drho, inv_depth, n_feat) && put(dfan, f_an, 2 * (size_t)n_feat) && put(dpos, positions, 3 * (size_t)n_feat) &&
            put(dz, z_cur, 2 * (size_t)n_feat) && put(dP, P, (size_t)D * D) && make(dH, (size_t)2 * n_feat * D) &&
            make(dr, 2 * (size_t)n_feat) && make(dg, n_feat) && make(dp, n_feat);
  if (!ok) return ORCVIO_ERR_CUDA;
  EkfRowArgs a{dcl.get(), dR.get(), dt.get(), n_clones, n_feat, dan.get(), drho.get(),
               dfan.get(), dpos.get(), dz.get(), dP.get(), D, noise_var,
               chi2_quantile(chi2_p, 2), dH.get(), dr.get(), dg.get(), dp.get()};
  k_ekf_rows<<<(n_feat + 63) / 64, 64>>>(a);
  check_launch("k_ekf_rows");
  ok = cudaMemcpy(H, dH.get(), (size_t)2 * n_feat * D * 8, cudaMemcpyDeviceToHost) == cudaSuccess &&
       cudaMemcpy(r, dr.get(), 2 * (size_t)n_feat * 8, cudaMemcpyDeviceToHost) == cudaSuccess &&
       cudaMemcpy(gamma, dg.get(), (size_t)n_feat * 8, cudaMemcpyDeviceToHost) == cudaSuccess &&
       cudaMemcpy(pass, dp.get(), (size_t)n_feat * 4, cudaMemcpyDeviceToHost) == cudaSuccess;
  return ok ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

extern "C" int orcvio_ekf_update_feature_cov(double* P, int D, const double* clone_R, const double* clone_p,
                                             int n_clones, const double* R_b2c, const double* t_c_b, int feat_idx,
                                             int old_idx, int new_idx, const double* p_w, double inv_depth_new,
                                             double* J_out) {
  using namespace ob;
  const int E = D - ORCVIO_LEG - 6 * n_clones;
  if (n_clones < 1 || E < 1 || feat_idx < 0 || feat_idx >= E || old_idx < 0 || old_idx >= n_clones || new_idx < 0 ||
      new_idx >= n_clones)
    return ORCVIO_ERR_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return ORCVIO_ERR_NO_DEVICE;
  const std::vector<double> cl = clone_records(clone_R, clone_p, n_clones);
  DeviceBuf<double> dcl, dR, dt, dP, dJ;
  bool ok = put(dcl, cl.data(), cl.size()) && put(dR, R_b2c, 9) && put(dt, t_c_b, 3) && put(dP, P, (size_t)D * D) &&
            make(dJ, D);
  if (!ok) return ORCVIO_ERR_CUDA;
  ReanchorArgs a{};
  a.clones = dcl.get(); a.Rbc = dR.get(); a.tcb = dt.get(); a.N = n_clones;
  a.feat_idx = feat_idx; a.old_idx = old_idx; a.new_idx = new_idx;
  for (int k = 0; k < 3; ++k) a.pw[k] = p_w[k];
  a.rho_new = inv_depth_new;
  a.P = dP.get(); a.D = D; a.J_out = dJ.get();
  k_ekf_reanchor<<<1, 256, 2 * (size_t)D * sizeof(double)>>>(a);
  check_launch("k_ekf_reanchor");
  ok = cudaMemcpy(P, dP.get(), (size_t)D * D * 8, cudaMemcpyDeviceToHost) == cudaSuccess &&
       (!J_out || cudaMemcpy(J_out, dJ.get(), (size_t)D * 8, cudaMemcpyDeviceToHost) == cudaSuccess);
  return ok ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

extern "C" int orcvio_ekf_remove_feature_cov(const double* P, int D, int n_clones, int feat_idx, double* P_out) {
  using namespace ob;
  const int E = D - ORCVIO_LEG - 6 * n_clones;
  if (n_clones < 1 || E < 1 || feat_idx < 0 || feat_idx >= E) return ORCVIO_ERR_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return ORCVIO_ERR_NO_DEVICE;
  DeviceBuf<double> dP, dO;
  const int Dn = D - 1;
  if (!put(dP, P, (size_t)D * D) || !make(dO, (size_t)Dn * Dn)) return ORCVIO_ERR_CUDA;
  k_ekf_drop_state<<<(Dn * Dn + 255) / 256, 256>>>(dP.get(), D, ORCVIO_LEG + 6 * n_clones + feat_idx, dO.get());
  check_launch("k_ekf_drop_state");
  return cudaMemcpy(P_out, dO.get(), (size_t)Dn * Dn * 8, cudaMemcpyDeviceToHost) == cudaSuccess ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

extern "C" int orcvio_ekf_new_feature_rows(const double* clone_R, const double* clone_p, int n_clones,
                                           const double* R_b2c, const double* t_c_b, const int* anchor,
                                           const double* inv_depth, const double* f_an, const double* positions,
                                           const int* feat_off, const int* obs_clone, const double* obs_z, int n_feat,
                                           int D, double* H_1, double* h_2, double* r_1, double* H_o, double* r_o,
                                           int* rows_out) {
  using namespace ob;
  if (n_clones < 1 || n_feat < 0 || D < ORCVIO_LEG + 6 * n_clones) return ORCVIO_ERR_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return ORCVIO_ERR_NO_DEVICE;
  std::vector<int> row_off(n_feat + 1, 0);
  for (int f = 0; f < n_feat; ++f) {
    if (anchor[f] < 0 || anchor[f] >= n_clones || !(inv_depth[f] != 0.0)) return ORCVIO_ERR_ARG;
    const int m = feat_off[f + 1] - feat_off[f];
    if (m < 1 || m > ORCVIO_MAX_OBS) return ORCVIO_ERR_ARG;
    int k = 0;
    for (int o = feat_off[f]; o < feat_off[f + 1]; ++o) {
      if (obs_clone[o] < 0 || obs_clone[o] >= n_clones) return ORCVIO_ERR_ARG;
      k += obs_clone[o] != anchor[f];
    }
    row_off[f + 1] = row_off[f] + std::max(2 * k - 1, 0);
  }
  if (rows_out) *rows_out = row_off[n_feat];
  if (n_feat == 0) return ORCVIO_OK;
  const int n_obs = feat_off[n_feat], n_ho = row_off[n_feat];
  const std::vector<double> cl = clone_records(clone_R, clone_p, n_clones);
  DeviceBuf<double> dcl, dR, dt, drho, dfan, dpos, doz, dH1, dh2, dr1, dHo, dr, dsc;
  DeviceBuf<int> dan, dfo, doc, dro;
  bool ok = put(dcl, cl.data(), cl.size()) && put(dR, R_b2c, 9) && put(dt, t_c_b, 3) && put(dan, anchor, n_feat) &&
            put(drho, inv_depth, n_feat) && put(dfan, f_an, 2 * (size_t)n_feat) && put(dpos, positions, 3 * (size_t)n_feat) &&
            put(dfo, feat_off, n_feat + 1) && put(doc, obs_clone, n_obs) && put(doz, obs_z, 2 * (size_t)n_obs) &&
            put(dro, row_off.data(), n_feat + 1) && make(dH1, (size_t)n_feat * D) && make(dh2, n_feat) &&
            make(dr1, n_feat) && make(dHo, (size_t)n_ho * D) && make(dr, n_ho) &&
            make(dsc, (size_t)n_feat * 64 * D);
  if (!ok) return ORCVIO_ERR_CUDA;
  cudaMemset(dH1.get(), 0, (size_t)n_feat * D * 8);
  cudaMemset(dh2.get(), 0, (size_t)n_feat * 8);
  cudaMemset(dr1.get(), 0, (size_t)n_feat * 8);
  EkfNewArgs a{dcl.get(), dR.get(), dt.get(), n_clones, D, dan.get(), drho.get(),
               dfan.get(), dpos.get(), dfo.get(), doc.get(), doz.get(), dro.get(),
               dH1.get(), dh2.get(), dr1.get(), dHo.get(), dr.get(), dsc.get()};
  k_ekf_new_rows<<<n_feat, 128>>>(a);
  check_launch("k_ekf_new_rows");
  ok = cudaMemcpy(H_1, dH1.get(), (size_t)n_feat * D * 8, cudaMemcpyDeviceToHost) == cudaSuccess &&
       cudaMemcpy(h_2, dh2.get(), (size_t)n_feat * 8, cudaMemcpyDeviceToHost) == cudaSuccess &&
       cudaMemcpy(r_1, dr1.get(), (size_t)n_feat * 8, cudaMemcpyDeviceToHost) == cudaSuccess &&
       (n_ho == 0 || (cudaMemcpy(H_o, dHo.get(), (size_t)n_ho * D * 8, cudaMemcpyDeviceToHost) == cudaSuccess &&
                      cudaMemcpy(r_o, dr.get(), (size_t)n_ho * 8, cudaMemcpyDeviceToHost) == cudaSuccess));
  return ok ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

extern "C" int orcvio_ekf_delayed_init(const double* P, int D, const double* dx_leg, const double* H_1, const double* h_2,
                                       const double* r_1, int n_new, double noise_var, double* dx_new, double* P_aug) {
  using namespace ob;
  if (D < 1 || n_new < 1) return ORCVIO_ERR_ARG;
  for (int j = 0; j < n_new; ++j)
    if (!(h_2[j] != 0.0)) return ORCVIO_ERR_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return ORCVIO_ERR_NO_DEVICE;
  const int Da = D + n_new;
  DeviceBuf<double> dP, ddx, dH1, dh2, dr1, dn, dxn, dPa;
  bool ok = put(dP, P, (size_t)D * D) && put(ddx, dx_leg, D) && put(dH1, H_1, (size_t)n_new * D) && put(dh2, h_2, n_new) &&
            put(dr1, r_1, n_new) && make(dn, (size_t)n_new * D) && make(dxn, n_new) &&
            make(dPa, (size_t)Da * Da);
  if (!ok) return ORCVIO_ERR_CUDA;
  EkfInitArgs a{dP.get(), D, n_new, ddx.get(), dH1.get(), dh2.get(), dr1.get(),
                noise_var, dn.get(), dxn.get(), dPa.get()};
  k_ekf_init_cross<<<n_new, 256, (size_t)D * sizeof(double)>>>(a);
  check_launch("k_ekf_init_cross");
  k_ekf_init_assemble<<<(int)(((size_t)Da * Da + 255) / 256), 256>>>(a);
  check_launch("k_ekf_init_assemble");
  ok = cudaMemcpy(dx_new, dxn.get(), (size_t)n_new * 8, cudaMemcpyDeviceToHost) == cudaSuccess &&
       cudaMemcpy(P_aug, dPa.get(), (size_t)Da * Da * 8, cudaMemcpyDeviceToHost) == cudaSuccess;
  return ok ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

extern "C" int orcvio_ekf_augment_cov(const double* P, int D, int n_clones, double* P_out) {
  using namespace ob;
  const int c0 = ORCVIO_LEG + 6 * n_clones;
  if (n_clones < 0 || D < c0) return ORCVIO_ERR_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return ORCVIO_ERR_NO_DEVICE;
  DeviceBuf<double> dP, dO;
  const int Dn = D + 6;
  if (!put(dP, P, (size_t)D * D) || !make(dO, (size_t)Dn * Dn)) return ORCVIO_ERR_CUDA;
  k_ekf_augment<<<(int)(((size_t)Dn * Dn + 255) / 256), 256>>>(dP.get(), D, c0, dO.get());
  check_launch("k_ekf_augment");
  return cudaMemcpy(P_out, dO.get(), (size_t)Dn * Dn * 8, cudaMemcpyDeviceToHost) == cudaSuccess ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

extern "C" int orcvio_ekf_remove_clone_cov(const double* P, int D, int n_clones, int clone_idx, double* P_out) {
  using namespace ob;
  if (n_clones < 1 || clone_idx < 0 || clone_idx >= n_clones || D < ORCVIO_LEG + 6 * n_clones) return ORCVIO_ERR_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return ORCVIO_ERR_NO_DEVICE;
  DeviceBuf<double> dP, dO;
  const int Dn = D - 6;
  if (!put(dP, P, (size_t)D * D) || !make(dO, (size_t)Dn * Dn)) return ORCVIO_ERR_CUDA;
  k_ekf_drop_block<<<(int)(((size_t)Dn * Dn + 255) / 256), 256>>>(dP.get(), D, ORCVIO_LEG + 6 * clone_idx, 6,
                                                                  dO.get());
  check_launch("k_ekf_drop_block");
  return cudaMemcpy(P_out, dO.get(), (size_t)Dn * Dn * 8, cudaMemcpyDeviceToHost) == cudaSuccess ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

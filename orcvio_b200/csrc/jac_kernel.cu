// Stage 2 -- measurement Jacobians, left-nullspace projection and chi-square gate, fused.
//
// Per candidate feature (m observations) this kernel computes what
//   OrcVIO::measurementJacobian_msckf   reference src/orcvio.cpp:1071-1168   (J1)
//   OrcVIO::featureJacobian_msckf       reference src/orcvio.cpp:1171-1226   (J2)
//   nullspace_project_inplace_svd       reference math_utils.hpp:287-312     (J3)
//   OrcVIO::gatingTestFeature           reference src/orcvio.cpp:1953-1976   (J4)
// compute, but without ever forming the dense (2m x D) H_j the reference allocates:
//   * H_j is block sparse (one 2x6 block per observation at its clone's columns), so
//     H_j P H_j^T is assembled from m^2 2x2 blocks  H_xi P[ci,cj] H_xj^T  (96 FMA each),
//   * the left nullspace of H_f (2m x 3) comes from 3 Householder reflections; the
//     orthogonal factor Q^T (2m x 2m) is formed once in shared memory and gives both
//     S = Q2^T (H P H^T) Q2 + sigma^2 I for the gate and the projected rows
//     H' = Q2^T H_x for the update.  Any orthonormal basis of null(H_f^T) gives the same
//     gate value and the same posterior (SURVEY 0 #1), the reference's SVD basis included.
// Output per candidate: status bit ST_GATE_PASS, gamma, and -- when it passes -- the
// compact projected block (r x 6(e-s+1), r = 2m-3) plus projected residual, which the QR
// compression consumes.
//
// Parallelisation: one warp per feature for m <= 8 (all shipped configs: max_track_len 6),
// one 128-thread CTA per feature for longer tracks (m <= 32).
#include "kernels.h"

namespace ob {

template <int TEAM>
__device__ __forceinline__ void team_sync() {
  if (TEAM == 32) __syncwarp();
  else __syncthreads();
}

// J1 for one observation.  Hx 2x6, Hf 2x3, r 2 (row-major); He optional.
__device__ __forceinline__ void measurement_jacobian(const double* cl, const double* Rbc,
                                                     const double* tcb, const double* pw,
                                                     double zu, double zv, int flags, double* Hx,
                                                     double* Hf, double* r, double* He) {
  const double* R = cl + CL_R;       // body -> world
  const double* p = cl + CL_P;
  // reference recomputes the camera pose from the clone's body pose (orcvio.cpp:1085-1092)
  double Rw2c[9];
  m3_mulT(Rbc, R, Rw2c);             // R_b2c * R_b2w^T
  double Rtc[3];
  m3_vec(R, tcb, Rtc);
  double tcw[3] = {p[0] + Rtc[0], p[1] + Rtc[1], p[2] + Rtc[2]};
  double d[3] = {pw[0] - tcw[0], pw[1] - tcw[1], pw[2] - tcw[2]};
  double pc[3];
  m3_vec(Rw2c, d, pc);
  double iz = 1 / pc[2];
  double dz[6] = {iz, 0, -pc[0] / (pc[2] * pc[2]), 0, iz, -pc[1] / (pc[2] * pc[2])};
  double pbf[3] = {pw[0] - p[0], pw[1] - p[1], pw[2] - p[2]};
  double Sk[9], A[9], B[9];
  double sign;
  // The OrcVIO branches go through wTc.inverse() (a general 4x4 inverse, :1136,1140), which
  // differs from the transpose when the yaml extrinsic rotation is only orthonormal to its
  // printed digits (kitti_odom.yaml: ~1e-8).  Rinv = (R_w2c^T)^-1 restates that inverse.
  double Rinv[9];
  if (!(flags & FL_LARVIO)) {
    const double* M = Rw2c;   // wTc.linear() = R_w2c^T ; inverse of the transpose = (M^-1)^T
    double c00 = M[4] * M[8] - M[5] * M[7], c01 = M[5] * M[6] - M[3] * M[8], c02 = M[3] * M[7] - M[4] * M[6];
    double c10 = M[2] * M[7] - M[1] * M[8], c11 = M[0] * M[8] - M[2] * M[6], c12 = M[1] * M[6] - M[0] * M[7];
    double c20 = M[1] * M[5] - M[2] * M[4], c21 = M[2] * M[3] - M[0] * M[5], c22 = M[0] * M[4] - M[1] * M[3];
    double det = (M[0] * c00 + M[1] * c01) + M[2] * c02;
    // M^-1 = adj(M)/det with adj = cofactor^T ; (M^-1)^T = cofactor/det
    Rinv[0] = c00 / det; Rinv[1] = c01 / det; Rinv[2] = c02 / det;
    Rinv[3] = c10 / det; Rinv[4] = c11 / det; Rinv[5] = c12 / det;
    Rinv[6] = c20 / det; Rinv[7] = c21 / det; Rinv[8] = c22 / det;
  }
  if (flags & FL_LARVIO) {
    // LARVIO (:1147-1149): [R_w2c [p_w - p]x | -R_w2c], H_x = dz * that.
    m3_skew(pbf, Sk);
    m3_mul(Rw2c, Sk, A);
    for (int i = 0; i < 9; ++i) B[i] = -Rw2c[i];
    sign = 1.0;
  } else if (flags & FL_LEFT) {
    // OrcVIO left perturbation (:1136): temp * cTw * odot([p_w;1]) * J_L reduces to
    // [cTw_R [p - p_w]x | cTw_R] and H_x = -dz * that, with cTw_R = wTc.inverse() rotation.
    m3_skew(pbf, Sk);
    m3_mul(Rinv, Sk, A);
    for (int i = 0; i < 9; ++i) B[i] = -Rinv[i];
    sign = 1.0;
  } else {
    // OrcVIO right perturbation (:1140-1143): [I, -[p_c']x] * [[-R_bc [t_cb]x, R_w2c],[R_bc, 0]]
    // with p_c' = (wTc.inverse() * [p_w;1]).head(3)
    double St[9], Sp[9], T1[9], T2[9], pci[3];
    m3_vec(Rinv, d, pci);
    m3_skew(tcb, St);
    m3_skew(pci, Sp);
    m3_mul(Rbc, St, T1);
    m3_mul(Sp, Rbc, T2);
    for (int i = 0; i < 9; ++i) { A[i] = -T1[i] - T2[i]; B[i] = Rw2c[i]; }
    sign = -1.0;
  }
  for (int i = 0; i < 2; ++i)
    for (int j = 0; j < 3; ++j) {
      double a = (dz[3 * i] * A[j] + dz[3 * i + 1] * A[3 + j]) + dz[3 * i + 2] * A[6 + j];
      double b = (dz[3 * i] * B[j] + dz[3 * i + 1] * B[3 + j]) + dz[3 * i + 2] * B[6 + j];
      Hx[6 * i + j] = sign * a;
      Hx[6 * i + 3 + j] = sign * b;
      Hf[3 * i + j] = (dz[3 * i] * Rw2c[j] + dz[3 * i + 1] * Rw2c[3 + j]) + dz[3 * i + 2] * Rw2c[6 + j];
    }
  r[0] = zu - pc[0] / pc[2];
  r[1] = zv - pc[1] / pc[2];
  if (He) {
    // dpc_dxe = [R_w2c [p_bf]x R_b2w - R_bc [t_cb]x | -R_bc]   (:1152-1160)
    double St[9], T1[9], T2[9], T3[9];
    m3_skew(pbf, Sk);
    m3_mul(Rw2c, Sk, T1);
    m3_mul(T1, R, T2);
    m3_skew(tcb, St);
    m3_mul(Rbc, St, T3);
    for (int i = 0; i < 2; ++i)
      for (int j = 0; j < 3; ++j) {
        double e0 = T2[j] - T3[j], e1 = T2[3 + j] - T3[3 + j], e2 = T2[6 + j] - T3[6 + j];
        He[6 * i + j] = (dz[3 * i] * e0 + dz[3 * i + 1] * e1) + dz[3 * i + 2] * e2;
        He[6 * i + 3 + j] = -((dz[3 * i] * Rbc[j] + dz[3 * i + 1] * Rbc[3 + j]) + dz[3 * i + 2] * Rbc[6 + j]);
      }
  }
}

template <int TEAM, int MAXM, int MINB>
__global__ void __launch_bounds__(128, MINB) k_jac_gate(JacArgs a) {
  constexpr int R2 = 2 * MAXM;
  constexpr int LDQ = R2 + 1;
  constexpr int TEAM_DOUBLES = R2 * 6 + R2 * 3 + R2 + 4 + 3 * R2 * LDQ + R2;
  extern __shared__ double smem[];
  pdl_launch_dependents();           // per-candidate overlap: the large-list grid may be scheduled behind this one
  const int teams_per_block = blockDim.x / TEAM;
  const int team = threadIdx.x / TEAM;
  const int lane = threadIdx.x % TEAM;
  const int li = blockIdx.x * teams_per_block + team;
  if (li >= a.n_list) return;
  const int c = a.cand_list ? a.cand_list[li] : li;
  Cand cd;
  if (a.feat_off) {                  // direct mode: feature c of the caller's list
    const int o0 = a.feat_off[c], mm = a.feat_off[c + 1] - o0;
    int s_ = 1 << 30, e_ = -1;
    for (int k = 0; k < mm; ++k) {
      const int ci = a.obs_clone[o0 + k];
      s_ = min(s_, ci);
      e_ = max(e_, ci);
    }
    cd.filter = 0; cd.slot = c;
    cd.jac_off = o0; cd.jac_m = mm;
    cd.s_blk = s_; cd.e_blk = e_;
    cd.row_off = a.rowoff_f[c];
    cd.hblk_off = a.hblkoff_f[c];
  } else {
    cd = a.cand[c];
  }
  // everything above reads host-built lists only; below: triangulation results
  if (a.tri_done) {
    // launched behind k_triangulate with programmatic stream serialisation: every triangulation CTA is resident (or
    // done) by now, so waiting for this candidate's flag cannot deadlock; the other inputs (P, clones, pools) were
    // complete before k_triangulate started
    if (lane == 0) {
      int v;
      for (;;) {                     // relaxed polls (L2, no L1 invalidation), one acquire fence at the end
        asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(a.tri_done + c) : "memory");
        if (v == a.tri_epoch) break;
        __nanosleep(400);
      }
      asm volatile("fence.acq_rel.gpu;" ::: "memory");
    }
    team_sync<TEAM>();
  }
  const int st_in = a.tri_status_f ? a.tri_status_f[cd.slot] : __ldcg(a.status + c);   // (L2: written by another SM moments ago)
  if (a.tri_status_f && lane == 0) a.status[c] = st_in;      // status by candidate, as the one-pass flow leaves it
  if (!(st_in & ST_TRI_VALID)) {
    if (lane == 0) a.gamma[c] = -1.0;
    return;
  }
  double* sm = smem + (size_t)team * TEAM_DOUBLES;
  double* Hx = sm;                 // [2m][6]
  double* Hf = Hx + R2 * 6;        // [2m][3]  (Householder vectors below the diagonal)
  double* rr = Hf + R2 * 3;        // [2m]
  double* tau = rr + R2;           // [3] (+pad)
  double* QT = tau + 4;            // [2m][LDQ]   Q^T
  double* Mm = QT + R2 * LDQ;      // [2m][LDQ]   H P H^T, later S
  double* Tm = Mm + R2 * LDQ;      // [2m][LDQ]   Q2^T M
  double* yv = Tm + R2 * LDQ;      // [2m]        projected residual / solve vector

  const int m = cd.jac_m;
  const int n2 = 2 * m;
  const int r = n2 - 3;
  const double* clones = a.clones + (size_t)cd.filter * a.clone_stride;
  const double* imu = a.imu + (size_t)cd.filter * IM_STRIDE;
  const double* fp = a.fpos + ((size_t)cd.filter * a.fcap + cd.slot) * FP_STRIDE;
  const int* oc = a.obs_clone + cd.jac_off;
  const double* oz = a.obs_z + 2 * (size_t)cd.jac_off;
  const double* P = a.P + (size_t)cd.filter * a.p_stride;
  const int ldp = a.ldp;

  // ---- J1: one observation per thread
  for (int i = lane; i < m; i += TEAM) {
    double pw[3] = {__ldcg(fp), __ldcg(fp + 1), __ldcg(fp + 2)};
    double hx[12], hf[6], ri[2], he[12];
    measurement_jacobian(clones + (size_t)oc[i] * CL_STRIDE, imu + IM_RBC, imu + IM_TCB, pw,
                         oz[2 * i], oz[2 * i + 1], a.flags, hx, hf, ri, a.raw_He ? he : nullptr);
    for (int k = 0; k < 12; ++k) Hx[12 * i + k] = hx[k];
    for (int k = 0; k < 6; ++k) Hf[6 * i + k] = hf[k];
    rr[2 * i] = ri[0];
    rr[2 * i + 1] = ri[1];
    if (a.raw_Hx) {
      size_t o = (size_t)(cd.jac_off + i);
      for (int k = 0; k < 12; ++k) a.raw_Hx[12 * o + k] = hx[k];
      for (int k = 0; k < 6; ++k) a.raw_Hf[6 * o + k] = hf[k];
      a.raw_r[2 * o] = ri[0];
      a.raw_r[2 * o + 1] = ri[1];
      if (a.raw_He)
        for (int k = 0; k < 12; ++k) a.raw_He[12 * o + k] = he[k];
    }
  }
  team_sync<TEAM>();
  if (r < 1) {   // not enough rows for a projection (reference: rows <= cols)
    if (lane == 0) a.gamma[c] = -1.0;
    return;
  }

  // ---- Householder QR of H_f (2m x 3); first warp of the team, rows over lanes
  if (lane < 32) {
    for (int k = 0; k < 3; ++k) {
      double sig = 0.0;
      for (int i = k + 1 + lane; i < n2; i += 32) sig += Hf[3 * i + k] * Hf[3 * i + k];
      for (int o = 16; o > 0; o >>= 1) sig += __shfl_xor_sync(0xffffffffu, sig, o);
      double akk = Hf[3 * k + k];
      double t = 0.0, v0 = 1.0, mu = akk;
      if (sig > 0.0) {
        mu = sqrt(akk * akk + sig);
        v0 = (akk <= 0.0) ? (akk - mu) : (-sig / (akk + mu));
        t = 2.0 * v0 * v0 / (sig + v0 * v0);
      }
      __syncwarp();
      for (int i = k + 1 + lane; i < n2; i += 32) Hf[3 * i + k] = Hf[3 * i + k] / v0;
      if (lane == 0) { Hf[3 * k + k] = mu; tau[k] = t; }
      __syncwarp();
      for (int j = k + 1; j < 3; ++j) {
        double dot = 0.0;
        for (int i = k + 1 + lane; i < n2; i += 32) dot += Hf[3 * i + k] * Hf[3 * i + j];
        for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
        dot += Hf[3 * k + j];
        __syncwarp();
        for (int i = k + 1 + lane; i < n2; i += 32) Hf[3 * i + j] -= t * dot * Hf[3 * i + k];
        if (lane == 0) Hf[3 * k + j] -= t * dot;
        __syncwarp();
      }
    }
  }
  team_sync<TEAM>();

  // ---- Q^T = H3 H2 H1 applied to the identity, one column per thread
  for (int j = lane; j < n2; j += TEAM) {
    for (int i = 0; i < n2; ++i) QT[i * LDQ + j] = (i == j) ? 1.0 : 0.0;
    for (int k = 0; k < 3; ++k) {
      double dot = QT[k * LDQ + j];
      for (int i = k + 1; i < n2; ++i) dot += Hf[3 * i + k] * QT[i * LDQ + j];
      double s = tau[k] * dot;
      QT[k * LDQ + j] -= s;
      for (int i = k + 1; i < n2; ++i) QT[i * LDQ + j] -= s * Hf[3 * i + k];
    }
  }
  // ---- M = H_x P H_x^T from 2x2 blocks (upper block triangle, mirrored)
  for (int bp = lane; bp < m * m; bp += TEAM) {
    int i = bp / m, j = bp % m;
    if (j < i) continue;
    const double* Pij = P + (size_t)(ORCVIO_LEG + 6 * oc[i]) * ldp + (ORCVIO_LEG + 6 * oc[j]);
    const double* Ai = Hx + 12 * i;
    const double* Aj = Hx + 12 * j;
    double t0[6], t1[6];    // rows of A_i * P_ij
    for (int q = 0; q < 6; ++q) {
      double s0 = 0.0, s1 = 0.0;
      for (int p_ = 0; p_ < 6; ++p_) {
        double pv = Pij[(size_t)p_ * ldp + q];
        s0 += Ai[p_] * pv;
        s1 += Ai[6 + p_] * pv;
      }
      t0[q] = s0;
      t1[q] = s1;
    }
    double m00 = 0, m01 = 0, m10 = 0, m11 = 0;
    for (int q = 0; q < 6; ++q) {
      m00 += t0[q] * Aj[q];
      m01 += t0[q] * Aj[6 + q];
      m10 += t1[q] * Aj[q];
      m11 += t1[q] * Aj[6 + q];
    }
    Mm[(2 * i) * LDQ + 2 * j] = m00;
    Mm[(2 * i) * LDQ + 2 * j + 1] = m01;
    Mm[(2 * i + 1) * LDQ + 2 * j] = m10;
    Mm[(2 * i + 1) * LDQ + 2 * j + 1] = m11;
    if (j > i) {
      Mm[(2 * j) * LDQ + 2 * i] = m00;
      Mm[(2 * j + 1) * LDQ + 2 * i] = m01;
      Mm[(2 * j) * LDQ + 2 * i + 1] = m10;
      Mm[(2 * j + 1) * LDQ + 2 * i + 1] = m11;
    }
  }
  team_sync<TEAM>();

  // ---- Tm = Q2^T M  (r x 2m),  projected residual
  for (int e = lane; e < r * n2; e += TEAM) {
    int ro = e / n2, j = e % n2;
    const double* q = QT + (3 + ro) * LDQ;
    double s = 0.0;
    for (int k = 0; k < n2; ++k) s += q[k] * Mm[k * LDQ + j];
    Tm[ro * LDQ + j] = s;
  }
  for (int ro = lane; ro < r; ro += TEAM) {
    const double* q = QT + (3 + ro) * LDQ;
    double s = 0.0;
    for (int k = 0; k < n2; ++k) s += q[k] * rr[k];
    yv[ro] = s;
  }
  team_sync<TEAM>();
  // ---- S = Tm Q2 + sigma^2 I  (lower triangle, stored in Mm)
  for (int e = lane; e < r * r; e += TEAM) {
    int i = e / r, j = e % r;
    if (j > i) continue;
    const double* q = QT + (3 + j) * LDQ;
    double s = 0.0;
    for (int k = 0; k < n2; ++k) s += Tm[i * LDQ + k] * q[k];
    if (i == j) s += a.sigma2;
    Mm[i * LDQ + j] = s;
  }
  // keep the projected residual for the output before the solve overwrites it
  double* rproj = rr;   // rr no longer needed after yv was formed
  team_sync<TEAM>();
  for (int ro = lane; ro < r; ro += TEAM) rproj[ro] = yv[ro];
  // ---- Cholesky S = L L^T and forward solve; gamma = |L^-1 r'|^2
  for (int k = 0; k < r; ++k) {
    team_sync<TEAM>();
    if (lane == 0) Mm[k * LDQ + k] = sqrt(Mm[k * LDQ + k]);
    team_sync<TEAM>();
    double dk = Mm[k * LDQ + k];
    for (int i = k + 1 + lane; i < r; i += TEAM) Mm[i * LDQ + k] = Mm[i * LDQ + k] / dk;
    if (lane == 0) yv[k] = yv[k] / dk;
    team_sync<TEAM>();
    int rem = r - k - 1;
    for (int e = lane; e < rem * rem; e += TEAM) {
      int i = k + 1 + e / rem, j = k + 1 + e % rem;
      if (j <= i) Mm[i * LDQ + j] -= Mm[i * LDQ + k] * Mm[j * LDQ + k];
    }
    for (int i = k + 1 + lane; i < r; i += TEAM) yv[i] -= Mm[i * LDQ + k] * yv[k];
  }
  team_sync<TEAM>();
  double g = 0.0;
  for (int i = 0; i < r; ++i) g += yv[i] * yv[i];
  const bool pass = g < a.chi2[r];        // dof = 2m - 3 (< 500 always: m <= 32)
  if (lane == 0) {
    a.gamma[c] = g;
    a.status[c] = st_in | (pass ? ST_GATE_PASS : 0);
  }
  if (!pass || a.hblk == nullptr) return;

  // ---- projected rows H' = Q2^T H_x in compact form: r x 6(e - s + 1)
  const int w = 6 * (cd.e_blk - cd.s_blk + 1);
  double* hb = a.hblk + cd.hblk_off;
  for (int e = lane; e < r * w; e += TEAM) hb[e] = 0.0;
  team_sync<TEAM>();
  for (int e = lane; e < r * m * 6; e += TEAM) {
    int ro = e / (m * 6);
    int rem = e % (m * 6);
    int i = rem / 6, q = rem % 6;
    const double* qt = QT + (3 + ro) * LDQ;
    double v = qt[2 * i] * Hx[12 * i + q] + qt[2 * i + 1] * Hx[12 * i + 6 + q];
    hb[(size_t)ro * w + 6 * (oc[i] - cd.s_blk) + q] = v;
  }
  double* rb = a.rblk + cd.row_off + 0;   // caller offsets rblk per filter via cd.row_off base
  for (int ro = lane; ro < r; ro += TEAM) rb[ro] = rproj[ro];
}

template <int TEAM, int MAXM, int MINB>
static void launch_one(const JacArgs& a, cudaStream_t s) {
  if (a.n_list <= 0) return;
  constexpr int R2 = 2 * MAXM;
  constexpr int LDQ = R2 + 1;
  constexpr int TEAM_DOUBLES = R2 * 6 + R2 * 3 + R2 + 4 + 3 * R2 * LDQ + R2;
  const int threads = 128;
  const int tpb = threads / TEAM;
  size_t smem = (size_t)tpb * TEAM_DOUBLES * sizeof(double);
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(k_jac_gate<TEAM, MAXM, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    attr_set = true;
  }
  int blocks = (a.n_list + tpb - 1) / tpb;
  if (a.tri_done) {
    // per-candidate overlap: programmatic stream serialisation lets the grid be scheduled while the previous kernel
    // (k_triangulate, or the small-list k_jac_gate ahead of the large list) still runs; the flags order the data
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(blocks);
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, k_jac_gate<TEAM, MAXM, MINB>, a);
  } else {
    k_jac_gate<TEAM, MAXM, MINB><<<blocks, threads, smem, s>>>(a);
  }
  check_launch("k_jac_gate");
}

void launch_jac_gate(const JacArgs& small_list, const JacArgs& large_list, cudaStream_t s) {
  launch_one<32, 8, 4>(small_list, s);   // 128 registers, 4 CTAs per SM: fewest waves (measured)
  launch_one<128, ORCVIO_MAX_OBS, 1>(large_list, s);
}

}  // namespace ob

// Trajectory metrics on the device (SURVEY 8f(4)): the reference's logger, System::publishGroundtruth
// (ros_wrapper/src/orcvio/src/System.cpp:885-943), for a batch of trajectories at once.
//
// Per trajectory: the first estimated pose is aligned with the first ground-truth pose,
//     T_from_est_to_gt = T_gt(0) T_est(0)^-1,        T_corrected(k) = T_from_est_to_gt T_est(k),
// and every frame contributes  rmse_pos = |p_corrected - p_gt|  and
// rmse_ori = (180 / pi) 2 |vec(q_corrected (x) q_gt^-1)|  (Hamilton quaternions x, y, z, w: math_utils.hpp:79-93,
// 164-227); the logger's result file holds the running means of the two.  One CTA per trajectory, frames over the
// threads, fixed-order tree reduction.  Outputs per trajectory: mean orientation error (deg), mean position error (m),
// position RMSE (m), final position error (m).
#include "../../include/orcvio_b200.h"
#include "devmem.h"
#include "kernels.h"
#include "svd3.cuh"

namespace ob {

namespace {

__device__ __forceinline__ void quat_to_R(const double* q, double* R) {     // quaternionToRotation, math_utils.hpp:164-177
  const double qx = q[0], qy = q[1], qz = q[2], qw = q[3];
  R[0] = 1 - 2 * (qy * qy + qz * qz); R[1] = 2 * (qx * qy - qw * qz); R[2] = 2 * (qx * qz + qw * qy);
  R[3] = 2 * (qx * qy + qw * qz); R[4] = 1 - 2 * (qx * qx + qz * qz); R[5] = 2 * (qy * qz - qw * qx);
  R[6] = 2 * (qx * qz - qw * qy); R[7] = 2 * (qy * qz + qw * qx); R[8] = 1 - 2 * (qx * qx + qy * qy);
}

__device__ __forceinline__ void R_to_quat(const double* R, double* q) {     // rotationToQuaternion, math_utils.hpp:188-227
  const double tr = R[0] + R[4] + R[8];
  const double score[4] = {R[0], R[4], R[8], tr};
  int best = 0;
  for (int i = 1; i < 4; ++i)
    if (score[i] > score[best]) best = i;
  if (best == 0) {
    q[0] = sqrt(1 + 2 * R[0] - tr) / 2.0;
    q[1] = (R[1] + R[3]) / (4 * q[0]);
    q[2] = (R[2] + R[6]) / (4 * q[0]);
    q[3] = (R[7] - R[5]) / (4 * q[0]);
  } else if (best == 1) {
    q[1] = sqrt(1 + 2 * R[4] - tr) / 2.0;
    q[0] = (R[1] + R[3]) / (4 * q[1]);
    q[2] = (R[5] + R[7]) / (4 * q[1]);
    q[3] = (R[2] - R[6]) / (4 * q[1]);
  } else if (best == 2) {
    q[2] = sqrt(1 + 2 * R[8] - tr) / 2.0;
    q[0] = (R[2] + R[6]) / (4 * q[2]);
    q[1] = (R[5] + R[7]) / (4 * q[2]);
    q[3] = (R[3] - R[1]) / (4 * q[2]);
  } else {
    q[3] = sqrt(1 + tr) / 2.0;
    q[0] = (R[7] - R[5]) / (4 * q[3]);
    q[1] = (R[2] - R[6]) / (4 * q[3]);
    q[2] = (R[3] - R[1]) / (4 * q[3]);
  }
  if (q[3] < 0)
    for (int i = 0; i < 4; ++i) q[i] = -q[i];
  const double n = sqrt((q[0] * q[0] + q[1] * q[1]) + (q[2] * q[2] + q[3] * q[3]));
  for (int i = 0; i < 4; ++i) q[i] /= n;
}

}  // namespace

// est / gt: n_traj x n_frames x 7 (px py pz qx qy qz qw); out: n_traj x 4
__global__ void __launch_bounds__(128) k_trajectory_metrics(const double* __restrict__ est, const double* __restrict__ gt,
                                                            int n_frames, double* __restrict__ out) {
  __shared__ double red[3][128];
  __shared__ double Ta[12];                              // T_from_est_to_gt: R (9) | t (3)
  const int tr = blockIdx.x, tid = threadIdx.x;
  const double* e = est + (size_t)tr * n_frames * 7;
  const double* g = gt + (size_t)tr * n_frames * 7;
  if (tid == 0) {
    double Re[9], Rg[9];
    quat_to_R(e + 3, Re);
    quat_to_R(g + 3, Rg);
    m3_mulT(Rg, Re, Ta);                                 // R_gt R_est^T
    double t[3];
    m3_vec(Ta, e, t);
    for (int i = 0; i < 3; ++i) Ta[9 + i] = g[i] - t[i];  // p_gt - R p_est
  }
  __syncthreads();
  double s_ori = 0.0, s_pos = 0.0, s_sq = 0.0;
  for (int k = tid; k < n_frames; k += 128) {
    double Re[9], Rc[9], pc[3], qc[4];
    quat_to_R(e + 7 * k + 3, Re);
    m3_mul(Ta, Re, Rc);
    m3_vec(Ta, e + 7 * k, pc);
    const double dx = pc[0] + Ta[9] - g[7 * k], dy = pc[1] + Ta[10] - g[7 * k + 1], dz = pc[2] + Ta[11] - g[7 * k + 2];
    const double ep = sqrt(dx * dx + dy * dy + dz * dz);
    R_to_quat(Rc, qc);
    // q_corrected (x) q_gt^-1 (Hamilton product, math_utils.hpp:79-93; the inverse of a unit quaternion: conjugate / |q|^2)
    const double* qg = g + 7 * k + 3;
    const double n2 = (qg[0] * qg[0] + qg[1] * qg[1]) + (qg[2] * qg[2] + qg[3] * qg[3]);
    const double b0 = -qg[0] / n2, b1 = -qg[1] / n2, b2 = -qg[2] / n2, b3 = qg[3] / n2;
    double d0 = qc[3] * b0 - qc[2] * b1 + qc[1] * b2 + qc[0] * b3;
    double d1 = qc[2] * b0 + qc[3] * b1 - qc[0] * b2 + qc[1] * b3;
    double d2 = -qc[1] * b0 + qc[0] * b1 + qc[3] * b2 + qc[2] * b3;
    double d3 = -qc[0] * b0 - qc[1] * b1 - qc[2] * b2 + qc[3] * b3;
    const double dn = sqrt((d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3));
    d0 /= dn; d1 /= dn; d2 /= dn;
    const double eo = (180.0 / 3.14159265358979323846) * 2 * sqrt(d0 * d0 + d1 * d1 + d2 * d2);
    s_ori += eo;
    s_pos += ep;
    s_sq += ep * ep;
    if (k == n_frames - 1) out[4 * (size_t)tr + 3] = ep;
  }
  red[0][tid] = s_ori; red[1][tid] = s_pos; red[2][tid] = s_sq;
  __syncthreads();
  for (int o = 64; o > 0; o >>= 1) {
    if (tid < o)
      for (int q = 0; q < 3; ++q) red[q][tid] += red[q][tid + o];
    __syncthreads();
  }
  if (tid == 0) {
    out[4 * (size_t)tr + 0] = red[0][0] / n_frames;
    out[4 * (size_t)tr + 1] = red[1][0] / n_frames;
    out[4 * (size_t)tr + 2] = sqrt(red[2][0] / n_frames);
  }
}

int trajectory_metrics(const double* est_pose7, const double* gt_pose7, int n_traj, int n_frames, double* out4) {
  if (n_traj < 1 || n_frames < 1) return ORCVIO_ERR_ARG;
  const size_t np = (size_t)n_traj * n_frames * 7, nb = np * sizeof(double);
  DeviceBuf<double> dE, dG, dO;
  if (!dE.alloc(np) || !dG.alloc(np) || !dO.alloc((size_t)n_traj * 4))
    return ORCVIO_ERR_CUDA;
  cudaMemcpy(dE.get(), est_pose7, nb, cudaMemcpyHostToDevice);
  cudaMemcpy(dG.get(), gt_pose7, nb, cudaMemcpyHostToDevice);
  k_trajectory_metrics<<<n_traj, 128>>>(dE.get(), dG.get(), n_frames, dO.get());
  check_launch("k_trajectory_metrics");
  const cudaError_t e = cudaMemcpy(out4, dO.get(), dO.bytes(), cudaMemcpyDeviceToHost);
  return e == cudaSuccess ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

// ---------------------------------------------------------------------------------------------------------------------
// KITTI-style relative error for a batch of trajectories (SURVEY 8f(4), second half): what the reference's
// python_scripts/trajectory_eval/traj_eval.py:61-90 computes through its vendored rpg_trajectory_evaluation
// (compute_trajectory_errors.py:10-67 compute_relative_error with T_cm = I and scale 1, trajectory_utils.py:11-37,
// trajectory.py:341-377 with max_dist_diff = 0.2 x length, :309-339 for the "TransError(%)" summary).
// One CTA per (sub-trajectory length, trajectory):
//   1. distance from the start along the GROUND TRUTH (a sequential cumulative sum, as numpy.cumsum);
//   2. for every start index the FIRST later index whose distance is closest to d + length within the tolerance
//      (threads over the starts, each scans forward until the distances pass the tolerance);
//   3. the matches are compacted IN ORDER and entry k is paired with start k -- the reference drops the starts without a
//      match from the list and then enumerates it (compute_trajectory_errors.py:30-31); kept as it is;
//   4. per pair E = (T_gt1^-1 T_gt2)^-1 (T_es1^-1 T_es2): |t(E)|, |t(E)| / length in %, angle(E) in degrees and per
//      metre (the rotation of E into the world frame, :45-48, changes neither); summed in sample order by one thread.
// Fewer than two samples: nothing is computed (the reference returns empty arrays).
// out: n_traj x n_len x 4 = (samples, mean translation error %, mean rotation error deg / m, mean translation error m).
namespace {

__device__ __forceinline__ void quat_to_R_rpg(const double* q, double* R) {      // transformations.py:1410-1429, x y z w
  double v[4] = {q[0], q[1], q[2], q[3]};
  const double nq = (v[0] * v[0] + v[1] * v[1]) + (v[2] * v[2] + v[3] * v[3]);
  if (nq < 8.881784197001252e-16) {                                              // _EPS = 4 eps
    for (int i = 0; i < 9; ++i) R[i] = (i % 4 == 0) ? 1.0 : 0.0;
    return;
  }
  const double sc = sqrt(2.0 / nq);
  for (int i = 0; i < 4; ++i) v[i] *= sc;
  auto Q = [&](int i, int j) { return v[i] * v[j]; };
  R[0] = 1.0 - Q(1, 1) - Q(2, 2); R[1] = Q(0, 1) - Q(2, 3); R[2] = Q(0, 2) + Q(1, 3);
  R[3] = Q(0, 1) + Q(2, 3); R[4] = 1.0 - Q(0, 0) - Q(2, 2); R[5] = Q(1, 2) - Q(0, 3);
  R[6] = Q(0, 2) - Q(1, 3); R[7] = Q(1, 2) + Q(0, 3); R[8] = 1.0 - Q(0, 0) - Q(1, 1);
}

// relative motion T1^-1 T2 of two poses (p, q): R = R1^T R2, t = R1^T (p2 - p1)
__device__ __forceinline__ void rel_motion(const double* a, const double* b, double* R, double* t) {
  double R1[9], R2[9];
  quat_to_R_rpg(a + 3, R1);
  quat_to_R_rpg(b + 3, R2);
  m3_Tmul(R1, R2, R);
  const double d[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]};
  m3_Tvec(R1, d, t);
}

}  // namespace

__global__ void __launch_bounds__(256) k_kitti_relative_error(const double* __restrict__ est, const double* __restrict__ gt,
                                                              int n_frames, const double* __restrict__ lengths, int n_len,
                                                              const double* __restrict__ scale, double* __restrict__ out) {
  extern __shared__ double ksm[];
  double* dist = ksm;                               // [n_frames]
  double* v_perc = dist + n_frames;                 // [n_frames] per-sample values, summed in order at the end
  double* v_rot = v_perc + n_frames;
  double* v_tr = v_rot + n_frames;
  int* match = reinterpret_cast<int*>(v_tr + n_frames);   // [n_frames]
  int* comps = match + n_frames;                    // [n_frames]
  __shared__ int s_k;
  const int li = blockIdx.x, tr = blockIdx.y, tid = threadIdx.x, nt = blockDim.x;
  const double* E = est + (size_t)tr * n_frames * 7;
  const double* G = gt + (size_t)tr * n_frames * 7;
  const double L = lengths[li], tol = 0.2 * L;
  if (tid == 0) {
    double acc = 0.0;
    dist[0] = 0.0;
    for (int k = 1; k < n_frames; ++k) {
      const double dx = G[7 * k] - G[7 * (k - 1)], dy = G[7 * k + 1] - G[7 * (k - 1) + 1], dz = G[7 * k + 2] - G[7 * (k - 1) + 2];
      acc += sqrt((dx * dx + dy * dy) + dz * dz);
      dist[k] = acc;
    }
  }
  __syncthreads();
  for (int idx = tid; idx < n_frames; idx += nt) {
    const double target = dist[idx] + L;
    int best = -1;
    double err = tol;
    for (int i = idx; i < n_frames; ++i) {
      const double e = fabs(dist[i] - target);
      if (e < err) { best = i; err = e; }
      else if (dist[i] - target > err) break;
    }
    match[idx] = best;
  }
  __syncthreads();
  if (tid == 0) {
    int k = 0;
    for (int idx = 0; idx < n_frames; ++idx)
      if (match[idx] >= 0) comps[k++] = match[idx];
    s_k = k;
  }
  __syncthreads();
  const int K = s_k;
  double* o = out + ((size_t)tr * n_len + li) * 4;
  if (K < 2) {
    if (tid == 0) { o[0] = 0.0; o[1] = 0.0; o[2] = 0.0; o[3] = 0.0; }
    return;
  }
  for (int k = tid; k < K; k += nt) {
    const int c = comps[k];
    double Rc[9], tc[3], Rm[9], tm[3];
    rel_motion(E + 7 * (size_t)k, E + 7 * (size_t)c, Rc, tc);       // T_c1_c2
    if (scale) { const double sc = scale[tr]; tc[0] *= sc; tc[1] *= sc; tc[2] *= sc; }     // (the sim3 alignment's scale, :33)
    rel_motion(G + 7 * (size_t)k, G + 7 * (size_t)c, Rm, tm);       // T_m1_m2
    // E = T_m1_m2^-1 T_c1_c2: R = Rm^T Rc, t = Rm^T (tc - tm)
    double Re[9], te[3];
    m3_Tmul(Rm, Rc, Re);
    const double d[3] = {tc[0] - tm[0], tc[1] - tm[1], tc[2] - tm[2]};
    m3_Tvec(Rm, d, te);
    const double tn = sqrt((te[0] * te[0] + te[1] * te[1]) + te[2] * te[2]);
    const double ang = acos(fmin(1.0, fmax(-1.0, ((Re[0] + Re[4] + Re[8]) - 1.0) / 2.0))) * 180.0 / 3.14159265358979323846;
    v_tr[k] = tn;
    v_perc[k] = tn / L * 100.0;
    v_rot[k] = ang / L;
  }
  __syncthreads();
  if (tid < 3) {
    const double* v = tid == 0 ? v_perc : tid == 1 ? v_rot : v_tr;
    double s = 0.0;
    for (int k = 0; k < K; ++k) s += v[k];
    o[1 + tid] = s / K;
  }
  if (tid == 3) o[0] = (double)K;
}

int kitti_relative_error(const double* est_pose7, const double* gt_pose7, int n_traj, int n_frames, const double* lengths,
                         int n_len, const double* scale, double* out4, double* trans_error_pct) {
  if (n_traj < 1 || n_frames < 2 || n_len < 1 || n_frames > 4096) return ORCVIO_ERR_ARG;
  const size_t np = (size_t)n_traj * n_frames * 7, nb = np * sizeof(double);
  DeviceBuf<double> dE, dG, dL, dO, dS;
  const size_t no = (size_t)n_traj * n_len * 4;
  if (!dE.alloc(np) || !dG.alloc(np) || !dL.alloc(n_len) || !dO.alloc(no) ||
      !dS.alloc(n_traj))
    return ORCVIO_ERR_CUDA;
  if (scale) cudaMemcpy(dS.get(), scale, n_traj * sizeof(double), cudaMemcpyHostToDevice);
  cudaMemcpy(dE.get(), est_pose7, nb, cudaMemcpyHostToDevice);
  cudaMemcpy(dG.get(), gt_pose7, nb, cudaMemcpyHostToDevice);
  cudaMemcpy(dL.get(), lengths, n_len * sizeof(double), cudaMemcpyHostToDevice);
  const size_t smem = (size_t)n_frames * (4 * sizeof(double) + 2 * sizeof(int));
  cudaFuncSetAttribute(k_kitti_relative_error, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  k_kitti_relative_error<<<dim3(n_len, n_traj), 256, smem>>>(dE.get(), dG.get(), n_frames, dL.get(), n_len,
                                                            scale ? dS.get() : nullptr, dO.get());
  check_launch("k_kitti_relative_error");
  const cudaError_t e = cudaMemcpy(out4, dO.get(), no * sizeof(double), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) return ORCVIO_ERR_CUDA;
  if (trans_error_pct)                 // write_kitti_errors_to_yaml: sum of the per-length means / (valid lengths + 1e-5)
    for (int t = 0; t < n_traj; ++t) {
      double tot = 0.0;
      int valid = 0;
      for (int l = 0; l < n_len; ++l) {
        const double* o = out4 + ((size_t)t * n_len + l) * 4;
        if (o[0] > 0.0) { ++valid; tot += o[1]; }
      }
      trans_error_pct[t] = tot / (valid + 1e-5);
    }
  return ORCVIO_OK;
}

// Umeyama alignment of an estimated trajectory onto its ground truth over all frames and the absolute translation
// error behind it -- Trajectory.align_trajectory / compute_absolute_error of the same package (trajectory.py:211-275,
// align_utils.py:79-110, align_trajectory.py:27-79, compute_trajectory_errors.py:70-72): gt ~ s R est + t with s = 1
// for "se3".  One CTA per trajectory: means, the 3 x 3 correlation and sigma^2 by fixed-order reductions, the SVD on
// one thread, then the errors.  out15 per trajectory: s, R (9, row-major), t (3), mean |e|, rmse |e| -- the mean is what
// write_kitti_errors_to_yaml labels "RMSE(m)".
__global__ void __launch_bounds__(128) k_umeyama_ate(const double* __restrict__ est, const double* __restrict__ gt, int n_frames,
                                                     int known_scale, double* __restrict__ out) {
  __shared__ double red[13][128];
  __shared__ double sh[32];
  const int tr = blockIdx.x, tid = threadIdx.x;
  const double* E = est + (size_t)tr * n_frames * 7;
  const double* G = gt + (size_t)tr * n_frames * 7;
  auto reduce = [&](int nq) {                       // red[q][0] <- sum over the threads, fixed tree
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
      if (tid < o)
        for (int q = 0; q < nq; ++q) red[q][tid] += red[q][tid + o];
      __syncthreads();
    }
  };
  double a[13];
  for (int q = 0; q < 6; ++q) a[q] = 0.0;
  for (int k = tid; k < n_frames; k += 128)
    for (int c = 0; c < 3; ++c) { a[c] += G[7 * (size_t)k + c]; a[3 + c] += E[7 * (size_t)k + c]; }
  for (int q = 0; q < 6; ++q) red[q][tid] = a[q];
  reduce(6);
  if (tid < 6) sh[tid] = red[tid][0] / n_frames;    // mu_M (gt), mu_D (est)
  __syncthreads();
  const double mm[3] = {sh[0], sh[1], sh[2]}, md[3] = {sh[3], sh[4], sh[5]};
  for (int q = 0; q < 10; ++q) a[q] = 0.0;
  for (int k = tid; k < n_frames; k += 128) {
    double m[3], d[3];
    for (int c = 0; c < 3; ++c) { m[c] = G[7 * (size_t)k + c] - mm[c]; d[c] = E[7 * (size_t)k + c] - md[c]; }
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) a[3 * i + j] += m[i] * d[j];
    a[9] += (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2];
  }
  __syncthreads();
  for (int q = 0; q < 10; ++q) red[q][tid] = a[q];
  reduce(10);
  if (tid == 0) {
    double Cm[9], U[9], S[3], V[9], VUt[9];
    for (int i = 0; i < 9; ++i) Cm[i] = red[i][0] / n_frames;
    const double sigma2 = red[9][0] / n_frames;
    svd3::svd3_hestenes(Cm, U, S, V);               // C = U diag(S) V^T
    // det(U) det(V) < 0 -> flip the last singular direction; R = U diag(1, 1, f) V^T
    const double f = (svd3::det3(U) * svd3::det3(V) < 0) ? -1.0 : 1.0;
    double R[9];
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) R[3 * i + j] = (U[3 * i] * V[3 * j] + U[3 * i + 1] * V[3 * j + 1]) + f * U[3 * i + 2] * V[3 * j + 2];
    const double sc = known_scale ? 1.0 : ((S[0] + S[1]) + f * S[2]) / sigma2;
    double Rd[3];
    m3_vec(R, md, Rd);
    sh[6] = sc;
    for (int i = 0; i < 9; ++i) sh[7 + i] = R[i];
    for (int i = 0; i < 3; ++i) sh[16 + i] = mm[i] - sc * Rd[i];
    (void)VUt;
  }
  __syncthreads();
  const double sc = sh[6];
  double s1 = 0.0, s2 = 0.0;
  for (int k = tid; k < n_frames; k += 128) {
    double pe[3], Rp[3];
    for (int c = 0; c < 3; ++c) pe[c] = E[7 * (size_t)k + c];
    m3_vec(sh + 7, pe, Rp);
    double e2 = 0.0;
    for (int c = 0; c < 3; ++c) { const double d = G[7 * (size_t)k + c] - (sc * Rp[c] + sh[16 + c]); e2 += d * d; }
    s1 += sqrt(e2);
    s2 += e2;
  }
  __syncthreads();
  red[0][tid] = s1; red[1][tid] = s2;
  reduce(2);
  if (tid == 0) {
    double* o = out + 15 * (size_t)tr;
    for (int i = 0; i < 13; ++i) o[i] = sh[6 + i];
    o[13] = red[0][0] / n_frames;
    o[14] = sqrt(red[1][0] / n_frames);
  }
}

int umeyama_ate(const double* est_pose7, const double* gt_pose7, int n_traj, int n_frames, int known_scale, double* out15) {
  if (n_traj < 1 || n_frames < 3) return ORCVIO_ERR_ARG;
  const size_t np = (size_t)n_traj * n_frames * 7, nb = np * sizeof(double);
  DeviceBuf<double> dE, dG, dO;
  if (!dE.alloc(np) || !dG.alloc(np) || !dO.alloc((size_t)n_traj * 15))
    return ORCVIO_ERR_CUDA;
  cudaMemcpy(dE.get(), est_pose7, nb, cudaMemcpyHostToDevice);
  cudaMemcpy(dG.get(), gt_pose7, nb, cudaMemcpyHostToDevice);
  k_umeyama_ate<<<n_traj, 128>>>(dE.get(), dG.get(), n_frames, known_scale, dO.get());
  check_launch("k_umeyama_ate");
  const cudaError_t e = cudaMemcpy(out15, dO.get(), dO.bytes(), cudaMemcpyDeviceToHost);
  return e == cudaSuccess ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

}  // namespace ob

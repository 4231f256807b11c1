// Filter consistency on the device: the covariance the filter reports against the errors it makes.
//
// k_capture_imu_cov (queued by Batch::replay after every frame): the leading 15 x 15 block of each filter's resident
// covariance -- error state [theta, v, p, b_g, b_a] -- into a device history [filter, frame].
//
// k_nees (one warp per (trajectory, frame) sample): the error of the estimate against the truth under the filter's own
// retraction (incrementState_IMUCam, src/orcvio.cpp:4468-4567):
//   orientation  R = Exp(dtheta) R_est  (use_larvio_flag || use_left_perturbation_flag)  ->  dtheta = Log(R R_est^T)
//                R = R_est Exp(dtheta)  (otherwise)                                      ->  dtheta = Log(R_est^T R)
//   v, p, b_g, b_a additive: d = true - est.
// The 15 x 15 block is factored once, P' = L L^T, in the order [theta, p, v, b_g, b_a]: theta, the pose [theta, p], the
// navigation state [theta, p, v] and the full IMU state are then leading blocks, and with y = L^-1 e' their NEES are
// prefix sums of y^2.  v and p alone take two 3 x 3 factorisations of their own diagonal blocks.  Row (8 doubles):
// NEES theta, v, p, pose, navigation, full, then |dtheta| in degrees and |dp| in metres; all NaN when an input is not
// finite or the block is not positive definite (a pivot <= 0).  Only the lower triangle of the (permuted) block is read.
//
// k_nees_summary (one CTA per frame): over the valid trajectories (finite full NEES), the ANEES of the six blocks, the
// RMS orientation (deg) and position (m) errors and the count.  Each thread sums a fixed stride of trajectories, then a
// fixed tree over the threads: the result depends only on the rows, bit for bit.
#include <cmath>

#include "../../include/orcvio_b200.h"
#include "devmem.h"
#include "kernels.h"

namespace ob {

namespace {

constexpr int NEES_WARPS = 8;          // samples per CTA of k_nees
constexpr int SUM_THREADS = 256;

// [theta, v, p, b_g, b_a] <-> [theta, p, v, b_g, b_a] (the permutation is its own inverse)
__device__ __forceinline__ int perm15(int n) { return (n >= 3 && n < 6) ? n + 3 : (n >= 6 && n < 9) ? n - 3 : n; }

// Log of a rotation matrix (row-major): the angle from atan2(|w|, (tr - 1) / 2), w = vee(R - R^T) / 2 = sin(angle) axis;
// near pi the axis comes from the symmetric part, R + R^T = 2 cos I + 2 (1 - cos) n n^T, with the sign of w.
__device__ void so3_log(const double* R, double* out) {
  const double w[3] = {0.5 * (R[7] - R[5]), 0.5 * (R[2] - R[6]), 0.5 * (R[3] - R[1])};
  const double c = 0.5 * ((R[0] + R[4] + R[8]) - 1.0);
  const double s = sqrt((w[0] * w[0] + w[1] * w[1]) + w[2] * w[2]);
  const double th = atan2(s, c);
  if (c > -0.9) {
    const double f = s > 0.0 ? th / s : 1.0;
    for (int k = 0; k < 3; ++k) out[k] = f * w[k];
    return;
  }
  double B[9];                                          // n n^T = ((R + R^T) / 2 - c I) / (1 - c)
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) B[3 * i + j] = (0.5 * (R[3 * i + j] + R[3 * j + i]) - (i == j ? c : 0.0)) / (1.0 - c);
  int k = 0;
  if (B[4] > B[0]) k = 1;
  if (B[8] > B[4 * k]) k = 2;
  const double r = sqrt(B[4 * k]);
  double n[3] = {B[3 * k] / r, B[3 * k + 1] / r, B[3 * k + 2] / r};
  const double nn = sqrt((n[0] * n[0] + n[1] * n[1]) + n[2] * n[2]);
  const double sg = ((n[0] * w[0] + n[1] * w[1]) + n[2] * w[2]) < 0.0 ? -1.0 : 1.0;
  for (int q = 0; q < 3; ++q) out[q] = sg * th * n[q] / nn;
}

// e^T B^-1 e of a 3 x 3 block (lower triangle of rows / columns b0 .. b0 + 2 of the 15 x 15 A), NaN if not PD
__device__ double nees3(const double* A, int b0, const double* e) {
  auto a = [&](int i, int j) { return A[(b0 + i) * 15 + b0 + j]; };
  const double d0 = a(0, 0);
  if (!(d0 > 0.0)) return NAN;
  const double l00 = sqrt(d0), l10 = a(1, 0) / l00, l20 = a(2, 0) / l00;
  const double d1 = a(1, 1) - l10 * l10;
  if (!(d1 > 0.0)) return NAN;
  const double l11 = sqrt(d1), l21 = (a(2, 1) - l20 * l10) / l11;
  const double d2 = a(2, 2) - l20 * l20 - l21 * l21;
  if (!(d2 > 0.0)) return NAN;
  const double l22 = sqrt(d2);
  const double y0 = e[b0] / l00, y1 = (e[b0 + 1] - l10 * y0) / l11, y2 = (e[b0 + 2] - l20 * y0 - l21 * y1) / l22;
  return (y0 * y0 + y1 * y1) + y2 * y2;
}

}  // namespace

__global__ void __launch_bounds__(128) k_capture_imu_cov(const double* __restrict__ P, size_t p_stride, int ldp,
                                                         double* __restrict__ hist, int n_frames, int frame) {
  const double* Pi = P + (size_t)blockIdx.x * p_stride;
  double* h = hist + ((size_t)blockIdx.x * n_frames + frame) * 225;
  for (int k = threadIdx.x; k < 225; k += blockDim.x) {
    const int r = k / 15, c = k - 15 * r;
    h[k] = Pi[(size_t)r * ldp + c];
  }
}

void launch_capture_imu_cov(const double* P, size_t p_stride, int ldp, int n_filters, double* hist, int n_frames,
                            int frame, cudaStream_t s) {
  k_capture_imu_cov<<<n_filters, 128, 0, s>>>(P, p_stride, ldp, hist, n_frames, frame);
  check_launch("k_capture_imu_cov");
}

// est / gt: n x 17 (t, p, q xyzw, v, b_g, b_a), cov: n x 225 (error state [theta, v, p, b_g, b_a]), out: n x 8
__global__ void __launch_bounds__(NEES_WARPS * 32) k_nees(const double* __restrict__ est, const double* __restrict__ gt,
                                                          const double* __restrict__ cov, long long n, int left,
                                                          double* __restrict__ out) {
  __shared__ double sA[NEES_WARPS][225];
  __shared__ double sE[NEES_WARPS][16];
  __shared__ double sX[NEES_WARPS][4];               // NEES p, NEES v, |dtheta| deg, |dp| m
  const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long s = (long long)blockIdx.x * NEES_WARPS + wi;
  if (s >= n) return;
  double* A = sA[wi];
  double* e = sE[wi];
  const double* C = cov + (size_t)s * 225;
  const double* E = est + (size_t)s * 17;
  const double* G = gt + (size_t)s * 17;
  bool bad = false;
  for (int k = lane; k < 225; k += 32) {             // A = P' (permuted), coalesced over the lanes
    const double v = C[k];
    bad |= !isfinite(v);
    const int r = k / 15, c = k - 15 * r;
    A[perm15(r) * 15 + perm15(c)] = v;
  }
  if (lane < 17) bad |= !(isfinite(E[lane]) && isfinite(G[lane]));
  bad = __any_sync(0xffffffffu, bad);
  double* o = out + (size_t)s * 8;
  if (bad) {
    if (lane < 8) o[lane] = NAN;
    return;
  }
  if (lane == 0) {
    double Re[9], Rg[9], D[9], dth[3];
    quat_xyzw_to_R(E + 4, Re);
    quat_xyzw_to_R(G + 4, Rg);
    if (left) m3_mulT(Rg, Re, D);                    // R R_est^T
    else m3_Tmul(Re, Rg, D);                         // R_est^T R
    so3_log(D, dth);
    for (int k = 0; k < 3; ++k) {
      e[k] = dth[k];
      e[3 + k] = G[1 + k] - E[1 + k];                // p
      e[6 + k] = G[8 + k] - E[8 + k];                // v
      e[9 + k] = G[11 + k] - E[11 + k];              // b_g
      e[12 + k] = G[14 + k] - E[14 + k];             // b_a
    }
    sX[wi][2] = v3_norm(dth) * (180.0 / 3.14159265358979323846);
    sX[wi][3] = v3_norm(e + 3);
  }
  __syncwarp();
  if (lane == 1) sX[wi][0] = nees3(A, 3, e);         // p alone
  if (lane == 2) sX[wi][1] = nees3(A, 6, e);         // v alone
  __syncwarp();
  // right-looking Cholesky of the lower triangle, columns in order; the pivot test is warp-uniform (same shared value)
  bool pd = true;
  for (int j = 0; j < 15; ++j) {
    const double d = A[j * 15 + j];
    __syncwarp();
    if (!(d > 0.0)) { pd = false; break; }
    const double ljj = sqrt(d);
    if (lane == j) A[j * 15 + j] = ljj;
    else if (lane > j && lane < 15) A[lane * 15 + j] /= ljj;
    __syncwarp();
    for (int idx = lane; idx < 225; idx += 32) {
      const int i = idx / 15, k = idx - 15 * i;
      if (k > j && k <= i) A[idx] -= A[i * 15 + j] * A[k * 15 + j];
    }
    __syncwarp();
  }
  if (lane != 0) return;
  if (!pd) {
    for (int k = 0; k < 8; ++k) o[k] = NAN;
    return;
  }
  // y = L^-1 e' in place of e' (entry i of e' is last read when y_i is formed); prefix sums of y^2 at 3, 6, 9, 15
  double acc = 0.0, pre[3] = {0.0, 0.0, 0.0};
  for (int i = 0; i < 15; ++i) {
    double t = e[i];
    for (int k = 0; k < i; ++k) t -= A[i * 15 + k] * e[k];
    t /= A[i * 15 + i];
    e[i] = t;
    acc += t * t;
    if (i == 2) pre[0] = acc;
    if (i == 5) pre[1] = acc;
    if (i == 8) pre[2] = acc;
  }
  o[0] = pre[0];          // theta
  o[1] = sX[wi][1];       // v
  o[2] = sX[wi][0];       // p
  o[3] = pre[1];          // pose [theta, p]
  o[4] = pre[2];          // navigation [theta, p, v]
  o[5] = acc;             // full IMU state
  o[6] = sX[wi][2];
  o[7] = sX[wi][3];
}

// nees: n_traj x n_frames x 8; out: n_frames x 9
__global__ void __launch_bounds__(SUM_THREADS) k_nees_summary(const double* __restrict__ nees, int n_traj, int n_frames,
                                                              double* __restrict__ out) {
  __shared__ double red[9][SUM_THREADS];
  const int f = blockIdx.x, tid = threadIdx.x;
  double a[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int t = tid; t < n_traj; t += SUM_THREADS) {
    const double* r = nees + ((size_t)t * n_frames + f) * 8;
    if (!isfinite(r[5])) continue;
    for (int q = 0; q < 6; ++q) a[q] += r[q];
    a[6] += r[6] * r[6];
    a[7] += r[7] * r[7];
    a[8] += 1.0;
  }
  for (int q = 0; q < 9; ++q) red[q][tid] = a[q];
  __syncthreads();
  for (int w = SUM_THREADS / 2; w > 0; w >>= 1) {
    if (tid < w)
      for (int q = 0; q < 9; ++q) red[q][tid] += red[q][tid + w];
    __syncthreads();
  }
  if (tid == 0) {
    double* o = out + (size_t)f * 9;
    const double cnt = red[8][0];
    for (int q = 0; q < 6; ++q) o[q] = cnt > 0 ? red[q][0] / cnt : NAN;
    o[6] = cnt > 0 ? sqrt(red[6][0] / cnt) : NAN;
    o[7] = cnt > 0 ? sqrt(red[7][0] / cnt) : NAN;
    o[8] = cnt;
  }
}

static bool have_device() {
  int ndev = 0;
  return cudaGetDeviceCount(&ndev) == cudaSuccess && ndev > 0;
}

int nees_summary(const double* nees8, int n_traj, int n_frames, double* summary9) {
  if (n_traj < 1 || n_frames < 1 || !nees8 || !summary9) return ORCVIO_ERR_ARG;
  if (!have_device()) return ORCVIO_ERR_NO_DEVICE;
  const size_t nr = (size_t)n_traj * n_frames * 8, ns = (size_t)n_frames * 9;
  DeviceBuf<double> dN, dS;
  if (!dN.alloc(nr) || !dS.alloc(ns)) return ORCVIO_ERR_CUDA;
  cudaMemcpy(dN.get(), nees8, nr * sizeof(double), cudaMemcpyHostToDevice);
  k_nees_summary<<<n_frames, SUM_THREADS>>>(dN.get(), n_traj, n_frames, dS.get());
  check_launch("k_nees_summary");
  const cudaError_t e = cudaMemcpy(summary9, dS.get(), ns * sizeof(double), cudaMemcpyDeviceToHost);
  return e == cudaSuccess ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

int trajectory_nees(const double* est17, const double* gt17, const double* cov15, int n_traj, int n_frames, int flags,
                    double* nees8, double* summary9) {
  if (n_traj < 1 || n_frames < 1 || !est17 || !gt17 || !cov15 || !nees8) return ORCVIO_ERR_ARG;
  if (!have_device()) return ORCVIO_ERR_NO_DEVICE;
  const long long n = (long long)n_traj * n_frames;
  const size_t ns = summary9 ? (size_t)n_frames * 9 : 0;
  DeviceBuf<double> dE, dG, dC, dO, dS;
  if (!dE.alloc(n * 17) || !dG.alloc(n * 17) || !dC.alloc(n * 225) || !dO.alloc(n * 8) || !dS.alloc(ns))
    return ORCVIO_ERR_CUDA;
  cudaMemcpy(dE.get(), est17, n * 17 * sizeof(double), cudaMemcpyHostToDevice);
  cudaMemcpy(dG.get(), gt17, n * 17 * sizeof(double), cudaMemcpyHostToDevice);
  cudaMemcpy(dC.get(), cov15, n * 225 * sizeof(double), cudaMemcpyHostToDevice);
  k_nees<<<(unsigned)((n + NEES_WARPS - 1) / NEES_WARPS), NEES_WARPS * 32>>>(dE.get(), dG.get(), dC.get(), n,
                                                                          (flags & 3) != 0, dO.get());
  check_launch("k_nees");
  if (ns) {
    k_nees_summary<<<n_frames, SUM_THREADS>>>(dO.get(), n_traj, n_frames, dS.get());
    check_launch("k_nees_summary");
  }
  cudaError_t e = cudaMemcpy(nees8, dO.get(), n * 8 * sizeof(double), cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && ns) e = cudaMemcpy(summary9, dS.get(), ns * sizeof(double), cudaMemcpyDeviceToHost);
  return e == cudaSuccess ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

}  // namespace ob

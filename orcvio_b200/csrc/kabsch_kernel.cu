// Object pose initialisation, first step (SURVEY 8f rank 2): the similarity / Kabsch fit of
// ObjectFeatureInitializer::single_object_initialization without RANSAC
// (src/obj/ObjectFeatureInitializer.cpp:99-111: findTransform :265-341, then poseSE32SE2
// include/orcvio/utils/se3_ops.hpp:272-300 when estimate_SE2_pose_flag is set), for a batch of objects:
// object o has the triangulated keypoints world[off[o] .. off[o+1]) and the matching mean-shape keypoints.
//
// One thread per object (an object has at most a dozen keypoints; the batch dimension is the parallelism).  The
// reference takes Eigen's JacobiSVD of the 3 x 3 cross-covariance; here a one-sided Jacobi (Hestenes) SVD: the columns
// of Cov are rotated until they are orthogonal, which keeps small singular values accurate, and a rank-2 covariance
// (coplanar keypoints: src/tests/test_kabsch.cpp test_planar) is completed with the cross product of the two leading
// left vectors -- the rotation V diag(1, 1, det(V U^T)) U^T does not depend on the sign of that third vector.
#include "../../include/orcvio_b200.h"
#include "devmem.h"
#include "kernels.h"
#include "svd3.cuh"

namespace ob {

namespace {

using svd3::svd3_hestenes;
using svd3::det3;

}  // namespace

// mean / world: 3 doubles per point, points of object o at off[o] .. off[o+1]; out: 16 doubles (row-major 4 x 4) per
// object; ok[o] = 0 when the object has fewer than 2 points or a degenerate polyline (the reference divides by zero)
__global__ void k_kabsch(const double* __restrict__ mean, const double* __restrict__ world, const int* __restrict__ off,
                         int n_obj, int se2, double* __restrict__ out, int* __restrict__ ok) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= n_obj) return;
  const int p0 = off[o], n = off[o + 1] - p0;
  const double* a = mean + 3 * (size_t)p0;
  const double* b = world + 3 * (size_t)p0;
  double* T = out + 16 * (size_t)o;
  for (int i = 0; i < 16; ++i) T[i] = (i % 5 == 0) ? 1.0 : 0.0;
  double din = 0.0, dout = 0.0;
  for (int c = 0; c + 1 < n; ++c) {
    double s0 = 0, s1 = 0;
    for (int k = 0; k < 3; ++k) {
      const double da = a[3 * (c + 1) + k] - a[3 * c + k], db = b[3 * (c + 1) + k] - b[3 * c + k];
      s0 += da * da;
      s1 += db * db;
    }
    din += sqrt(s0);
    dout += sqrt(s1);
  }
  if (n < 2 || !(din > 0.0) || !(dout > 0.0)) { ok[o] = 0; return; }
  const double scale = dout / din;
  double ca[3] = {0, 0, 0}, cb[3] = {0, 0, 0};
  for (int c = 0; c < n; ++c)
    for (int k = 0; k < 3; ++k) { ca[k] += a[3 * c + k]; cb[k] += b[3 * c + k] / scale; }
  for (int k = 0; k < 3; ++k) { ca[k] /= n; cb[k] /= n; }
  double C[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};               // in * out^T
  for (int c = 0; c < n; ++c)
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) C[3 * i + j] += (a[3 * c + i] - ca[i]) * (b[3 * c + j] / scale - cb[j]);
  double U[9], S[3], V[9], VUt[9], R[9];
  svd3_hestenes(C, U, S, V);
  m3_mulT(V, U, VUt);
  const double d = det3(VUt) > 0 ? 1.0 : -1.0;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) R[3 * i + j] = (V[3 * i] * U[3 * j] + V[3 * i + 1] * U[3 * j + 1]) + d * V[3 * i + 2] * U[3 * j + 2];
  double Rc[3];
  m3_vec(R, ca, Rc);
  double M[16];
  for (int i = 0; i < 16; ++i) M[i] = (i % 5 == 0) ? 1.0 : 0.0;
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) M[4 * i + j] = scale * R[3 * i + j];
    M[4 * i + 3] = scale * (cb[i] - Rc[i]);
  }
  if (se2) {                                 // poseSE32SE2, literally (yaw = pi / atan2(r21, r11), z = 0)
    double yaw = 3.14159265358979323846 / atan2(M[4], M[0]);
    if (!isfinite(yaw)) yaw = 0.0;
    const double tx = M[3], ty = M[7];
    for (int i = 0; i < 16; ++i) M[i] = (i % 5 == 0) ? 1.0 : 0.0;
    M[0] = cos(yaw); M[1] = -sin(yaw); M[3] = tx;
    M[4] = sin(yaw); M[5] = cos(yaw); M[7] = ty;
  }
  for (int i = 0; i < 16; ++i) T[i] = M[i];
  ok[o] = 1;
}

int kabsch_init(const double* mean_pts, const double* world_pts, const int* off, int n_obj, int se2, double* wTq16,
                int* ok) {
  if (n_obj < 1 || !mean_pts || !world_pts || !off || !wTq16 || !ok) return ORCVIO_ERR_ARG;
  const int n_pts = off[n_obj];
  if (n_pts < 0) return ORCVIO_ERR_ARG;
  DeviceBuf<double> dA, dB, dT;
  DeviceBuf<int> dOff, dOk;
  const size_t np = 3 * (size_t)std::max(n_pts, 1);
  if (!dA.alloc(np) || !dB.alloc(np) || !dT.alloc(16 * (size_t)n_obj) || !dOff.alloc(n_obj + 1) || !dOk.alloc(n_obj))
    return ORCVIO_ERR_CUDA;
  cudaMemcpy(dA.get(), mean_pts, sizeof(double) * 3 * n_pts, cudaMemcpyHostToDevice);
  cudaMemcpy(dB.get(), world_pts, sizeof(double) * 3 * n_pts, cudaMemcpyHostToDevice);
  cudaMemcpy(dOff.get(), off, sizeof(int) * (n_obj + 1), cudaMemcpyHostToDevice);
  k_kabsch<<<(n_obj + 63) / 64, 64>>>(dA.get(), dB.get(), dOff.get(), n_obj, se2, dT.get(), dOk.get());
  check_launch("k_kabsch");
  const bool good = cudaMemcpy(wTq16, dT.get(), sizeof(double) * 16 * n_obj, cudaMemcpyDeviceToHost) == cudaSuccess &&
                    cudaMemcpy(ok, dOk.get(), sizeof(int) * n_obj, cudaMemcpyDeviceToHost) == cudaSuccess;
  return good ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

}  // namespace ob

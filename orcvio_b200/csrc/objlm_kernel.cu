// Object state optimiser (SURVEY 8f rank 2), the step immediately before stage 3, for a BATCH of objects of one class:
//   ObjectFeatureInitializer::single_object_initialization   src/obj/ObjectFeatureInitializer.cpp:33-111
//     keypoint triangulation single_triangulation_common     src/feat/FeatureInitializer.cpp:6-110
//     findTransform + poseSE32SE2                            (kabsch_kernel.cu)
//   ObjectFeatureInitializer::single_levenberg_marquardt     src/obj/ObjectFeatureInitializer.cpp:346-381
//     ObjectLM::operator() / df over its four functors       src/obj/ObjectLM.cpp:272-371, 443-632, 652-816
//     LMObjectState operator+ / scaled_norm                  src/obj/ObjectLM.cpp:63-70, 211-227, ObjectLM.h:236-249
//     the vendored MINPACK driver                            (lm.h / lm.cpp)
//
// Device side.  `k_kp_triangulate`: one thread per (object, keypoint) streams the 2 x 3 rows of the linear triangulation
// through Givens rotations into a 3 x 3 triangle (the reference solves the stacked system with a column-pivoted QR;
// this is the same least-squares solution with O(1) memory).  `k_object_lm_eval`: one CTA per evaluation request =
// (object, trial state); thread (lane, slot) walks the frames lane, lane + 8, ... of ONE keypoint or ONE bounding-box
// line (slot), so its rows all touch the same 9 columns [pose 6 | own keypoint 3] or [pose 6 | shape 3] and the
// thread accumulates a 9 x 9 block of J^T J, 9 entries of J^T f and f^T f in registers; the lanes are reduced in a fixed
// order (shuffle, then shared memory), the blocks are scattered into the n x n normal matrix (n = 9 + 3K <= 45) and
// the two regularisers (identity Jacobians, repeated once per frame like the reference does) are added in closed form.
// The 600 x 45 Jacobian of the reference never exists.  Host side: one LmSolver per object advanced in lock-step, one
// launch + one 17 KB-per-object read-back per round.
#include <cmath>
#include <vector>

#include "../../include/orcvio_b200.h"
#include "devmem.h"
#include "kernels.h"
#include "lm.h"
#include "obj_math.cuh"

namespace ob {

namespace {

using namespace objm;

constexpr int LM_SLOTS = 16;     // K keypoints + 4 bounding-box lines <= 16
constexpr int LM_LANES = 8;
constexpr int LM_ACC = 55;       // 45 (upper 9 x 9) + 9 + 1

__device__ __forceinline__ int up9(int a, int b) { return a * 9 - a * (a - 1) / 2 + (b - a); }   // a <= b

struct ObjLmArgs {
  const double* frames_wTc;   // sumT x 16
  const double* zs;           // sumT x K x 2 (NaN = not observed)
  const double* zb;           // sumT x 4
  const int* frame_off;       // n_obj + 1
  const int* req_obj;         // request -> object
  const double* xs;           // request -> [wTo 16 | shape 3 | kps 3K]
  const double* kps_mean;     // K x 3
  const double* mean_shape;   // 3
  double w[4];
  int K, flags;
  double* out;                // request -> [|f| | J^T f (n) | J^T J (n x n row-major)]
};

__device__ void acc_row(double* acc, const double* j9, double r) {
#pragma unroll
  for (int a = 0; a < 9; ++a) {
#pragma unroll
    for (int b = a; b < 9; ++b) acc[up9(a, b)] += j9[a] * j9[b];
    acc[45 + a] += j9[a] * r;
  }
  acc[54] += r * r;
}

__global__ void __launch_bounds__(LM_SLOTS * LM_LANES) k_object_lm_eval(ObjLmArgs a) {
  __shared__ double red[4][LM_SLOTS][LM_ACC];
  __shared__ double sx[19 + 36];
  const int r = blockIdx.x, tid = threadIdx.x, slot = tid % LM_SLOTS, lane = tid / LM_SLOTS;
  const int K = a.K, n = 9 + 3 * K, xdim = 19 + 3 * K;
  const int o = a.req_obj[r], f0 = a.frame_off[o], T = a.frame_off[o + 1] - f0;
  const bool left = (a.flags & 1) != 0, new_res = (a.flags & 2) != 0;
  for (int i = tid; i < xdim; i += blockDim.x) sx[i] = a.xs[(size_t)r * xdim + i];
  __syncthreads();
  const double* wTo = sx;
  const double* shape = sx + 16;
  double acc[LM_ACC];
#pragma unroll
  for (int i = 0; i < LM_ACC; ++i) acc[i] = 0.0;
  if (slot < K + 4) {
    for (int f = lane; f < T; f += LM_LANES) {
      double wTc[16], cTw[16], Pm[16];
      for (int i = 0; i < 16; ++i) wTc[i] = a.frames_wTc[(size_t)(f0 + f) * 16 + i];
      inv_rigid(wTc, cTw);
      mm<4, 4, 4>(cTw, wTo, Pm);
      if (slot < K) {
        // ---- keypoint rows (ObjectLM::ErrorFeatureQuadric, ObjectLM.cpp:272-349)
        const double zu = a.zs[((size_t)(f0 + f) * K + slot) * 2], zv = a.zs[((size_t)(f0 + f) * K + slot) * 2 + 1];
        if (!(isfinite(zu) && isfinite(zv))) continue;
        const double X[4] = {sx[19 + 3 * slot], sx[19 + 3 * slot + 1], sx[19 + 3 * slot + 2], 1.0};
        double Y[4], Z[4], d[6], O[24], cO[24], J26[12], PW[9], J23[6];
        mm<4, 4, 1>(wTo, X, Y);
        mm<4, 4, 1>(cTw, Y, Z);
        dpi_of(Z, d);
        if (left) {                                   // dpi P odot(wTo X)
          odot(Y, O);
          mm<4, 4, 6>(cTw, O, cO);
        } else {                                      // dpi P wTo odot(X)
          odot(X, O);
          mm<4, 4, 6>(Pm, O, cO);
        }
        mm<2, 3, 6>(d, cO, J26);
        for (int i = 0; i < 3; ++i)
          for (int j = 0; j < 3; ++j) PW[3 * i + j] = Pm[4 * i + j];
        mm<2, 3, 3>(d, PW, J23);
        const double res[2] = {Z[0] / Z[2] - zu, Z[1] / Z[2] - zv};
        for (int q = 0; q < 2; ++q) {
          double j9[9];
          for (int c = 0; c < 6; ++c) j9[c] = a.w[0] * J26[6 * q + c];
          for (int c = 0; c < 3; ++c) j9[6 + c] = a.w[0] * J23[3 * q + c];
          acc_row(acc, j9, a.w[0] * res[q]);
        }
      } else {
        // ---- bounding-box line (ObjectLM::ErrorBBoxQuadric, ObjectLM.cpp:443-612)
        const int i = slot - K;
        const double* zb = a.zb + (size_t)(f0 + f) * 4;
        const double px[4] = {zb[0], zb[2], zb[2], zb[0]}, py[4] = {zb[1], zb[1], zb[3], zb[3]};
        const double ax = px[i], ay = py[i], bx = px[(i + 1) & 3], by = py[(i + 1) & 3];
        const double line[3] = {ay * 1.0 - 1.0 * by, 1.0 * bx - ax * 1.0, ax * by - ay * bx};
        const double v2[3] = {shape[0] * shape[0], shape[1] * shape[1], shape[2] * shape[2]};
        double ub[4], res;
        for (int c = 0; c < 4; ++c) ub[c] = (Pm[c] * line[0] + Pm[4 + c] * line[1]) + Pm[8 + c] * line[2];
        if (!new_res) {
          res = ((v2[0] * ub[0] * ub[0] + v2[1] * ub[1] * ub[1]) + v2[2] * ub[2] * ub[2]) - ub[3] * ub[3];
        } else {
          const double bn = sqrt((ub[0] * ub[0] + ub[1] * ub[1]) + ub[2] * ub[2]);
          const double sq = sqrt((v2[0] * ub[0] * ub[0] + v2[1] * ub[1] * ub[1]) + v2[2] * ub[2] * ub[2]);
          res = (ub[3] - (ub[3] > 0 ? 1.0 : -1.0) * sq) / bn;
        }
        double yyw[4], yyo[4], wToT[16], Cc[24], CcT[24], Jo[6], Js[3];
        for (int c = 0; c < 4; ++c) yyw[c] = (line[0] * cTw[c] + line[1] * cTw[4 + c]) + line[2] * cTw[8 + c];
        for (int c = 0; c < 4; ++c)
          yyo[c] = ((yyw[0] * wTo[c] + yyw[1] * wTo[4 + c]) + yyw[2] * wTo[8 + c]) + yyw[3] * wTo[12 + c];
        tr<4, 4>(wTo, wToT);
        if (!new_res) {
          const double Q[4] = {v2[0], v2[1], v2[2], -1.0};
          double yq[4], t4[4];
          for (int c = 0; c < 4; ++c) yq[c] = 2 * yyo[c] * Q[c];
          if (left) {
            mm<1, 4, 4>(yq, wToT, t4);
            circ(yyw, Cc);
            tr<6, 4>(Cc, CcT);
            mm<1, 4, 6>(t4, CcT, Jo);
          } else {
            double wy[4];
            mm<4, 4, 1>(wToT, yyw, wy);
            circ(wy, Cc);
            tr<6, 4>(Cc, CcT);
            mm<1, 4, 6>(yq, CcT, Jo);
          }
          for (int c = 0; c < 3; ++c) Js[c] = 2 * shape[c] * (yyo[c] * yyo[c]);
        } else {
          // the reference evaluates the plane of the new residual's Jacobian from P = K cTw (ObjectLM.cpp:559-560)
          const double bn = sqrt((yyw[0] * yyw[0] + yyw[1] * yyw[1]) + yyw[2] * yyw[2]);
          const double sq = sqrt((v2[0] * yyw[0] * yyw[0] + v2[1] * yyw[1] * yyw[1]) + v2[2] * yyw[2] * yyw[2]);
          const double sign = yyw[3] > 0 ? 1.0 : -1.0;
          double pa[4], M44[16], chain[4], D46[24];
          for (int c = 0; c < 4; ++c) pa[c] = (c == 3 ? 1.0 : 0.0) - sign * (c < 3 ? yyw[c] * v2[c] : 0.0) / sq;
          const double bn3 = bn * bn * bn;
          for (int p = 0; p < 4; ++p)
            for (int c = 0; c < 4; ++c) M44[4 * p + c] = (p == c ? 1.0 / bn : 0.0) - (c < 3 ? yyw[p] * yyw[c] : 0.0) / bn3;
          mm<1, 4, 4>(pa, M44, chain);
          if (left) {
            circ(yyw, Cc);
            tr<6, 4>(Cc, CcT);
            mm<4, 4, 6>(wToT, CcT, D46);
          } else {
            double wy[4];
            mm<4, 4, 1>(wToT, yyw, wy);
            circ(wy, Cc);
            tr<6, 4>(Cc, D46);
          }
          mm<1, 4, 6>(chain, D46, Jo);
          for (int c = 0; c < 3; ++c) Js[c] = (shape[c] * (yyw[c] * yyw[c])) / (bn * sq);
        }
        double j9[9];
        for (int c = 0; c < 6; ++c) j9[c] = a.w[1] * Jo[c];
        for (int c = 0; c < 3; ++c) j9[6 + c] = a.w[1] * Js[c];
        acc_row(acc, j9, a.w[1] * res);
      }
    }
  }
  // lanes 2w, 2w+1 share a warp (threads slot, slot + 16): one shuffle, then the four warps in order
  const int warp = tid >> 5;
#pragma unroll
  for (int i = 0; i < LM_ACC; ++i) {
    const double other = __shfl_down_sync(0xffffffffu, acc[i], 16);
    if ((tid & 31) < 16) red[warp][slot][i] = acc[i] + other;
  }
  __syncthreads();
  double* blk = &red[0][0][0];                       // red[0][slot][i] <- sum over the warps
  for (int e = tid; e < LM_SLOTS * LM_ACC; e += blockDim.x)
    blk[e] = ((blk[e] + blk[LM_SLOTS * LM_ACC + e]) + blk[2 * LM_SLOTS * LM_ACC + e]) + blk[3 * LM_SLOTS * LM_ACC + e];
  __syncthreads();
  // ---- assembly
  double* out = a.out + (size_t)r * (1 + n + n * n);
  const double reg2 = T * a.w[2] * a.w[2], reg3 = T * a.w[3] * a.w[3];
  auto B = [&](int s, int p, int q) { return red[0][s][p <= q ? up9(p, q) : up9(q, p)]; };
  for (int e = tid; e < n * n; e += blockDim.x) {
    const int p = e / n, q = e - p * n;
    const int lo = p < q ? p : q, hi = p < q ? q : p;
    double v = 0.0;
    if (hi < 6) {
      for (int s = 0; s < K + 4; ++s) v += B(s, lo, hi);
    } else if (hi < 9) {                             // shape column: bounding-box slots only
      for (int s = K; s < K + 4; ++s) v += B(s, lo, hi);
      if (lo == hi) v += reg3;
    } else {
      const int k = (hi - 9) / 3, c = (hi - 9) % 3;
      if (lo < 6) v = B(k, lo, 6 + c);
      else if (lo >= 9 && (lo - 9) / 3 == k) v = B(k, 6 + (lo - 9) % 3, 6 + c) + (lo == hi ? reg2 : 0.0);
    }
    out[1 + n + e] = v;
  }
  for (int p = tid; p < n; p += blockDim.x) {
    double v = 0.0;
    if (p < 6) {
      for (int s = 0; s < K + 4; ++s) v += red[0][s][45 + p];
    } else if (p < 9) {
      for (int s = K; s < K + 4; ++s) v += red[0][s][45 + p];
      v += reg3 * (shape[p - 6] - a.mean_shape[p - 6]);
    } else {
      const int k = (p - 9) / 3, c = (p - 9) % 3;
      v = red[0][k][45 + 6 + c] + reg2 * (sx[19 + 3 * k + c] - a.kps_mean[3 * k + c]);
    }
    out[1 + p] = v;
  }
  if (tid == 0) {
    double ss = 0.0;
    for (int s = 0; s < K + 4; ++s) ss += red[0][s][54];
    double d2 = 0.0, d3 = 0.0;
    for (int i = 0; i < 3 * K; ++i) { const double d = sx[19 + i] - a.kps_mean[i]; d2 += d * d; }
    for (int i = 0; i < 3; ++i) { const double d = shape[i] - a.mean_shape[i]; d3 += d * d; }
    out[0] = sqrt(ss + reg2 * d2 + reg3 * d3);
  }
}

// one thread per valid (object, keypoint): kp_list[i] = (object, keypoint, output point index)
__global__ void k_kp_triangulate(const double* __restrict__ frames_wTc, const double* __restrict__ zs,
                                 const int* __restrict__ frame_off, const int* __restrict__ kp_list, int n_list, int K,
                                 double* __restrict__ pts) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_list) return;
  const int o = kp_list[3 * i], k = kp_list[3 * i + 1], dst = kp_list[3 * i + 2];
  const int f0 = frame_off[o], f1 = frame_off[o + 1];
  int fa = -1;                                      // anchor = the last observing frame (FeatureInitializer.cpp:33-36)
  for (int f = f1 - 1; f >= f0; --f) {
    const double u = zs[((size_t)f * K + k) * 2], v = zs[((size_t)f * K + k) * 2 + 1];
    if (isfinite(u) && isfinite(v)) { fa = f; break; }
  }
  if (fa < 0) return;
  double RA[9], pA[3];
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) RA[3 * r + c] = frames_wTc[(size_t)fa * 16 + 4 * r + c];
    pA[r] = frames_wTc[(size_t)fa * 16 + 4 * r + 3];
  }
  double R[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, d[3] = {0, 0, 0};
  for (int f = f0; f <= fa; ++f) {
    const double u = zs[((size_t)f * K + k) * 2], v = zs[((size_t)f * K + k) * 2 + 1];
    if (!(isfinite(u) && isfinite(v))) continue;
    double Ri[9], dp[3], t[3], b[3], pc[3];
    for (int r = 0; r < 3; ++r) {
      for (int c = 0; c < 3; ++c) Ri[3 * r + c] = frames_wTc[(size_t)f * 16 + 4 * r + c];
      dp[r] = frames_wTc[(size_t)f * 16 + 4 * r + 3] - pA[r];
    }
    const double uv1[3] = {u, v, 1.0};
    m3_vec(Ri, uv1, t);                             // R_AtoCi^T b = R_A^T R_i b
    m3_Tvec(RA, t, b);
    const double bn = v3_norm(b);
    for (int c = 0; c < 3; ++c) b[c] /= bn;
    m3_Tvec(RA, dp, pc);                            // p_CiinA
    double rows[2][4] = {{-b[2], 0.0, b[0], 0.0}, {0.0, b[2], -b[1], 0.0}};
    for (int q = 0; q < 2; ++q) {
      rows[q][3] = (rows[q][0] * pc[0] + rows[q][1] * pc[1]) + rows[q][2] * pc[2];
      for (int c = 0; c < 3; ++c) {                 // rotate the row into the triangle
        const double x = rows[q][c];
        if (x == 0.0) continue;
        const double rr = R[4 * c], h = hypot(rr, x), cs = rr / h, sn = x / h;
        for (int j = c; j < 3; ++j) {
          const double up = R[3 * c + j], lo = rows[q][j];
          R[3 * c + j] = cs * up + sn * lo;
          rows[q][j] = cs * lo - sn * up;
        }
        const double up = d[c], lo = rows[q][3];
        d[c] = cs * up + sn * lo;
        rows[q][3] = cs * lo - sn * up;
      }
    }
  }
  double x[3];
  x[2] = d[2] / R[8];
  x[1] = (d[1] - R[5] * x[2]) / R[4];
  x[0] = ((d[0] - R[1] * x[1]) - R[2] * x[2]) / R[0];
  double g[3];
  m3_vec(RA, x, g);
  for (int c = 0; c < 3; ++c) pts[3 * (size_t)dst + c] = g[c] + pA[c];
}

// k_kabsch lives in kabsch_kernel.cu
bool valid_obs(const double* zs, int K, int f, int k) {
  return std::isfinite(zs[((size_t)f * K + k) * 2]) && std::isfinite(zs[((size_t)f * K + k) * 2 + 1]);
}

}  // namespace

int object_init(int n_obj, const int* frame_off, const double* frames_wTc, const double* zs, int K, const double* kps_mean,
                int se2, int min_obs, double* wTq16, int* ok, double* kp_world, int* kp_valid) {
  if (n_obj < 1 || !frame_off || !frames_wTc || !zs || !kps_mean || !wTq16 || !ok || K < 1) return ORCVIO_ERR_ARG;
  const int sumT = frame_off[n_obj];
  for (int o = 0; o < n_obj; ++o)
    if (frame_off[o + 1] < frame_off[o]) return ORCVIO_ERR_ARG;
  // keypoints seen in MORE than min_obs frames are triangulated (ObjectFeature::zs_to_uvnorm, ObjectFeature.cpp:86-127)
  std::vector<int> list, off(n_obj + 1, 0), valid((size_t)n_obj * K, 0);
  std::vector<double> mean_sel;
  for (int o = 0; o < n_obj; ++o) {
    int cnt = 0;
    for (int k = 0; k < K; ++k) {
      int seen = 0;
      for (int f = frame_off[o]; f < frame_off[o + 1]; ++f) seen += valid_obs(zs, K, f, k);
      const bool use = seen > min_obs;
      valid[(size_t)o * K + k] = use;
      if (kp_valid) kp_valid[(size_t)o * K + k] = use;
      if (!use) continue;
      list.push_back(o);
      list.push_back(k);
      list.push_back(off[o] + cnt);
      for (int c = 0; c < 3; ++c) mean_sel.push_back(kps_mean[3 * k + c]);
      ++cnt;
    }
    off[o + 1] = off[o] + cnt;
  }
  const int n_list = off[n_obj];
  std::vector<double> pts(3 * (size_t)std::max(n_list, 1), 0.0);
  if (n_list > 0) {
    DeviceBuf<double> dF, dZ, dP;
    DeviceBuf<int> dOff, dList;
    if (!dF.alloc(16 * (size_t)sumT) || !dZ.alloc(2 * (size_t)K * sumT) || !dOff.alloc(n_obj + 1) ||
        !dList.alloc(3 * (size_t)n_list) || !dP.alloc(3 * (size_t)n_list))
      return ORCVIO_ERR_CUDA;
    cudaMemcpy(dF.get(), frames_wTc, sizeof(double) * 16 * sumT, cudaMemcpyHostToDevice);
    cudaMemcpy(dZ.get(), zs, sizeof(double) * 2 * K * sumT, cudaMemcpyHostToDevice);
    cudaMemcpy(dOff.get(), frame_off, sizeof(int) * (n_obj + 1), cudaMemcpyHostToDevice);
    cudaMemcpy(dList.get(), list.data(), sizeof(int) * 3 * n_list, cudaMemcpyHostToDevice);
    k_kp_triangulate<<<(n_list + 63) / 64, 64>>>(dF.get(), dZ.get(), dOff.get(), dList.get(), n_list, K, dP.get());
    check_launch("k_kp_triangulate");
    if (cudaMemcpy(pts.data(), dP.get(), sizeof(double) * 3 * n_list, cudaMemcpyDeviceToHost) != cudaSuccess) return ORCVIO_ERR_CUDA;
  }
  if (kp_world)
    for (int o = 0; o < n_obj; ++o) {
      int cnt = 0;
      for (int k = 0; k < K; ++k) {
        double* dst = kp_world + 3 * ((size_t)o * K + k);
        const bool use = valid[(size_t)o * K + k] != 0;
        for (int c = 0; c < 3; ++c) dst[c] = use ? pts[3 * (size_t)(off[o] + cnt) + c] : NAN;
        cnt += use;
      }
    }
  // more than 3 triangulated keypoints -> findTransform (+ poseSE32SE2); else identity, not ok (:84-111)
  std::vector<int> sel, off2(1, 0);
  std::vector<double> m2, p2;
  for (int o = 0; o < n_obj; ++o) {
    for (int i = 0; i < 16; ++i) wTq16[16 * (size_t)o + i] = (i % 5 == 0) ? 1.0 : 0.0;
    ok[o] = 0;
    if (off[o + 1] - off[o] <= 3) continue;
    sel.push_back(o);
    m2.insert(m2.end(), mean_sel.begin() + 3 * (size_t)off[o], mean_sel.begin() + 3 * (size_t)off[o + 1]);
    p2.insert(p2.end(), pts.begin() + 3 * (size_t)off[o], pts.begin() + 3 * (size_t)off[o + 1]);
    off2.push_back(off2.back() + off[o + 1] - off[o]);
  }
  if (!sel.empty()) {
    std::vector<double> T(16 * sel.size());
    std::vector<int> okk(sel.size());
    const int rc = kabsch_init(m2.data(), p2.data(), off2.data(), (int)sel.size(), se2, T.data(), okk.data());
    if (rc != ORCVIO_OK) return rc;
    for (size_t i = 0; i < sel.size(); ++i) {
      ok[sel[i]] = okk[i];
      if (okk[i]) std::copy(T.begin() + 16 * i, T.begin() + 16 * (i + 1), wTq16 + 16 * (size_t)sel[i]);
    }
  }
  return ORCVIO_OK;
}

int object_lm(int n_obj, const int* frame_off, const double* frames_wTc, const double* zs, const double* zb, int K,
              const double* kps_mean, const double* mean_shape, const double* weights4, int flags, const double* wTo_init,
              double* wTo_out, double* shape_out, double* kps_out, double* kps_world_out, int* status, int* nfev,
              int* njev, double* fnorm, int* rounds_out) {
  if (n_obj < 1 || !frame_off || !frames_wTc || !zs || !zb || !kps_mean || !mean_shape || !weights4 || !wTo_init ||
      !wTo_out || !shape_out || !kps_out || !status)
    return ORCVIO_ERR_ARG;
  if (K < 1 || K + 4 > LM_SLOTS) return ORCVIO_ERR_ARG;
  const int sumT = frame_off[n_obj];
  for (int o = 0; o < n_obj; ++o)
    if (frame_off[o + 1] <= frame_off[o]) return ORCVIO_ERR_ARG;
  const int n = 9 + 3 * K, xdim = 19 + 3 * K, odim = 1 + n + n * n;
  DeviceBuf<double> dF, dZ, dB, dX, dMean, dShape, dOut;
  DeviceBuf<int> dOff, dReq;
  if (!dF.alloc(16 * (size_t)sumT) || !dZ.alloc(2 * (size_t)K * sumT) || !dB.alloc(4 * (size_t)sumT) ||
      !dOff.alloc(n_obj + 1) || !dReq.alloc(n_obj) || !dX.alloc((size_t)xdim * n_obj) || !dMean.alloc(3 * (size_t)K) ||
      !dShape.alloc(3) || !dOut.alloc((size_t)odim * n_obj))
    return ORCVIO_ERR_CUDA;
  cudaMemcpy(dF.get(), frames_wTc, sizeof(double) * 16 * sumT, cudaMemcpyHostToDevice);
  cudaMemcpy(dZ.get(), zs, sizeof(double) * 2 * K * sumT, cudaMemcpyHostToDevice);
  cudaMemcpy(dB.get(), zb, sizeof(double) * 4 * sumT, cudaMemcpyHostToDevice);
  cudaMemcpy(dOff.get(), frame_off, sizeof(int) * (n_obj + 1), cudaMemcpyHostToDevice);
  cudaMemcpy(dMean.get(), kps_mean, sizeof(double) * 3 * K, cudaMemcpyHostToDevice);
  cudaMemcpy(dShape.get(), mean_shape, sizeof(double) * 3, cudaMemcpyHostToDevice);
  ObjLmArgs a{};
  a.frames_wTc = dF.get(); a.zs = dZ.get(); a.zb = dB.get(); a.frame_off = dOff.get();
  a.req_obj = dReq.get(); a.xs = dX.get(); a.kps_mean = dMean.get(); a.mean_shape = dShape.get();
  for (int i = 0; i < 4; ++i) a.w[i] = weights4[i];
  a.K = K; a.flags = flags; a.out = dOut.get();

  // LMObjectState operator+ (always a left retraction) and scaled_norm (a sum of block norms)
  PlusFn plus = [K](const std::vector<double>& x, const double* dx, std::vector<double>& out) {
    out.resize(x.size());
    double E[16];
    se3_exp(dx, E);
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < 4; ++j) {
        double acc = 0.0;
        for (int k = 0; k < 4; ++k) acc += E[4 * i + k] * x[4 * k + j];
        out[4 * i + j] = acc;
      }
    for (int i = 0; i < 3 + 3 * K; ++i) out[16 + i] = x[16 + i] + dx[6 + i];
  };
  NormFn norm = [K](const double* diag, const std::vector<double>& x) {
    double xi[6], s = 0.0, acc = 0.0;
    se3_log(x.data(), xi);
    for (int i = 0; i < 6; ++i) acc += diag[i] * xi[i] * diag[i] * xi[i];
    s += std::sqrt(acc);
    for (int b = 0; b < 1 + K; ++b) {
      acc = 0.0;
      for (int c = 0; c < 3; ++c) { const double v = diag[6 + 3 * b + c] * x[16 + 3 * b + c]; acc += v * v; }
      s += std::sqrt(acc);
    }
    return s;
  };
  LmOptions opt;
  opt.factor = 10.0;                                  // lm.setFactor(10), ObjectFeatureInitializer.cpp:370
  std::vector<LmSolver> solvers(n_obj);
  for (int o = 0; o < n_obj; ++o) {
    std::vector<double> x0(xdim);
    std::copy(wTo_init + 16 * (size_t)o, wTo_init + 16 * (size_t)(o + 1), x0.begin());
    std::copy(mean_shape, mean_shape + 3, x0.begin() + 16);
    std::copy(kps_mean, kps_mean + 3 * K, x0.begin() + 19);
    solvers[o].start(n, x0, opt, plus, norm);
  }
  std::vector<int> req;
  std::vector<double> xs, out;
  int rounds = 0;
  for (;;) {
    req.clear();
    xs.clear();
    for (int o = 0; o < n_obj; ++o)
      if (solvers[o].running()) {
        req.push_back(o);
        xs.insert(xs.end(), solvers[o].request().begin(), solvers[o].request().end());
      }
    if (req.empty()) break;
    const int nr = (int)req.size();
    cudaMemcpy(dReq.get(), req.data(), sizeof(int) * nr, cudaMemcpyHostToDevice);
    cudaMemcpy(dX.get(), xs.data(), sizeof(double) * xdim * nr, cudaMemcpyHostToDevice);
    k_object_lm_eval<<<nr, LM_SLOTS * LM_LANES>>>(a);
    check_launch("k_object_lm_eval");
    out.resize((size_t)odim * nr);
    if (cudaMemcpy(out.data(), dOut.get(), sizeof(double) * odim * nr, cudaMemcpyDeviceToHost) != cudaSuccess) return ORCVIO_ERR_CUDA;
    for (int i = 0; i < nr; ++i) {
      const double* r = out.data() + (size_t)odim * i;
      solvers[req[i]].feed(r[0], r + 1 + n, r + 1);
    }
    ++rounds;
  }
  for (int o = 0; o < n_obj; ++o) {
    const LmSolver& s = solvers[o];
    std::copy(s.x.begin(), s.x.begin() + 16, wTo_out + 16 * (size_t)o);
    std::copy(s.x.begin() + 16, s.x.begin() + 19, shape_out + 3 * (size_t)o);
    std::copy(s.x.begin() + 19, s.x.end(), kps_out + 3 * (size_t)K * o);
    if (kps_world_out)                               // transform_mean_keypoints_to_global, ObjectState.cpp:15-40
      for (int k = 0; k < K; ++k)
        for (int r = 0; r < 3; ++r)
          kps_world_out[3 * ((size_t)K * o + k) + r] =
              ((s.x[4 * r] * s.x[19 + 3 * k] + s.x[4 * r + 1] * s.x[19 + 3 * k + 1]) + s.x[4 * r + 2] * s.x[19 + 3 * k + 2]) + s.x[4 * r + 3];
    status[o] = s.res.status;
    if (nfev) nfev[o] = s.res.nfev;
    if (njev) njev[o] = s.res.njev;
    if (fnorm) fnorm[o] = s.res.fnorm;
  }
  if (rounds_out) *rounds_out = rounds;
  return ORCVIO_OK;
}

// one evaluation of the LM model (|f|, J^T f, J^T J) at given states: the element-wise parity surface of the kernel
int object_lm_eval(int n_obj, const int* frame_off, const double* frames_wTc, const double* zs, const double* zb, int K,
                   const double* kps_mean, const double* mean_shape, const double* weights4, int flags, const double* xs,
                   double* out) {
  if (n_obj < 1 || !frame_off || !frames_wTc || !zs || !zb || !kps_mean || !mean_shape || !weights4 || !xs || !out)
    return ORCVIO_ERR_ARG;
  if (K < 1 || K + 4 > LM_SLOTS) return ORCVIO_ERR_ARG;
  const int sumT = frame_off[n_obj];
  const int n = 9 + 3 * K, xdim = 19 + 3 * K, odim = 1 + n + n * n;
  DeviceBuf<double> dF, dZ, dB, dX, dMean, dShape, dOut;
  DeviceBuf<int> dOff, dReq;
  if (!dF.alloc(16 * (size_t)sumT) || !dZ.alloc(2 * (size_t)K * sumT) || !dB.alloc(4 * (size_t)sumT) ||
      !dOff.alloc(n_obj + 1) || !dReq.alloc(n_obj) || !dX.alloc((size_t)xdim * n_obj) || !dMean.alloc(3 * (size_t)K) ||
      !dShape.alloc(3) || !dOut.alloc((size_t)odim * n_obj))
    return ORCVIO_ERR_CUDA;
  std::vector<int> req(n_obj);
  for (int o = 0; o < n_obj; ++o) req[o] = o;
  cudaMemcpy(dF.get(), frames_wTc, sizeof(double) * 16 * sumT, cudaMemcpyHostToDevice);
  cudaMemcpy(dZ.get(), zs, sizeof(double) * 2 * K * sumT, cudaMemcpyHostToDevice);
  cudaMemcpy(dB.get(), zb, sizeof(double) * 4 * sumT, cudaMemcpyHostToDevice);
  cudaMemcpy(dOff.get(), frame_off, sizeof(int) * (n_obj + 1), cudaMemcpyHostToDevice);
  cudaMemcpy(dMean.get(), kps_mean, sizeof(double) * 3 * K, cudaMemcpyHostToDevice);
  cudaMemcpy(dShape.get(), mean_shape, sizeof(double) * 3, cudaMemcpyHostToDevice);
  cudaMemcpy(dReq.get(), req.data(), sizeof(int) * n_obj, cudaMemcpyHostToDevice);
  cudaMemcpy(dX.get(), xs, sizeof(double) * xdim * n_obj, cudaMemcpyHostToDevice);
  ObjLmArgs a{};
  a.frames_wTc = dF.get(); a.zs = dZ.get(); a.zb = dB.get(); a.frame_off = dOff.get();
  a.req_obj = dReq.get(); a.xs = dX.get(); a.kps_mean = dMean.get(); a.mean_shape = dShape.get();
  for (int i = 0; i < 4; ++i) a.w[i] = weights4[i];
  a.K = K; a.flags = flags; a.out = dOut.get();
  k_object_lm_eval<<<n_obj, LM_SLOTS * LM_LANES>>>(a);
  check_launch("k_object_lm_eval");
  return cudaMemcpy(out, dOut.get(), sizeof(double) * odim * n_obj, cudaMemcpyDeviceToHost) == cudaSuccess ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

// the two known-answer problems of src/tests/test_levenberg_marquardt.cpp through the same driver (host only)
int lm_known_answer(int which, double* x_out, int* status, int* nfev, int* njev, double* fnorm) {
  PlusFn plus = [](const std::vector<double>& x, const double* dx, std::vector<double>& out) {
    out.resize(x.size());
    for (size_t i = 0; i < x.size(); ++i) out[i] = x[i] + dx[i];
  };
  NormFn norm = [](const double* diag, const std::vector<double>& x) {
    double s = 0.0;
    for (size_t i = 0; i < x.size(); ++i) s += diag[i] * x[i] * diag[i] * x[i];
    return std::sqrt(s);
  };
  LmOptions opt;
  std::vector<double> x;
  LmResult res;
  if (which == 0) {          // MINPACK's lmder1 example (:27-90): tol = sqrt(eps), maxfev = 100 (n + 1)
    static const double y[15] = {1.4e-1, 1.8e-1, 2.2e-1, 2.5e-1, 2.9e-1, 3.2e-1, 3.5e-1, 3.9e-1,
                                 3.7e-1, 5.8e-1, 7.3e-1, 9.6e-1, 1.34, 2.1, 4.39};
    x.assign(3, 1.0);
    opt.maxfev = 100 * (3 + 1);
    EvalFn eval = [](const std::vector<double>& x, double* JtJ, double* Jtf) {
      double ss = 0.0;
      for (int i = 0; i < 9; ++i) JtJ[i] = 0.0;
      for (int i = 0; i < 3; ++i) Jtf[i] = 0.0;
      for (int i = 0; i < 15; ++i) {
        const double t1 = i + 1.0, t2 = 16.0 - i - 1.0, t3 = i >= 8 ? t2 : t1;
        const double den = x[1] * t2 + x[2] * t3;
        const double f = y[i] - (x[0] + t1 / den);
        const double j[3] = {-1.0, t1 * t2 / (den * den), t1 * t3 / (den * den)};
        for (int a = 0; a < 3; ++a) {
          for (int b = 0; b < 3; ++b) JtJ[3 * a + b] += j[a] * j[b];
          Jtf[a] += j[a] * f;
        }
        ss += f * f;
      }
      return std::sqrt(ss);
    };
    res = lm_minimize(3, eval, x, opt, plus, norm);
  } else if (which == 1) {   // minimise (x - 10)^2 (:92-140)
    x.assign(1, 1.0);
    EvalFn eval = [](const std::vector<double>& x, double* JtJ, double* Jtf) {
      JtJ[0] = 1.0;
      Jtf[0] = x[0] - 10.0;
      return std::fabs(x[0] - 10.0);
    };
    res = lm_minimize(1, eval, x, opt, plus, norm);
  } else if (which == 2 || which == 3) {
    // two of MINPACK's own test functions, for which the real MINPACK (scipy.optimize.leastsq -> lmder) gives the
    // answer on the CPU test side: Rosenbrock (n = m = 2, start (-1.2, 1)) and Freudenstein-Roth (start (0.5, -2));
    // lmder1 settings (tol = sqrt(eps), maxfev = 100 (n + 1), factor 100)
    const bool rosen = which == 2;
    x = rosen ? std::vector<double>{-1.2, 1.0} : std::vector<double>{0.5, -2.0};
    opt.maxfev = 100 * (2 + 1);
    EvalFn eval = [rosen](const std::vector<double>& x, double* JtJ, double* Jtf) {
      double f[2], J[2][2];
      if (rosen) {
        f[0] = 10 * (x[1] - x[0] * x[0]); f[1] = 1 - x[0];
        J[0][0] = -20 * x[0]; J[0][1] = 10.0; J[1][0] = -1.0; J[1][1] = 0.0;
      } else {
        f[0] = -13 + x[0] + ((5 - x[1]) * x[1] - 2) * x[1];
        f[1] = -29 + x[0] + ((x[1] + 1) * x[1] - 14) * x[1];
        J[0][0] = 1.0; J[0][1] = 10 * x[1] - 3 * x[1] * x[1] - 2;
        J[1][0] = 1.0; J[1][1] = 3 * x[1] * x[1] + 2 * x[1] - 14;
      }
      for (int a = 0; a < 2; ++a) {
        for (int b = 0; b < 2; ++b) JtJ[2 * a + b] = J[0][a] * J[0][b] + J[1][a] * J[1][b];
        Jtf[a] = J[0][a] * f[0] + J[1][a] * f[1];
      }
      return std::sqrt(f[0] * f[0] + f[1] * f[1]);
    };
    res = lm_minimize(2, eval, x, opt, plus, norm);
  } else {
    return ORCVIO_ERR_ARG;
  }
  for (size_t i = 0; i < x.size(); ++i) x_out[i] = x[i];
  if (status) *status = res.status;
  if (nfev) *nfev = res.nfev;
  if (njev) *njev = res.njev;
  if (fnorm) *fnorm = res.fnorm;
  return ORCVIO_OK;
}

}  // namespace ob

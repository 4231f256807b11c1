// Stage 1 -- per-feature triangulation kernel (one warp per candidate feature).
//
// Computes what Feature::checkMotion + Feature::initializePosition[_AssignAnchor] +
// Feature::triangulate_position compute in the reference
// (include/orcvio/feat/feature.hpp:271-351, 353-396, 398-500, 583-719): 2-view depth
// initial guess, Levenberg-Marquardt on (alpha, beta, rho) in the last camera frame with a
// Huber weight, pivoted 3x3 LDL^T solves, the lambda /10 | x10 schedule with the
// post-increment loop counters, and the three validity tests.
//
// The LM accept/reject decisions are rounding sensitive, so this file is compiled with
// --fmad=false and every expression is written in one fixed association order; the CPU
// oracle (oracle/feature.py, oracle/cpu_ref.cpp) uses the same order and agrees bit for bit.
//
// Parallelisation: one warp per feature, lane k owns observation k (relative pose, Jacobian row,
// cost term); the per-observation terms are summed in observation order (through shared memory /
// shuffles) so that every rounding step matches the sequential oracle bit for bit, and one LM
// iteration costs the latency of ONE observation instead of m.  The kernel is bound by the serial
// latency of the slowest feature's LM chain (FP64 divide / sqrt), not by HBM or FP64 throughput.
#include <cstdio>
#include <cstdlib>
#include "kernels.h"

namespace ob {

__device__ __forceinline__ void ldlt3_solve(const double* M, const double* b, double* x) {
  double a[3][3];
  int tr[3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) a[i][j] = M[3 * i + j];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    int big = k;
    double bigv = fabs(a[k][k]);
    for (int i = k + 1; i < 3; ++i) {
      if (fabs(a[i][i]) > bigv) {
        bigv = fabs(a[i][i]);
        big = i;
      }
    }
    tr[k] = big;
    if (big != k) {
      for (int j = 0; j < k; ++j) { double t = a[k][j]; a[k][j] = a[big][j]; a[big][j] = t; }
      for (int i = big + 1; i < 3; ++i) { double t = a[i][k]; a[i][k] = a[i][big]; a[i][big] = t; }
      { double t = a[k][k]; a[k][k] = a[big][big]; a[big][big] = t; }
      for (int i = k + 1; i < big; ++i) { double t = a[i][k]; a[i][k] = a[big][i]; a[big][i] = t; }
    }
    if (k > 0) {
      double temp[3];
      for (int j = 0; j < k; ++j) temp[j] = a[j][j] * a[k][j];
      double s = 0.0;
      for (int j = 0; j < k; ++j) s = s + a[k][j] * temp[j];
      a[k][k] = a[k][k] - s;
      for (int i = k + 1; i < 3; ++i) {
        s = 0.0;
        for (int j = 0; j < k; ++j) s = s + a[i][j] * temp[j];
        a[i][k] = a[i][k] - s;
      }
    }
    double akk = a[k][k];
    if (fabs(akk) > 0.0) {
      for (int i = k + 1; i < 3; ++i) a[i][k] = a[i][k] / akk;
    }
  }
  x[0] = b[0]; x[1] = b[1]; x[2] = b[2];
  for (int k = 0; k < 3; ++k)
    if (tr[k] != k) { double t = x[k]; x[k] = x[tr[k]]; x[tr[k]] = t; }
  for (int i = 0; i < 3; ++i)
    for (int r = i + 1; r < 3; ++r) x[r] = x[r] - x[i] * a[r][i];
  const double tol = 2.2250738585072014e-308;
  for (int i = 0; i < 3; ++i) {
    if (fabs(a[i][i]) > tol) x[i] = x[i] / a[i][i];
    else x[i] = 0.0;
  }
  for (int i = 1; i >= 0; --i) {
    double s = 0.0;
    for (int j = i + 1; j < 3; ++j) s = s + a[j][i] * x[j];
    x[i] = x[i] - s;
  }
  for (int k = 2; k >= 0; --k)
    if (tr[k] != k) { double t = x[k]; x[k] = x[tr[k]]; x[tr[k]] = t; }
}

__device__ __forceinline__ void tri_h(const double* R, const double* t, const double* x, double* h) {
  h[0] = ((R[0] * x[0] + R[1] * x[1]) + R[2] * 1.0) + x[2] * t[0];
  h[1] = ((R[3] * x[0] + R[4] * x[1]) + R[5] * 1.0) + x[2] * t[1];
  h[2] = ((R[6] * x[0] + R[7] * x[1]) + R[8] * 1.0) + x[2] * t[2];
}

__device__ __forceinline__ double tri_cost(const double* R, const double* t, const double* x,
                                           double zu, double zv) {
  double h[3];
  tri_h(R, t, x, h);
  double d0 = h[0] / h[2] - zu;
  double d1 = h[1] / h[2] - zv;
  return d0 * d0 + d1 * d1;
}

// Relative pose of observation clone `c` w.r.t. the last camera (Rl, tl): feature.hpp:600-612.
__device__ __forceinline__ void rel_pose(const double* c, const double* Rl, const double* tl, double* R, double* t) {
  const double* Ri = c + CL_RC;
  const double* ti = c + CL_PC;
  double tinv[3], rt[3];
  m3_Tvec(Ri, ti, tinv);
  m3_Tmul(Ri, Rl, R);
  m3_Tvec(Ri, tl, rt);
  t[0] = rt[0] + (-tinv[0]);
  t[1] = rt[1] + (-tinv[1]);
  t[2] = rt[2] + (-tinv[2]);
}

// sum_{k<m} v_k accumulated in observation order (total = total + v_k), v_k held by lane k
__device__ __forceinline__ double ordered_sum(double v, int m) {
  // the shuffles do not depend on the running sum: fetch eight terms at once, then add them in order (the chain is the
  // m additions, not m shuffle round trips)
  double s = 0.0;
  for (int k0 = 0; k0 < m; k0 += 8) {
    double t[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) t[j] = __shfl_sync(0xffffffffu, v, (k0 + j) & 31);
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (k0 + j < m) s = s + t[j];
  }
  return s;
}

constexpr int TRI_SM_STRIDE = 13;   // 12 contributions per observation, padded: conflict-free both ways

// One WARP per feature: lane k owns observation k (m <= 32), i.e. its relative pose, its row of the
// Jacobian and its cost term; the per-observation terms are then added in observation order so that
// every rounding step matches the sequential oracle.  The 3 x 3 solve and the LM bookkeeping run
// redundantly on all lanes (warp-uniform control flow).  `sm`: 32 * TRI_SM_STRIDE doubles per warp.
// Returns status bit0 = valid.  pos_io: previous world position when is_init, result on exit
// (written only when valid, like the reference's `position = ...` under is_valid_solution).
__device__ int triangulate_feature(const double* __restrict__ clones, int m,
                                   const int* __restrict__ oc, const double* __restrict__ oz,
                                   bool is_init, double* pos_io, const TriCfg& cfg, int* iters,
                                   double* cost_out, double* __restrict__ sm, double* fin_out = nullptr) {
  const int lane = threadIdx.x & 31;
  const bool act = lane < m;
  const double* cl = clones + (size_t)oc[m - 1] * CL_STRIDE;
  double Rl[9], tl[3];
  for (int i = 0; i < 9; ++i) Rl[i] = cl[CL_RC + i];
  for (int i = 0; i < 3; ++i) tl[i] = cl[CL_PC + i];
  double R[9], t[3], zu = 0.0, zv = 0.0;
  {
    const int k = act ? lane : 0;
    rel_pose(clones + (size_t)oc[k] * CL_STRIDE, Rl, tl, R, t);
    zu = oz[2 * k];
    zv = oz[2 * k + 1];
  }
  double init[3];
  if (!is_init) {
    // generateInitialGuess(rel pose 0, z_last, z_first), feature.hpp:331-351
    double R0[9], t0[3];
    rel_pose(clones + (size_t)oc[0] * CL_STRIDE, Rl, tl, R0, t0);
    double z1u = oz[2 * (m - 1)], z1v = oz[2 * (m - 1) + 1];
    double z2u = oz[0], z2v = oz[1];
    double mv[3], zz[3] = {z1u, z1v, 1.0};
    m3_vec(R0, zz, mv);
    double A0 = mv[0] - z2u * mv[2];
    double A1 = mv[1] - z2v * mv[2];
    double b0 = z2u * t0[2] - t0[0];
    double b1 = z2v * t0[2] - t0[1];
    double inv = 1.0 / (A0 * A0 + A1 * A1);
    double depth = (inv * A0) * b0 + (inv * A1) * b1;
    init[0] = z1u * depth;
    init[1] = z1v * depth;
    init[2] = depth;
  } else {
    double tinv[3], rp[3];
    m3_Tvec(Rl, tl, tinv);
    m3_Tvec(Rl, pos_io, rp);
    init[0] = rp[0] + (-tinv[0]);
    init[1] = rp[1] + (-tinv[1]);
    init[2] = rp[2] + (-tinv[2]);
  }
  double sol[3] = {init[0] / init[2], init[1] / init[2], 1.0 / init[2]};
  double lam = cfg.initial_damping;
  int inner = 0, outer = 0, n_inner_total = 0;
  bool reduced = false;
  double delta_norm = 0.0;
  double total_cost = ordered_sum(tri_cost(R, t, sol, zu, zv), m);

  while (true) {
    // this lane's observation: 9 + 3 contributions to A and b
    {
      double h[3];
      tri_h(R, t, sol, h);
      double W[3][3] = {{R[0], R[1], t[0]}, {R[3], R[4], t[1]}, {R[6], R[7], t[2]}};
      double ih3 = 1 / h[2];
      double c0 = h[0] / (h[2] * h[2]);
      double c1 = h[1] / (h[2] * h[2]);
      double J[2][3];
      for (int j = 0; j < 3; ++j) {
        J[0][j] = ih3 * W[0][j] - c0 * W[2][j];
        J[1][j] = ih3 * W[1][j] - c1 * W[2][j];
      }
      double r0 = h[0] / h[2] - zu;
      double r1 = h[1] / h[2] - zv;
      double e = sqrt(r0 * r0 + r1 * r1);
      double* my = sm + lane * TRI_SM_STRIDE;
      if (e <= cfg.huber_epsilon) {
        for (int a_ = 0; a_ < 3; ++a_) {
          for (int c_ = 0; c_ < 3; ++c_) my[3 * a_ + c_] = (J[0][a_] * J[0][c_] + J[1][a_] * J[1][c_]);
          my[9 + a_] = (J[0][a_] * r0 + J[1][a_] * r1);
        }
      } else {
        double w = sqrt(2.0 * cfg.huber_epsilon / e);
        double w2 = w * w;
        for (int a_ = 0; a_ < 3; ++a_) {
          for (int c_ = 0; c_ < 3; ++c_)
            my[3 * a_ + c_] = ((w2 * J[0][a_]) * J[0][c_] + (w2 * J[1][a_]) * J[1][c_]);
          my[9 + a_] = ((w2 * J[0][a_]) * r0 + (w2 * J[1][a_]) * r1);
        }
      }
    }
    __syncwarp();
    double acc = 0.0;           // lane j < 12 sums entry j over the observations, in order
    if (lane < 12)
      for (int k0 = 0; k0 < m; k0 += 8) {      // eight loads in flight, then the ordered additions
        double t[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) t[j] = (k0 + j < m) ? sm[(k0 + j) * TRI_SM_STRIDE + lane] : 0.0;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (k0 + j < m) acc = acc + t[j];
      }
    __syncwarp();
    double A[9], b[3];
    for (int i = 0; i < 9; ++i) A[i] = __shfl_sync(0xffffffffu, acc, i);
    for (int i = 0; i < 3; ++i) b[i] = __shfl_sync(0xffffffffu, acc, 9 + i);
    while (true) {
      double M[9];
      for (int i = 0; i < 9; ++i) M[i] = A[i];
      M[0] = A[0] + lam;
      M[4] = A[4] + lam;
      M[8] = A[8] + lam;
      double delta[3];
      ldlt3_solve(M, b, delta);
      double ns[3] = {sol[0] - delta[0], sol[1] - delta[1], sol[2] - delta[2]};
      delta_norm = sqrt((delta[0] * delta[0] + delta[1] * delta[1]) + delta[2] * delta[2]);
      double new_cost = ordered_sum(tri_cost(R, t, ns, zu, zv), m);
      ++n_inner_total;
      if (new_cost < total_cost) {
        reduced = true;
        sol[0] = ns[0]; sol[1] = ns[1]; sol[2] = ns[2];
        total_cost = new_cost;
        lam = lam / 10 > 1e-10 ? lam / 10 : 1e-10;
      } else {
        reduced = false;
        lam = lam * 10 < 1e12 ? lam * 10 : 1e12;
      }
      bool cont = (inner < cfg.inner_max) && !reduced;
      ++inner;
      if (!cont) break;
    }
    inner = 0;
    bool cont = (outer < cfg.outer_max) && (delta_norm > cfg.estimation_precision);
    ++outer;
    if (!cont) break;
  }
  double fin[3] = {sol[0] / sol[2], sol[1] / sol[2], 1.0 / sol[2]};
  int valid = 1;
  {
    double pz = ((R[6] * fin[0] + R[7] * fin[1]) + R[8] * fin[2]) + t[2];
    if (__any_sync(0xffffffffu, act && pz <= 0)) valid = 0;
  }
  double normalized_cost = total_cost / (double)(2 * m * m);
  double d0 = fin[0] - init[0], d1 = fin[1] - init[1], d2 = fin[2] - init[2];
  if (sqrt((d0 * d0 + d1 * d1) + d2 * d2) > cfg.init_final_dist_threshold) valid = 0;
  if (normalized_cost > cfg.cost_threshold) valid = 0;
  if (iters) { iters[0] = outer; iters[1] = n_inner_total; }
  if (cost_out) *cost_out = total_cost;
  if (valid) {
    double pw[3];
    m3_vec(Rl, fin, pw);
    pos_io[0] = pw[0] + tl[0];
    pos_io[1] = pw[1] + tl[1];
    pos_io[2] = pw[2] + tl[2];
    if (fin_out) { fin_out[0] = fin[0]; fin_out[1] = fin[1]; fin_out[2] = fin[2]; }
  }
  return valid;
}

// Feature::checkMotion, feature.hpp:353-396: first obs vs last obs (second to last when the
// feature is tracked in the current frame).
__device__ __forceinline__ bool check_motion(const double* clones, int first_clone, int last_clone,
                                             double zu, double zv, double thr) {
  const double* c0 = clones + (size_t)first_clone * CL_STRIDE;
  const double* c1 = clones + (size_t)last_clone * CL_STRIDE;
  double d[3] = {zu, zv, 1.0};
  double n = sqrt((d[0] * d[0] + d[1] * d[1]) + d[2] * d[2]);
  d[0] = d[0] / n; d[1] = d[1] / n; d[2] = d[2] / n;
  double dw[3];
  m3_vec(c0 + CL_RC, d, dw);
  double tr[3] = {c1[CL_PC] - c0[CL_PC], c1[CL_PC + 1] - c0[CL_PC + 1], c1[CL_PC + 2] - c0[CL_PC + 2]};
  double par = (tr[0] * dw[0] + tr[1] * dw[1]) + tr[2] * dw[2];
  double o0 = tr[0] - par * dw[0], o1 = tr[1] - par * dw[1], o2 = tr[2] - par * dw[2];
  return sqrt((o0 * o0 + o1 * o1) + o2 * o2) > thr;
}

// One warp per candidate.  Candidates of all filters of the batch are concatenated;
// cand.filter selects the clone array / feature-position table of its filter.
constexpr int TRI_WARPS = 4;

// MINB = resident CTAs per SM the register allocation is held to (launch bound; chosen from the grid size by
// launch_triangulate(): the kernel is one LM latency chain per warp, so whole waves are what cost time).
template <int MINB>
__global__ void __launch_bounds__(32 * TRI_WARPS, MINB) k_triangulate(TriArgs a) {
  __shared__ double sm_all[TRI_WARPS][32 * TRI_SM_STRIDE];
  pdl_launch_dependents();            // the Jacobian kernel may be scheduled behind this grid's last wave
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x * TRI_WARPS + warp;
  if (c >= a.n_cand) return;
  Cand cd;
  if (a.feat_off) {                   // direct mode: feature c of the caller's list
    const int o0 = a.feat_off[c], m = a.feat_off[c + 1] - o0;
    // the host may still be validating these lists: a malformed feature must neither read out of bounds nor be used
    bool bad = m < 1 || m > ORCVIO_MAX_OBS || o0 < 0 || o0 + m > a.direct_n_obs;
    if (!bad)
      for (int k = lane; k < m; k += 32) bad |= (unsigned)a.obs_clone[o0 + k] >= (unsigned)a.direct_n_clones;
    if (__any_sync(0xffffffffu, bad)) {
      if (lane == 0) {
        a.status[c] = 0;
        if (a.done) {
          __threadfence();
          asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(a.done + c), "r"(a.epoch) : "memory");
        }
      }
      return;
    }
    cd.filter = 0; cd.slot = c; cd.gen = c + 1; cd.flags = CAND_FORCE_TRI;
    cd.tri_off = o0; cd.tri_m = m;
    cd.cm_first_clone = a.obs_clone[o0];
    cd.cm_last_clone = a.obs_clone[o0 + m - 1];
    cd.cm_zu = a.obs_z[2 * (size_t)o0];
    cd.cm_zv = a.obs_z[2 * (size_t)o0 + 1];
  } else {
    cd = a.cand[c];
  }
  const double* clones = a.clones + (size_t)cd.filter * a.clone_stride;
  double* fp = a.fpos + ((size_t)cd.filter * a.fcap + cd.slot) * FP_STRIDE;
  long long* fgen = a.fgen + (size_t)cd.filter * a.fcap + cd.slot;
  int status = 0;
  int iters[2] = {0, 0};
  double cost = 0.0;
  bool is_init = (*fgen == cd.gen);   // initialised earlier in this track's life
  __syncwarp();                       // every lane has read fgen before lane 0 may overwrite it
  if (is_init && !(cd.flags & CAND_FORCE_TRI)) {
    status = ST_TRI_VALID;
  } else {
    const int* oc = a.obs_clone + cd.tri_off;
    const double* oz = a.obs_z + 2 * (size_t)cd.tri_off;
    int m = cd.tri_m;
    // checkMotion looks at the *full* observation list of the feature (jac list may be a
    // subset in the prune phase), first vs last-or-second-to-last.
    bool motion = check_motion(clones, cd.cm_first_clone, cd.cm_last_clone, cd.cm_zu, cd.cm_zv,
                               a.cfg.translation_threshold);
    if (motion && m >= 1) {
      double pos[3] = {fp[0], fp[1], fp[2]};
      __syncwarp();
      double fin[3] = {0.0, 0.0, 0.0};
      int v = triangulate_feature(clones, m, oc, oz, is_init, pos, a.cfg, iters, &cost, sm_all[warp],
                                  a.final_pos ? fin : nullptr);
      if (v) {
        if (lane == 0) {
          fp[0] = pos[0]; fp[1] = pos[1]; fp[2] = pos[2];
          *fgen = cd.gen;
          if (a.final_pos) { a.final_pos[3 * (size_t)c] = fin[0]; a.final_pos[3 * (size_t)c + 1] = fin[1]; a.final_pos[3 * (size_t)c + 2] = fin[2]; }
        }
        status = ST_TRI_VALID;
      }
    }
  }
  if (lane == 0) {
    a.status[c] = status;
    if (a.iters) { a.iters[2 * c] = iters[0]; a.iters[2 * c + 1] = iters[1]; }
    if (a.cost) a.cost[c] = cost;
    if (a.done) {                     // position, serial and status first, then the flag (release)
      __threadfence();
      asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(a.done + c), "r"(a.epoch) : "memory");
    }
  }
}

static int g_launch_errors = 0;
void check_launch(const char* name) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    ++g_launch_errors;
    std::fprintf(stderr, "[orcvio_b200] kernel launch failed: %s: %s\n", name, cudaGetErrorString(e));
  }
}
int launch_error_count() { return g_launch_errors; }
int env_int(const char* name, int dflt) {
  const char* e = std::getenv(name);
  return e ? std::atoi(e) : dflt;
}

void launch_triangulate(const TriArgs& a, cudaStream_t s) {
  if (a.n_cand <= 0) return;
  int blocks = (a.n_cand + TRI_WARPS - 1) / TRI_WARPS;
  // 158 registers (3 CTAs per SM) is the fastest single wave; past two waves of that (measured at 4096 features)
  // the 128-register build with 4 CTAs per SM wins
  if (blocks > 888) k_triangulate<4><<<blocks, 32 * TRI_WARPS, 0, s>>>(a);
  else k_triangulate<3><<<blocks, 32 * TRI_WARPS, 0, s>>>(a);
  check_launch("k_triangulate");
}

}  // namespace ob

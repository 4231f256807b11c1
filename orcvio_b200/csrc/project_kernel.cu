// Stage 3, object update -- dense left-nullspace projection of the stacked object block
// [H_f | H_x | r] with Householder reflections (objects.cu calls launch_project_dense).
#include "kernels.h"

namespace ob {

// Row-circular, column-absolute accessor of a row-major block.
struct Front {
  double* base;
  int ld;        // leading dimension (doubles)
  int rcap;      // number of physical rows (circular)
  int row0;      // physical index of logical row 0
  int cmask;     // physical column = j & cmask (power-of-two ring) ; ~0 = no wrap
  int rhs;       // physical column of the right-hand side
  __device__ __forceinline__ double& at(int i, int j) const {
    int pr = row0 + i;
    if (pr >= rcap) pr -= rcap;
    const int pc = (j < 0) ? rhs : (j & cmask);   // j = -1 addresses the right-hand side
    return base[(size_t)pr * ld + pc];
  }
};
#define FRONT_RHS (-1)

// CTA-wide Householder triangularisation of the logical rows [0, m) of `f` over the columns
// [c0, c1) plus the right-hand-side column.  On exit the block is upper
// trapezoidal (entries below the diagonal are zeroed).  All threads of the CTA call this.
__device__ void cta_householder(const Front& f, int m, int c0, int c1, double* sh, int nelim = -1) {
  const int tid = threadIdx.x, nt = blockDim.x;
  const int warp = tid >> 5, lane = tid & 31, nw = nt >> 5;
  const int ncol = c1 - c0;
  const int steps = min(nelim >= 0 ? nelim : ncol, m - 1);
  for (int k = 0; k < steps; ++k) {
    const int ck = c0 + k;
    // sigma = sum_{i>k} a(i,ck)^2 : warp partial sums -> shared
    double part = 0.0;
    for (int i = k + 1 + tid; i < m; i += nt) {
      double v = f.at(i, ck);
      part += v * v;
    }
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0) sh[warp] = part;
    __syncthreads();
    double sig = 0.0;
    for (int w = 0; w < nw; ++w) sig += sh[w];
    const double akk = f.at(k, ck);
    double t = 0.0, v0 = 1.0, mu = akk;
    if (sig > 0.0) {
      mu = sqrt(akk * akk + sig);
      v0 = (akk <= 0.0) ? (akk - mu) : (-sig / (akk + mu));
      t = 2.0 * v0 * v0 / (sig + v0 * v0);
    }
    __syncthreads();                       // everyone has read sh[] and a(k,ck)
    if (sig > 0.0) {
      const double iv0 = 1.0 / v0;
      for (int i = k + 1 + tid; i < m; i += nt) f.at(i, ck) *= iv0;   // v below the diagonal
      if (tid == 0) f.at(k, ck) = mu;
      __syncthreads();
      // apply to the remaining columns (one warp per column, rows over lanes)
      const int ntrail = (c1 - ck - 1) + 1;
      for (int jj = warp; jj < ntrail; jj += nw) {
        const int cj = (jj < c1 - ck - 1) ? (ck + 1 + jj) : FRONT_RHS;
        double dot = 0.0;
        for (int i = k + 1 + lane; i < m; i += 32) dot += f.at(i, ck) * f.at(i, cj);
        for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
        dot += f.at(k, cj);
        const double s = t * dot;
        __syncwarp();
        for (int i = k + 1 + lane; i < m; i += 32) f.at(i, cj) -= s * f.at(i, ck);
        if (lane == 0) f.at(k, cj) -= s;
      }
      __syncthreads();
      for (int i = k + 1 + tid; i < m; i += nt) f.at(i, ck) = 0.0;
    }
    // (next iteration touches column ck+1 first; the zeroing above cannot race with it)
  }
  __syncthreads();
}

// Left-nullspace projection of a dense block (removeLostObjects, src/orcvio.cpp:2162 ->
// nullspace_project_inplace_svd, math_utils.hpp:287-312): M = [H_f | H_x | r] (rows x ncols,
// row-major in global memory); Householder-eliminates the first `nelim` columns and applies the
// reflections to every column.  Rows [nelim, rows) of the trailing columns are A^T H_x, A^T r for
// an orthonormal basis A of null(H_f^T) (any basis gives the same gate value and posterior).
//
// k_project_dense_panel (the default): the reflections only depend on the H_f panel (rows x nelim <= 560 x 45), so
// every CTA keeps its own copy of the panel in shared memory, column-major (lanes over rows: conflict-free), factors
// it redundantly -- the same arithmetic in the same order in every CTA -- and carries PD_COLS trailing columns
// through the reflections IN REGISTERS (one warp per two columns, rows over lanes).  Each warp recomputes the
// column norm of step k itself, so a step costs ONE __syncthreads (the panel columns right of k are updated by the
// warps in turn) instead of three plus a pass over global memory: 140 x 154 block 2170 -> ~60 us.  Only the trailing
// columns are written back (the triangular factor of H_f is not used by the update).
constexpr int PD_THREADS = 512, PD_WARPS = PD_THREADS / 32, PD_CPW = 2, PD_COLS = PD_WARPS * PD_CPW;

// PD_RPL = rows per lane (rows <= 32 PD_RPL): 6 / 12 / 18 for blocks of up to 192 / 384 / 576 rows
template <int PD_RPL>
__global__ void __launch_bounds__(PD_THREADS) k_project_dense_panel(double* M, int rows, int ld, int nelim, int ncols) {
  extern __shared__ double pan[];                       // nelim columns of rpad doubles
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int rpad = (rows + 31) & ~31;
  for (int e = tid; e < rpad * nelim; e += PD_THREADS) pan[e] = 0.0;
  __syncthreads();
  for (int e = tid; e < rows * nelim; e += PD_THREADS) {  // coalesced along the rows of M
    const int i = e / nelim, c = e - i * nelim;
    pan[(size_t)c * rpad + i] = M[(size_t)i * ld + c];
  }
  double x[PD_CPW][PD_RPL];
  int cj[PD_CPW];
#pragma unroll
  for (int q = 0; q < PD_CPW; ++q) {
    cj[q] = nelim + blockIdx.x * PD_COLS + warp * PD_CPW + q;
#pragma unroll
    for (int j = 0; j < PD_RPL; ++j) {
      const int i = lane + 32 * j;
      x[q][j] = (cj[q] < ncols && i < rows) ? M[(size_t)i * ld + cj[q]] : 0.0;
    }
  }
  __syncthreads();
  const int steps = min(nelim, rows - 1);
  for (int k = 0; k < steps; ++k) {
    const double* ck = pan + (size_t)k * rpad;
    double sig = 0.0;
#pragma unroll
    for (int j = 0; j < PD_RPL; ++j) {
      const int i = lane + 32 * j;
      if (i > k && i < rows) { const double v = ck[i]; sig += v * v; }
    }
    for (int o = 16; o > 0; o >>= 1) sig += __shfl_xor_sync(0xffffffffu, sig, o);
    if (sig > 0.0) {                                   // (uniform over the CTA: every warp computes the same sig)
      const double akk = ck[k];
      const double mu = sqrt(akk * akk + sig);
      const double v0 = (akk <= 0.0) ? (akk - mu) : (-sig / (akk + mu));
      const double t = 2.0 * v0 * v0 / (sig + v0 * v0), iv0 = 1.0 / v0;
      // v = column k below the diagonal / v0: in registers while they last, else re-read from shared memory at each use
      constexpr bool VREG = PD_RPL <= 12;
      double v[VREG ? PD_RPL : 1];
      if (VREG) {
#pragma unroll
        for (int j = 0; j < PD_RPL; ++j) {
          const int i = lane + 32 * j;
          v[j] = (i > k && i < rows) ? ck[i] * iv0 : 0.0;
        }
      }
      auto vj = [&](int j) {
        if (VREG) return v[j];
        const int i = lane + 32 * j;
        return (i > k && i < rows) ? ck[i] * iv0 : 0.0;
      };
      const int jk = k >> 5, lk = k & 31;              // row k lives in lane lk, register jk
      // panel columns right of k, the warps in turn
      for (int c = k + 1 + warp; c < nelim; c += PD_WARPS) {
        double* cc = pan + (size_t)c * rpad;
        double dot = 0.0;
#pragma unroll
        for (int j = 0; j < PD_RPL; ++j) {
          const int i = lane + 32 * j;
          if (i > k && i < rows) dot += vj(j) * cc[i];
        }
        for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
        const double s = t * (dot + cc[k]);
        __syncwarp();
#pragma unroll
        for (int j = 0; j < PD_RPL; ++j) {
          const int i = lane + 32 * j;
          if (i > k && i < rows) cc[i] -= s * vj(j);
        }
        if (lane == lk) cc[k] -= s;
      }
      // own trailing columns
#pragma unroll
      for (int q = 0; q < PD_CPW; ++q) {
        double dot = 0.0, xk = 0.0;
#pragma unroll
        for (int j = 0; j < PD_RPL; ++j) {
          dot += vj(j) * x[q][j];
          if (j == jk) xk = x[q][j];
        }
        for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
        xk = __shfl_sync(0xffffffffu, xk, lk);
        const double s = t * (dot + xk);
#pragma unroll
        for (int j = 0; j < PD_RPL; ++j) {
          x[q][j] -= s * vj(j);
          if (j == jk && lane == lk) x[q][j] -= s;
        }
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int q = 0; q < PD_CPW; ++q)
    if (cj[q] < ncols) {
#pragma unroll
      for (int j = 0; j < PD_RPL; ++j) {
        const int i = lane + 32 * j;
        if (i < rows) M[(size_t)i * ld + cj[q]] = x[q][j];
      }
    }
}

// fallback for blocks whose panel does not fit in shared memory: one CTA on global memory
__global__ void __launch_bounds__(QR_THREADS) k_project_dense(double* M, int rows, int ld, int nelim, int ncols) {
  __shared__ double red[32];
  Front f{M, ld, rows, 0, 0x7fffffff, ncols - 1};
  cta_householder(f, rows, 0, ncols - 1, red, nelim);
}

void launch_project_dense(double* M, int rows, int ld, int nelim, int ncols, cudaStream_t s) {
  const int rpad = (rows + 31) & ~31;
  const size_t smem = (size_t)rpad * nelim * sizeof(double);
  if (rows <= 32 * 18 && smem <= 220 * 1024 && ncols > nelim) {
    static bool attr = false;
    if (!attr) {
      cudaFuncSetAttribute(k_project_dense_panel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
      cudaFuncSetAttribute(k_project_dense_panel<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
      cudaFuncSetAttribute(k_project_dense_panel<18>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
      attr = true;
    }
    const int grid = (ncols - nelim + PD_COLS - 1) / PD_COLS;
    if (rows <= 32 * 6) k_project_dense_panel<6><<<grid, PD_THREADS, smem, s>>>(M, rows, ld, nelim, ncols);
    else if (rows <= 32 * 12) k_project_dense_panel<12><<<grid, PD_THREADS, smem, s>>>(M, rows, ld, nelim, ncols);
    else k_project_dense_panel<18><<<grid, PD_THREADS, smem, s>>>(M, rows, ld, nelim, ncols);
    check_launch("k_project_dense_panel");
    return;
  }
  k_project_dense<<<1, QR_THREADS, 0, s>>>(M, rows, ld, nelim, ncols);
  check_launch("k_project_dense");
}

}  // namespace ob

// Stages 4+5 -- measurement compression in the whitened ("A") form and the EKF
// update written around it.
//
// Reference: OrcVIO::measurementUpdate_msckf / measurementUpdate_hybrid
// (src/orcvio.cpp:1654-1763, 1766-1950): when rows > cols the stacked H (M x (L+6N)) is
// compressed with SuiteSparseQR to H_thin = (Q^T H).topRows, then
//     S = H P H^T + s^2 I,  K = P H^T S^-1,  dx = K r,  P <- (I - K H) P,  P <- (P + P^T)/2.
// On a GPU the QR is a chain of ~6N dependent Householder steps per clone block (pure latency:
// milliseconds on the stress frame, DESIGN.md).  This file produces the same posterior from
// massively parallel dense kernels:
//   P = F F^T                 Cholesky of the prior in the order [clones | IMU]  (k_chol_prior,
//                             on a second stream, overlapped with triangulation + Jacobians);
//                             F_1 = first 6N columns, F_2 = the rest, L = F[clones, clones]
//   A = H' L                  every gated, nullspace-projected row times L        (k_aform)
//   W = s^2 I + A^T A, v = A^T r'                                                 (k_syrk, k_syrk_reduce)
//   W = C C^T, Y = C^-1 F_1^T, y = C^-1 v     Cholesky with F_1 and v carried as extra rows
//                                              (k_chol_w_solve, strips of F_1 on separate SMs)
//   dx = Y^T y                                                                    (k_dx)
//   P+ = s^2 Y^T Y + F_2 F_2^T                                                    (k_pinfo)
// Derivation: with A = H L the gain is K = F_1 (A^T A + s^2 I)^-1 A^T (push-through identity),
// hence dx = F_1 W^-1 A^T r and P+ = P - F_1 (I - s^2 W^-1) F_1^T = s^2 F_1 W^-1 F_1^T + F_2 F_2^T:
// exactly the reference's posterior, symmetric positive semidefinite by construction (the
// reference's trailing (P + P^T)/2 is the identity on it).
// Numerics: H' L is formed ROW BY ROW before anything is squared.  A VIO prior has a large
// common-mode variance (global position / yaw) along which every row of H' is (numerically) zero;
// multiplying by L first performs that cancellation inside one row (error eps |h| |L|), whereas
// forming G = H'^T H' first and then L^T G L loses a factor ~rows (measured 2e-9 vs 1e-12 on the
// Unity-shaped sequence; DESIGN.md "numerics").
#include "kernels.h"
#include "increment.cuh"
#include "chol.cuh"

namespace ob {

// ---------------------------------------------------------------- prior factor
// P = F F^T in the order [clone columns 22..D-1 | IMU columns 0..21].  Outputs
//   FT (n x ldt, UpdArgs::T): FT[k][c] = F[perm(c)][k] for k < n, c = original column index,
//   Ls (22 x 22): the trailing factor of the IMU block given the clones (F_2 F_2^T = Ls Ls^T).
__global__ void __launch_bounds__(CHOL_THREADS) k_chol_prior(UpdArgs a) {
  extern __shared__ double sm[];
  __shared__ __align__(16) CholShared cs;
  const int fi = blockIdx.x;
  const FilterWork fw = a.fw[fi];
  if (!fw.active) return;
  const int D = fw.D, n = fw.D - ORCVIO_LEG, L = ORCVIO_LEG;   // n = 6N (+ E feature states behind the clones)
  const double* P = a.P + (size_t)fi * a.p_stride;
  double* FT = a.T + (size_t)fi * a.t_stride;
  double* A = sm;
  double* tol = A + chol_smem_doubles(n, L);
  const int tid = threadIdx.x, nt = blockDim.x;
  const int warp = tid >> 5, lane = tid & 31, nw = nt >> 5;
  auto orig = [&](int q) { return q < n ? L + q : q - n; };
  // only the n clone (+ feature) columns are pivots: the 22 IMU rows ride along as carried rows, so the chain is n / 8
  // steps long and F_1 is complete when it ends; the IMU block's own factor (k_imu_factor) is off the critical path
  chol_init(A, cs, n, L);
  __syncthreads();
  const int ldp = a.ldp;
  chol_load_rows(A, n, 0, D, [&](int i, int j) { return P + (size_t)orig(i) * ldp + orig(j); });
  for (int i = tid; i < n; i += nt) tol[i] = 1e-12 * fabs(P[(size_t)orig(i) * (ldp + 1)]);
  // entries above the diagonal of F are structural zeros: FT[k][orig(i)] = 0 for i < k
  for (int k = warp; k < n; k += nw)
    for (int i = lane; i < k; i += 32) FT[(size_t)k * a.ldt + L + i] = 0.0;
  chol_cp_async_wait();
  cta_cholesky(A, cs, tol, n, L);
  const int ldt = a.ldt;
  chol_for_rows(A, n, L, 0, [&](int i, int k, double l) { FT[(size_t)k * ldt + orig(i)] = l; });
}

// Ls Ls^T = P_II - X X^T: the factor of the IMU block given the clones (F_2 F_2^T = Ls Ls^T), X = the IMU rows of F_1
// (FT[k][0..21]).  One CTA per filter, behind k_chol_prior on the side stream; only k_pinfo needs it.  Pivots
// <= 1e-12 P_kk are exact zeros (rows 15..21 are zero and, after augmentation, the IMU pose duplicates the newest clone).
__global__ void __launch_bounds__(256) k_imu_factor(UpdArgs a, double* Ls_all) {
  extern __shared__ double sm[];                          // X^T: n x 22, then S: 22 x 23
  constexpr int L = ORCVIO_LEG;
  const int fi = blockIdx.x;
  const FilterWork fw = a.fw[fi];
  if (!fw.active) return;
  const int n = fw.D - L;
  const double* P = a.P + (size_t)fi * a.p_stride;
  const double* FT = a.T + (size_t)fi * a.t_stride;
  double* Ls = Ls_all + (size_t)fi * L * L;
  double* X = sm;
  double* S = sm + (size_t)n * L;
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int e = tid; e < n * L; e += nt) X[e] = FT[(size_t)(e / L) * a.ldt + e % L];
  __syncthreads();
  for (int e = tid; e < L * L; e += nt) {
    const int i = e / L, j = e % L;
    if (j > i) continue;
    double s0 = 0.0, s1 = 0.0;
    int k = 0;
    for (; k + 1 < n; k += 2) {
      s0 += X[(size_t)k * L + i] * X[(size_t)k * L + j];
      s1 += X[(size_t)(k + 1) * L + i] * X[(size_t)(k + 1) * L + j];
    }
    if (k < n) s0 += X[(size_t)k * L + i] * X[(size_t)k * L + j];
    S[i * (L + 1) + j] = P[(size_t)i * a.ldp + j] - (s0 + s1);
  }
  __syncthreads();
  if (tid < 32) {                                         // lane i owns row i
    const int i = tid;
    const double tol_i = i < L ? 1e-12 * fabs(P[(size_t)i * (a.ldp + 1)]) : 0.0;
    for (int c = 0; c < L; ++c) {
      const double pv = S[c * (L + 1) + c];
      __syncwarp();                                       // every lane has the pivot before lane c overwrites it
      const double tc = __shfl_sync(0xffffffffu, tol_i, c);
      const bool ok = pv > tc;
      const double d = ok ? sqrt(pv) : 0.0;
      const double id = ok ? 1.0 / d : 0.0;
      double lic = 0.0;
      if (i < L && i >= c) {
        lic = (i == c) ? d : S[i * (L + 1) + c] * id;
        S[i * (L + 1) + c] = lic;
      }
      __syncwarp();
      if (i < L && i > c)
        for (int j = c + 1; j <= i; ++j) S[i * (L + 1) + j] -= lic * S[j * (L + 1) + c];
      __syncwarp();
    }
  }
  __syncthreads();
  for (int e = tid; e < L * L; e += nt) {
    const int i = e / L, j = e % L;
    Ls[e] = j <= i ? S[i * (L + 1) + j] : 0.0;
  }
}

// ---------------------------------------------------------------- A = [r' | H' L]   (FP64 tensor cores)
// One CTA per row tile (features sorted by first clone; window [c0, c1) of clone blocks, <= 64 rows).
// The gated rows are assembled densely in shared memory (Hs, rows x W); the tile of A is the product
// Hs (rows x W) * Lwin (W x 6 c1) with Lwin = L[6 c0 .. 6 c1, 0 .. 6 c1): L is lower triangular, so A is
// structurally zero right of column 6 c1 (the staircase k_syrk exploits).  Every warp owns 8-column
// fragments of A: the B operand (8 columns of L over the window rows) is read once from the prior factor
// into registers, the A operand comes from shared memory (row stride == 4 mod 8: conflict-free 64-bit
// fragment loads), eight m8n8k4 accumulators (64 rows) are in flight per warp.
// Column layout of A: column 0 = projected residual r', column 1 + j = (H' L)[:, j].
constexpr int AF_THREADS = 192;              // x 3 CTAs per SM (launch bound): the tiles of a 4096-feature frame in one wave
constexpr int AF_KS = 9;                     // k-steps (of 4) per register chunk of the B operand: 36 columns

__device__ __forceinline__ int aform_stride(int W) {          // smallest stride >= W with stride % 8 == 4
  const int k4 = (W + 3) & ~3;
  return (k4 & 7) == 4 ? k4 : k4 + 4;
}

__global__ void __launch_bounds__(AF_THREADS, 3) k_aform(AformArgs a, const double* FT_all, size_t t_stride, int ldt,
                                                      double* Amat, int lda, int* tile_rows) {
  extern __shared__ double smem[];
  __shared__ int rowbase[256];
  __shared__ int wsum[AF_THREADS / 32];
  __shared__ double res[AFORM_TILE_ROWS];
  const Tile tl = a.tiles[blockIdx.x];
  const FilterWork fw = a.fw[tl.filter];
  const int W = 6 * (tl.c1_blk - tl.c0_blk);
  const int Wp = aform_stride(W);
  const int tid = threadIdx.x, nt = blockDim.x;
  const int warp = tid >> 5, lane = tid & 31, nw = nt >> 5;
  const int nc = tl.cand_end - tl.cand_begin;      // host guarantees nc <= 256
  const int rows_ub = tl.rows;                     // <= AFORM_TILE_ROWS
  const int rows8 = (rows_ub + 7) & ~7;
  for (int e = tid; e < rows8 * Wp; e += nt) smem[e] = 0.0;
  if (tid < AFORM_TILE_ROWS) res[tid] = 0.0;
  // ---- row bases of the gated candidates (block scan)
  int total = 0;
  for (int base = 0; base < nc; base += nt) {
    const int q = base + tid;
    int r = 0;
    if (q < nc) {
      const int c = tl.cand_begin + q;
      if (a.order_f) {                // direct mode: candidate c is feature order_f[c]
        const int f = a.order_f[c];
        if (a.status_f[f] & ST_GATE_PASS) r = 2 * (a.feat_off[f + 1] - a.feat_off[f]) - 3;
      } else {
        const int st = a.status_f ? a.status_f[a.cand[c].slot] : a.status[c];
        if (st & ST_GATE_PASS) r = 2 * a.cand[c].jac_m - 3;
      }
    }
    int incl = r;
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    int off = total;
    for (int w2 = 0; w2 < warp; ++w2) off += wsum[w2];
    if (q < nc) rowbase[q] = (r > 0) ? (off + incl - r) : -1;
    for (int w2 = 0; w2 < nw; ++w2) total += wsum[w2];
    __syncthreads();
  }
  const int m = total;
  if (tid == 0) tile_rows[blockIdx.x] = m;
  __syncthreads();
  for (int q = warp; q < nc; q += nw) {
    if (rowbase[q] < 0) continue;
    const int c = tl.cand_begin + q;
    Cand cd;
    if (a.order_f) {
      const int f = a.order_f[c];
      cd.jac_m = a.feat_off[f + 1] - a.feat_off[f];
      cd.s_blk = a.sblk_f[f]; cd.e_blk = a.eblk_f[f];
      cd.hblk_off = a.hblkoff_f[f]; cd.row_off = a.rowoff_f[f];
    } else {
      cd = a.cand[c];
    }
    const int r = 2 * cd.jac_m - 3;
    const int w = 6 * (cd.e_blk - cd.s_blk + 1);
    const int coff = 6 * (cd.s_blk - tl.c0_blk);
    const double* hb = a.hblk + cd.hblk_off;
#pragma unroll 4
    for (int e = lane; e < r * w; e += 32) {
      const int i = e / w, j = e - i * w;
      smem[(size_t)(rowbase[q] + i) * Wp + coff + j] = hb[e];
    }
    for (int i = lane; i < r; i += 32) res[rowbase[q] + i] = a.rblk[cd.row_off + i];
  }
  __syncthreads();
  // ---- fragments: A columns [8 cf, 8 cf + 8); A column ac <-> column ac - 1 of L
  const int ncol_nz = 6 * tl.c1_blk + 1;           // structurally non-zero columns of A for this tile
  const int ncf = (ncol_nz + 7) >> 3;
  const int fr = lane >> 2, fk = lane & 3;
  const double* FT = FT_all + (size_t)tl.filter * t_stride;
  double* Arow = Amat + (size_t)tl.arow * lda;
  const int nrf = rows8 >> 3;                      // row fragments (<= 8)
  // flat sequence of steps (column fragment, 36-column chunk of the window); the B operand of step s + 1 is
  // fetched from the prior factor (L2) while the MMAs of step s run
  const int nchunk = (W + 4 * AF_KS - 1) / (4 * AF_KS);
  const int nsteps = ((ncf - warp + nw - 1) / nw) * nchunk;      // steps of this warp (ncf > warp, else <= 0)
  auto load_b = [&](int step, double* b) {
    const int cf = warp + nw * (step / nchunk), k0 = (step % nchunk) * 4 * AF_KS;
    const int jl = 8 * cf + fr - 1;                  // column of L behind this lane's B elements
    const bool jok = (jl >= 0) && (jl < 6 * tl.c1_blk);
    // L[k][jl] = FT[jl][22 + k] (zero above the diagonal, stored explicitly), k = 6 c0 + window column
    const double* src = FT + (size_t)(jok ? jl : 0) * ldt + ORCVIO_LEG + 6 * tl.c0_blk;
#pragma unroll
    for (int s2 = 0; s2 < AF_KS; ++s2) {
      const int k = k0 + 4 * s2 + fk;
      b[s2] = (jok && k < W) ? src[k] : 0.0;
    }
  };
  double bn[AF_KS];
  if (nsteps > 0) load_b(0, bn);
  double2 acc[8];
  for (int step = 0; step < nsteps; ++step) {
    const int cf = warp + nw * (step / nchunk), ch = step % nchunk, k0 = ch * 4 * AF_KS;
    double b[AF_KS];
#pragma unroll
    for (int s2 = 0; s2 < AF_KS; ++s2) b[s2] = bn[s2];
    if (step + 1 < nsteps) load_b(step + 1, bn);
    if (ch == 0) {
#pragma unroll
      for (int u = 0; u < 8; ++u) acc[u] = make_double2(0.0, 0.0);
    }
#pragma unroll
    for (int s2 = 0; s2 < AF_KS; ++s2) {
      if (k0 + 4 * s2 < W) {
        const double* hs = smem + (size_t)fr * Wp + k0 + 4 * s2 + fk;
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (u < nrf) dmma884(acc[u].x, acc[u].y, hs[(size_t)(8 * u) * Wp], b[s2]);
      }
    }
    if (ch == nchunk - 1) {
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int row = 8 * u + fr;
        if (u < nrf && row < rows_ub) {
          double2 v = acc[u];
          if (cf == 0 && fk == 0) v.x = res[row];    // column 0: the projected residual
          *reinterpret_cast<double2*>(Arow + (size_t)row * lda + 8 * cf + 2 * fk) = v;
        }
      }
    }
  }
  // ---- explicit zeros right of the staircase, as far as k_syrk reads this tile's rows: column tile J is read
  // from row jrow0[J] on, and tiles are not strictly ordered by c1
  int zend = 8 * ncf;
  for (int J = 0; J < SY_MAXT; ++J)
    if (fw.jrow0[J] <= tl.arow - fw.arow0) zend = max(zend, min(lda, SY_TILE * (J + 1)));
  const int z0 = 8 * ncf, zw = zend - z0;
  if (zw > 0)
    for (int e = tid; e < rows_ub * zw; e += nt) {
      const int row = e / zw, c = e - row * zw;
      Arow[(size_t)row * lda + z0 + c] = 0.0;
    }
}

// Dense variant for the object update: A = [r' | Hp L] for a projected dense block Hp (rows x n,
// row-major with leading dimension ldh, residual in column n of Hp).
__global__ void __launch_bounds__(256) k_aform_dense(const double* Hp, int ldh, int rows, int n, const double* FT,
                                                     int ldt, double* Amat, int lda) {
  const int row = blockIdx.x;
  if (row >= rows) return;
  const double* h = Hp + (size_t)row * ldh;
  for (int j = threadIdx.x; j <= n; j += blockDim.x) {
    if (j == n) { Amat[(size_t)row * lda] = h[n]; continue; }
    // L[k][j] = FT[j][22 + k], zero for k < j
    const double* src = FT + (size_t)j * ldt + ORCVIO_LEG;
    double s0 = 0.0, s1 = 0.0;
    int k = j;
    for (; k + 1 < n; k += 2) { s0 += h[k] * src[k]; s1 += h[k + 1] * src[k + 1]; }
    if (k < n) s0 += h[k] * src[k];
    Amat[(size_t)row * lda + 1 + j] = s0 + s1;
  }
  // columns (n, lda) of the last column tile must read as zeros in k_syrk
  for (int c = n + 1 + threadIdx.x; c < lda; c += blockDim.x) Amat[(size_t)row * lda + c] = 0.0;
}

// ---------------------------------------------------------------- W_aug = s^2 I + A^T A  (FP64 tensor cores)
// grid (work units, filters).  A work unit is one 64 x 64 tile (I <= J) of A^T A over one chunk of rows
// (syrk_plan): pair (I, J) only covers the rows [jrow0[J], arows) -- above them column tile J of A is
// structurally zero.  8 warps x (32 x 16) warp tiles = 4 x 2 accumulator fragments of mma.m8n8k4.f64 per
// warp, operands staged through shared memory in 32-row slabs (row stride 68 doubles: the four k-rows of
// a fragment start 8 banks apart, so the 64-bit fragment loads are conflict-free).
// Split-K, two levels, no atomics on data: every chunk stores its partial tile; the last chunk of a GROUP
// to arrive (device-scope counter) adds the group's partials in chunk order and stores the group sum; the
// last group to arrive adds the group sums in group order.  Grouping is static, so the summation order is
// fixed and the result is bitwise reproducible.  The final reducer writes the lower triangle of
// W_aug ((n+1) x ldr, UpdArgs::S): A's column 0 (the residual) maps to row n (v = A^T r', corner r'^T r'),
// column 1 + j to index j, with s^2 added on the first n diagonal entries.
constexpr int SY_T = SY_TILE, SY_KS = 32, SY_LD = 68;
// Operand pipeline: SY_STAGES slabs of 32 rows x 64 columns of A (column tile I) and of column tile J (a diagonal pair:
// 64 rows of its one tile), brought in by cp.async (LDGSTS, 16 bytes per copy, zero-fill past the end of the chunk) one
// slab ahead of the MMAs; one __syncthreads per slab.  (A TMA variant -- one cp.async.bulk per slab row, mbarrier
// producer warp -- was built and measured slower; deeper rings and 64-row slabs for every unit change nothing: DESIGN.md.)
constexpr int SY_THREADS = 256;
constexpr int SY_STAGES = 2;
constexpr int SY_STAGE_DOUBLES = 2 * SY_KS * SY_LD;

__device__ __forceinline__ unsigned int smem_u32(const void* p) { return (unsigned int)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned int parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tSY_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra SY_DONE;\n\tbra SY_WAIT;\n\tSY_DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long* bar, unsigned int bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned int bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ORCVIO_SYRK_DBG=1: per-CTA time stamps (globaltimer, ns) of the phases of k_syrk, read back by orcvio_syrk_debug()
__device__ long long* g_syrk_dbg = nullptr;
constexpr int SY_DBG_N = 8;
__device__ __forceinline__ void sy_stamp(int unit, int k) {
  if (g_syrk_dbg && threadIdx.x == 0) {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_syrk_dbg[(size_t)unit * SY_DBG_N + k] = t;
  }
}

// Diagonal pair (I, I): of the 8 x 8 grid of 8 x 8 fragments only those with fragment row <= fragment column hold an
// element that is ever emitted -- 36 of 64.  They are dealt to the warps so that the two warps of a scheduler (w and
// w + 4) carry 9 of them (fragment rows 0 + 7, 1 + 6, 2 + 5, 3 + 4): the tensor pipe is per scheduler, so a diagonal
// unit does 9/16 of the DMMA work of an off-diagonal one per slab and gets 13/8 as many rows (syrk_plan).
// Entry = fragment row << 4 | fragment column; 0xff = none.
__constant__ unsigned char SY_DIAG_FRAG[8][5] = {
    {0x00, 0x01, 0x02, 0x03, 0x04}, {0x11, 0x12, 0x13, 0x14, 0x15}, {0x22, 0x23, 0x24, 0x25, 0x26},
    {0x33, 0x34, 0x35, 0x36, 0x37}, {0x05, 0x06, 0x07, 0x77, 0xff}, {0x16, 0x17, 0x66, 0x67, 0xff},
    {0x27, 0x55, 0x56, 0x57, 0xff}, {0x44, 0x45, 0x46, 0x47, 0xff}};

__global__ void __launch_bounds__(SY_THREADS) k_syrk(UpdArgs a, const double* __restrict__ Amat, int lda, double* part,
                                                     int max_units, int cta_budget, int group, const Tile* tiles,
                                                     const int* tile_rows, int* filter_rows, unsigned int* counters,
                                                     int spin_reduce) {
  extern __shared__ __align__(128) double sy_sm[];
  const int fi = blockIdx.y;
  const FilterWork fw = a.fw[fi];
  const int tid = threadIdx.x;
  const int unit = blockIdx.x;
  sy_stamp(unit, 0);
  if (unit == 0 && tid < 32) {                           // gated rows of this filter (k_pinfo skips P when 0): warp 0
    int rows = 0;
    if (fw.active) {
      if (tiles == nullptr) rows = (tid == 0) ? fw.arows : 0;   // dense (object) update: every row counts
      else {
        for (int t = fw.tile_begin + tid; t < fw.tile_end; t += 32) rows += tile_rows[t];
        if (tid == 0) rows += fw.dense_rows;             // hybrid mode: rows of the EKF-SLAM features
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rows += __shfl_xor_sync(0xffffffffu, rows, o);
    if (tid == 0) filter_rows[fi] = rows;
  }
  if (!fw.active) return;
  const int n = fw.D - ORCVIO_LEG, n1 = n + 1;
  const SyrkPlan pl = syrk_plan(fw, cta_budget);
  if (unit >= pl.total) return;
  // work unit -> pair (I, J), I <= J, and chunk
  int I = 0, J = 0, pidx = 0;
  {
    int q = 0;
    for (int ii = 0; ii < pl.nt; ++ii)
      for (int jj = ii; jj < pl.nt; ++jj) {
        if (unit >= pl.first[q]) { I = ii; J = jj; pidx = q; }
        ++q;
      }
  }
  const int chunk = unit - pl.first[pidx];
  const int nchunks = pl.first[pidx + 1] - pl.first[pidx];
  const bool diag = (I == J);
  const int kc = diag ? pl.kcd : pl.kc;
  const int row_begin = min(fw.arows, fw.jrow0[J] + chunk * kc);
  const int row_end = min(fw.arows, row_begin + kc);
  const double* A = Amat + (size_t)fw.arow0 * lda;
  __shared__ int s_last;
  const int warp = tid >> 5, lane = tid & 31;
  const int i0 = I * SY_T, j0 = J * SY_T;
  // a diagonal pair needs one matrix, so its stage holds 64 rows of it (the A half and the B half) per barrier
  const int slab_rows = diag ? 2 * SY_KS : SY_KS;
  const int nslab = (row_end - row_begin + slab_rows - 1) / slab_rows;
  double2 acc[4][2];
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int v = 0; v < 2; ++v) acc[u][v] = make_double2(0.0, 0.0);
  const int fr = lane >> 2, fk = lane & 3;               // fragment row (or column) / k index
  const int wi = (warp & 1) * 32, wj = (warp >> 1) * 16;
  int du[5], dv[5];                                      // diagonal pair: this warp's fragments (acc[t >> 1][t & 1])
#pragma unroll
  for (int t = 0; t < 5; ++t) {
    const int f = SY_DIAG_FRAG[warp][t];
    du[t] = (f == 0xff) ? -1 : 8 * (f >> 4);
    dv[t] = (f == 0xff) ? 0 : 8 * (f & 15);
  }
  // loader: 32 rows x 64 columns per matrix = 1024 x 16 bytes, four per thread and matrix (rows lr, lr+8, lr+16, lr+24);
  // rows past the end of A and columns past lda are zero-filled by the copy itself (src-size 0)
  const int lr = tid >> 5, lc = (tid & 31) * 2;
  const bool ci_ok = (i0 + lc < lda), cj_ok = (j0 + lc < lda);
  auto issue = [&](int it) {
    if (it < nslab) {
      const int st = it % SY_STAGES;
      double* sa = sy_sm + (size_t)st * SY_STAGE_DOUBLES;
      const int r0 = row_begin + it * slab_rows;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int rl = lr + 8 * q, r = r0 + rl;
        const bool rok = r < row_end;
        const double* src = A + (size_t)(rok ? r : row_begin) * lda;
        const unsigned int da = smem_u32(sa + rl * SY_LD + lc);
        const int na = (rok && ci_ok) ? 16 : 0;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(da), "l"(src + (ci_ok ? i0 + lc : 0)), "r"(na) : "memory");
        if (!diag) {
          const int nb = (rok && cj_ok) ? 16 : 0;
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(da + (unsigned int)(SY_KS * SY_LD * sizeof(double))),
                       "l"(src + (cj_ok ? j0 + lc : 0)), "r"(nb) : "memory");
        } else {                                         // rows 32 .. 63 of the slab, same columns
          const bool rok2 = r + SY_KS < row_end;
          const double* src2 = A + (size_t)(rok2 ? r + SY_KS : row_begin) * lda;
          const int nb = (rok2 && ci_ok) ? 16 : 0;
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(da + (unsigned int)(SY_KS * SY_LD * sizeof(double))),
                       "l"(src2 + (ci_ok ? i0 + lc : 0)), "r"(nb) : "memory");
        }
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  sy_stamp(unit, 1);
  if (g_syrk_dbg && tid == 0 && spin_reduce) {             // (slots 5 .. 7 are free in the spin path)
    g_syrk_dbg[(size_t)unit * SY_DBG_N + 5] = row_end - row_begin;
    g_syrk_dbg[(size_t)unit * SY_DBG_N + 6] = I * 16 + J;
    g_syrk_dbg[(size_t)unit * SY_DBG_N + 7] = fw.jrow0[J];
  }
#pragma unroll
  for (int it = 0; it < SY_STAGES - 1; ++it) issue(it);
  for (int it = 0; it < nslab; ++it) {
    asm volatile("cp.async.wait_group %0;" ::"n"(SY_STAGES - 2) : "memory");
    __syncthreads();                                     // slab `it` has landed for everyone; slab it-1 is consumed
    issue(it + SY_STAGES - 1);
    const int st = it % SY_STAGES;
    const double(*As)[SY_LD] = reinterpret_cast<const double(*)[SY_LD]>(sy_sm + (size_t)st * SY_STAGE_DOUBLES);
    if (diag) {
#pragma unroll 8
      for (int k4 = 0; k4 < 2 * SY_KS; k4 += 4) {
        double af[5], bf[5];
#pragma unroll
        for (int t = 0; t < 5; ++t) {
          af[t] = As[k4 + fk][max(du[t], 0) + fr];
          bf[t] = As[k4 + fk][dv[t] + fr];
        }
#pragma unroll
        for (int t = 0; t < 5; ++t)
          if (du[t] >= 0) dmma884(acc[t >> 1][t & 1].x, acc[t >> 1][t & 1].y, af[t], bf[t]);
      }
      continue;
    }
    const double(*Bp)[SY_LD] = As + SY_KS;
#pragma unroll
    for (int k4 = 0; k4 < SY_KS; k4 += 4) {
      double af[4], bf[2];
#pragma unroll
      for (int u = 0; u < 4; ++u) af[u] = As[k4 + fk][wi + 8 * u + fr];
#pragma unroll
      for (int v = 0; v < 2; ++v) bf[v] = Bp[k4 + fk][wj + 8 * v + fr];
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 2; ++v) dmma884(acc[u][v].x, acc[u][v].y, af[u], bf[v]);
    }
  }
  sy_stamp(unit, 2);
  // tile element (ii, jj) = (A^T A)[i0 + ii][j0 + jj]; fragment (u, v): ii = wi + 8u + fr, jj = wj + 8v + 2fk (+1)
  double* S = a.S + (size_t)fi * a.r_stride;
  auto emit = [&](int ii, int jj, double s) {
    const int ga = i0 + ii, gb = j0 + jj;                // columns of A, each unordered pair once: ga <= gb
    if (gb > n || ga > gb) return;
    if (ga == 0) { S[(size_t)n * a.ldr + (gb == 0 ? n : gb - 1)] = s; return; }   // v = A^T r', corner r'^T r'
    if (ga == gb) s += a.sigma2;
    S[(size_t)(gb - 1) * a.ldr + (ga - 1)] = s;          // lower triangle of W
  };
  (void)n1;
  if (nchunks == 1) {
    if (diag) {
#pragma unroll
      for (int t = 0; t < 5; ++t)
        if (du[t] >= 0) {
          emit(du[t] + fr, dv[t] + 2 * fk, acc[t >> 1][t & 1].x);
          emit(du[t] + fr, dv[t] + 2 * fk + 1, acc[t >> 1][t & 1].y);
        }
      return;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int v = 0; v < 2; ++v) {
        emit(wi + 8 * u + fr, wj + 8 * v + 2 * fk, acc[u][v].x);
        emit(wi + 8 * u + fr, wj + 8 * v + 2 * fk + 1, acc[u][v].y);
      }
    return;
  }
  double* base = part + ((size_t)fi * max_units + pl.first[pidx]) * (SY_T * SY_T);
  const size_t cstride = (size_t)(SY_T * SY_T);
  double* out = base + (size_t)chunk * cstride;
  if (diag) {                                            // (the fragments below the diagonal are never stored nor read)
#pragma unroll
    for (int t = 0; t < 5; ++t)
      if (du[t] >= 0) *reinterpret_cast<double2*>(out + (du[t] + fr) * SY_T + dv[t] + 2 * fk) = acc[t >> 1][t & 1];
  } else {
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int v = 0; v < 2; ++v)
        *reinterpret_cast<double2*>(out + (wi + 8 * u + fr) * SY_T + wj + 8 * v + 2 * fk) = acc[u][v];
  }
  if (spin_reduce) {
    // Every chunk of this pair is resident (the host only sets spin_reduce when the whole grid fits the GPU at once):
    // wait until all of them have stored their partial, then reduce ONE SLICE of the tile over all chunks -- in chunk
    // order, so the sum is reproducible -- and emit it.  All CTAs of the pair reduce in parallel: one L2 round trip
    // instead of the two serial last-arriver passes below.
    unsigned int* cnt = counters + ((size_t)fi * SY_MAXP + pidx) * (SY_MAXG + 1);
    __threadfence();
    __syncthreads();
    if (tid == 0) {
      atomicAdd(cnt, 1u);
      unsigned int v;
      for (;;) {
        asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(cnt) : "memory");
        if (v >= (unsigned int)nchunks) break;
        __nanosleep(64);
      }
      asm volatile("fence.acq_rel.gpu;" ::: "memory");
    }
    __syncthreads();
    sy_stamp(unit, 3);
    const int per = (SY_T * SY_T + nchunks - 1) / nchunks;
    const int e0 = chunk * per, e1 = min(SY_T * SY_T, e0 + per);
    // same association as the two-level path below (chunks in order inside a group of gsz, then the group sums in
    // order), so a filter gives the same bits whichever of the two reductions its batch ends up with
    int gsz = group;
    if ((nchunks + gsz - 1) / gsz > SY_MAXG) gsz = (nchunks + SY_MAXG - 1) / SY_MAXG;
    const int ngroups = (nchunks + gsz - 1) / gsz;
    for (int e = e0 + tid; e < e1; e += 256) {
      if (diag && ((e >> 6) >> 3) > ((e & 63) >> 3)) continue;   // a fragment below the diagonal: nothing was stored
      const double* p0 = base + e;
      double total = 0.0;
      for (int g0 = 0; g0 < nchunks; g0 += gsz) {
        const int g1 = min(nchunks, g0 + gsz);
        double gs = 0.0;
        int c = g0;
        for (; c + 3 < g1; c += 4) {
          const double x0 = __ldcg(p0 + (size_t)c * cstride), x1 = __ldcg(p0 + (size_t)(c + 1) * cstride);
          const double x2 = __ldcg(p0 + (size_t)(c + 2) * cstride), x3 = __ldcg(p0 + (size_t)(c + 3) * cstride);
          gs = (((gs + x0) + x1) + x2) + x3;
        }
        for (; c < g1; ++c) gs += __ldcg(p0 + (size_t)c * cstride);
        total = (ngroups > 1) ? total + gs : gs;
      }
      emit(e >> 6, e & 63, total);
    }
    sy_stamp(unit, 4);
    __syncthreads();
    if (tid == 0 && atomicAdd(cnt + 1, 1u) == (unsigned int)(nchunks - 1)) { cnt[0] = 0u; cnt[1] = 0u; }   // ready for the next launch
    return;
  }
  // ---- level 1: the last chunk of a group sums the group (16 tile elements per thread)
  int gsz = group;
  if ((nchunks + gsz - 1) / gsz > SY_MAXG) gsz = (nchunks + SY_MAXG - 1) / SY_MAXG;
  const int ngroups = (nchunks + gsz - 1) / gsz;
  const int g = chunk / gsz;
  const int c_begin = g * gsz, c_end = min(nchunks, c_begin + gsz);
  unsigned int* cnt = counters + ((size_t)fi * SY_MAXP + pidx) * (SY_MAXG + 1);
  __threadfence();
  __syncthreads();
  if (tid == 0) s_last = (atomicAdd(cnt + 1 + g, 1u) == (unsigned int)(c_end - c_begin - 1));
  __syncthreads();
  sy_stamp(unit, 3);
  if (!s_last) return;
  __threadfence();
  double s[16];
  unsigned int need = 0xffffu;                            // diagonal pair: elements of fragments that were stored
  if (diag) {
    need = 0u;
#pragma unroll
    for (int q = 0; q < 16; ++q)
      if ((((tid >> 6) + 4 * q) >> 3) <= ((tid & 63) >> 3)) need |= 1u << q;
  }
  auto ldp = [&](const double* p, int q) { return ((need >> q) & 1u) ? __ldcg(p) : 0.0; };
  auto sum_slots = [&](int first, int last, int step) {   // slots first, first + step, ... < last, in order
#pragma unroll
    for (int q = 0; q < 16; ++q) s[q] = 0.0;
    int c = first;
    for (; c + 3 * step < last; c += 4 * step) {          // four slots in flight
      const double* p0 = base + (size_t)c * cstride + tid;
      const size_t ss = (size_t)step * cstride;
      double x0[16], x1[16], x2[16], x3[16];
#pragma unroll
      for (int q = 0; q < 16; ++q) x0[q] = ldp(p0 + 256 * q, q);
#pragma unroll
      for (int q = 0; q < 16; ++q) x1[q] = ldp(p0 + ss + 256 * q, q);
#pragma unroll
      for (int q = 0; q < 16; ++q) x2[q] = ldp(p0 + 2 * ss + 256 * q, q);
#pragma unroll
      for (int q = 0; q < 16; ++q) x3[q] = ldp(p0 + 3 * ss + 256 * q, q);
#pragma unroll
      for (int q = 0; q < 16; ++q) s[q] = (((s[q] + x0[q]) + x1[q]) + x2[q]) + x3[q];
    }
    for (; c < last; c += step) {
      const double* p0 = base + (size_t)c * cstride + tid;
#pragma unroll
      for (int q = 0; q < 16; ++q) s[q] += ldp(p0 + 256 * q, q);
    }
  };
  sum_slots(c_begin, c_end, 1);
  sy_stamp(unit, 4);
  if (ngroups > 1) {
    // ---- level 2: the group sum replaces the group's first partial; the last group sums the groups
    double* gout = base + (size_t)c_begin * cstride + tid;
#pragma unroll
    for (int q = 0; q < 16; ++q)
      if ((need >> q) & 1u) __stcg(gout + 256 * q, s[q]);
    __threadfence();
    __syncthreads();
    if (tid == 0) {
      cnt[1 + g] = 0u;
      s_last = (atomicAdd(cnt, 1u) == (unsigned int)(ngroups - 1));
    }
    __syncthreads();
    sy_stamp(unit, 5);
    if (!s_last) return;
    __threadfence();
    sum_slots(0, nchunks, gsz);
    sy_stamp(unit, 6);
    if (tid == 0) cnt[0] = 0u;
  } else if (tid == 0) {
    cnt[1 + g] = 0u;                                      // ready for the next launch
  }
#pragma unroll
  for (int q = 0; q < 16; ++q) {
    const int e = tid + 256 * q;
    emit(e >> 6, e & 63, s[q]);
  }
  sy_stamp(unit, 7);
}

static long long* g_syrk_dbg_host = nullptr;
static int g_syrk_dbg_units = 0;
int syrk_debug_read(long long* out, int cap) {
  if (!g_syrk_dbg_host) return 0;
  const int n = std::min(cap, g_syrk_dbg_units * SY_DBG_N);
  cudaDeviceSynchronize();
  cudaMemcpy(out, g_syrk_dbg_host, (size_t)n * sizeof(long long), cudaMemcpyDeviceToHost);
  return n;
}

// ---------------------------------------------------------------- W = C C^T with F_1, v carried; dx
// grid (strips, filters).  Every CTA factors W (redundantly -- the factorisation is latency, not
// throughput) and carries its strip of CS rows of F_1 plus the vector v through it: the strip
// leaves as the matching columns of Y = C^-1 F_1^T, v leaves as y = C^-1 v, and the strip's part of
// dx = Y^T y (src/orcvio.cpp:1820 `dx_leg = K * r_o`) is formed on the spot from the tiles.
constexpr int CS = 16;

__global__ void __launch_bounds__(CHOL_THREADS) k_chol_w_solve(UpdArgs a) {
  extern __shared__ double sm[];
  __shared__ __align__(16) CholShared cs;
  const int fi = blockIdx.y;
  const FilterWork fw = a.fw[fi];
  if (!fw.active) return;
  const int n = fw.D - ORCVIO_LEG, D = fw.D;
  const int d0 = blockIdx.x * CS;
  if (d0 >= D) return;
  const int nd = min(CS, D - d0);
  const int nx = nd + 1;
  const double* S = a.S + (size_t)fi * a.r_stride;
  double* T = a.T + (size_t)fi * a.t_stride;
  double* yv = a.yv + (size_t)fi * a.ldr;
  double* A = sm;
  const int Tm = (n + 7) >> 3;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  chol_init(A, cs, n, nx);
  __syncthreads();
  const int ldr = a.ldr, ldt0 = a.ldt;
  // triangle rows: W;  carried rows: row n + q = F_1[d0 + q][:] = FT[:][d0 + q];  last row: v = S[n][:]
  chol_load_rows(A, n, 0, n + nx, [&](int i, int j) -> const double* {
    if (i < n) return S + (size_t)i * ldr + j;
    const int q = i - n;
    return q < nd ? T + (size_t)j * ldt0 + d0 + q : S + (size_t)n * ldr + j;
  });
  chol_cp_async_wait();
  cta_cholesky(A, cs, nullptr, n, nx);
  const int ldt = a.ldt;
  const bool strip0 = (blockIdx.x == 0);
  chol_for_rows(A, n, nx, n, [&](int i, int k, double l) {
    const int q = i - n;
    if (q < nd) T[(size_t)k * ldt + d0 + q] = l;         // Y[k][d0 + q]
    else if (strip0) yv[k] = l;
  });
  // dx[d0 + q] = sum_k Y[k][d0 + q] y[k]: warp q, lanes over k, fixed-order shuffle tree
  if (warp < nd) {
    const int iy = n + nd, iq = n + warp;
    double s0 = 0.0, s1 = 0.0;
    int k = lane;
    for (; k + 32 < n; k += 64) {
      s0 += A[chol_at(iq, k, Tm)] * A[chol_at(iy, k, Tm)];
      s1 += A[chol_at(iq, k + 32, Tm)] * A[chol_at(iy, k + 32, Tm)];
    }
    if (k < n) s0 += A[chol_at(iq, k, Tm)] * A[chol_at(iy, k, Tm)];
    double sv = s0 + s1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sv += __shfl_xor_sync(0xffffffffu, sv, o);
    if (lane == 0) a.dx[(size_t)fi * a.lddx + d0 + warp] = sv;
  }
}

// ---------------------------------------------------------------- P+ = s^2 Y^T Y + F_2 F_2^T and the state increment
// 32 x 32 output tile per CTA; both strips of Y (n x 32) are staged in shared memory with one
// round trip, then the k loop runs without barriers.  One extra CTA per filter (blockIdx.y ==
// gridDim.y - 1) applies dx to the state (incrementState_IMUCam, src/orcvio.cpp:4468-4567).
constexpr int PT = 32;
constexpr int PI_LD = 36;                 // strip row stride in doubles (== 4 mod 16: conflict-free 64-bit fragment loads)
constexpr int PI_THREADS = 1024;          // 32 warps: 16 fragments (8 x 8) of the 32 x 32 tile x 2 halves of k

__global__ void __launch_bounds__(PI_THREADS) k_pinfo(UpdArgs a, const double* Ls_all, const int* filter_rows) {
  extern __shared__ double sm[];
  const int fi = blockIdx.z;
  const FilterWork fw = a.fw[fi];
  if (!fw.active) return;
  const int n = fw.D - ORCVIO_LEG, D = fw.D, L = ORCVIO_LEG;
  const int tid = threadIdx.x;
  if (blockIdx.y == gridDim.y - 1) {
    if (blockIdx.x != 0) return;
    double* dxs = sm;
    for (int i = tid; i < D; i += blockDim.x) dxs[i] = a.dx[(size_t)fi * a.lddx + i];
    __syncthreads();
    cta_increment_state(dxs, a.imu + (size_t)fi * IM_STRIDE, a.clones + (size_t)fi * a.clone_stride, fw.N, a.flags,
                        &a.dx[(size_t)fi * a.lddx + a.lddx - 1]);
    return;
  }
  if (filter_rows[fi] == 0) return;                     // no gated rows: posterior == prior, P untouched
  const int i0 = blockIdx.y * PT, j0 = blockIdx.x * PT;
  if (i0 >= D || j0 >= D) return;
  const double* Y = a.T + (size_t)fi * a.t_stride;
  double* P = a.P + (size_t)fi * a.p_stride;
  const int n4 = (n + 3) & ~3;                          // k padded to the MMA depth (zero rows)
  double* Ys_i = sm;                                    // [n4][PI_LD]
  double* Ys_j = sm + (size_t)n4 * PI_LD;
  // both strips with 16-byte cp.async: every load of the CTA is in flight at once (one L2 round trip)
  {
    const int ldt = a.ldt;
    const bool same = (i0 == j0);
    for (int e = tid; e < n4 * (PT / 2); e += PI_THREADS) {
      const int k = e / (PT / 2), c = 2 * (e - k * (PT / 2));
      double* di_ = Ys_i + (size_t)k * PI_LD + c;
      double* dj_ = Ys_j + (size_t)k * PI_LD + c;
      if (k < n && i0 + c < D) {                         // (columns past D of Y are never written)
        const unsigned int d = (unsigned int)__cvta_generic_to_shared(di_);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(Y + (size_t)k * ldt + i0 + c) : "memory");
      } else {
        *reinterpret_cast<double2*>(di_) = make_double2(0.0, 0.0);
      }
      if (same) continue;
      if (k < n && j0 + c < D) {
        const unsigned int d = (unsigned int)__cvta_generic_to_shared(dj_);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(Y + (size_t)k * ldt + j0 + c) : "memory");
      } else {
        *reinterpret_cast<double2*>(dj_) = make_double2(0.0, 0.0);
      }
    }
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
    if (same) Ys_j = Ys_i;
  }
  __syncthreads();
  // Y_i^T Y_j on the FP64 tensor cores: warp w owns fragment (w & 15) over half (w >> 4) of k, two accumulators
  // alternate over the k steps (a dependent DFMA / DMMA costs tens of cycles: the k loop is latency, not flops);
  // the upper-half warps hand their partial fragment over through shared memory, added in a fixed order
  const int warp = tid >> 5, lane = tid & 31;
  const int fr = lane >> 2, fk = lane & 3;
  const int fidx = warp & 15, half = warp >> 4;
  const int fi8 = (fidx >> 2) * 8, fj8 = (fidx & 3) * 8;
  const int ksteps = n4 >> 2, khalf = (ksteps + 1) >> 1;
  const int ks0 = half * khalf, ks1 = min(ksteps, ks0 + khalf);
  double2 c0 = make_double2(0.0, 0.0), c1 = make_double2(0.0, 0.0);
  {
    const double* pa = Ys_i + (size_t)fk * PI_LD + fi8 + fr;
    const double* pb = Ys_j + (size_t)fk * PI_LD + fj8 + fr;
    int ks = ks0;
    for (; ks + 1 < ks1; ks += 2) {
      const double a0 = pa[(size_t)(4 * ks) * PI_LD], b0 = pb[(size_t)(4 * ks) * PI_LD];
      const double a1 = pa[(size_t)(4 * ks + 4) * PI_LD], b1 = pb[(size_t)(4 * ks + 4) * PI_LD];
      dmma884(c0.x, c0.y, a0, b0);
      dmma884(c1.x, c1.y, a1, b1);
    }
    if (ks < ks1) dmma884(c0.x, c0.y, pa[(size_t)(4 * ks) * PI_LD], pb[(size_t)(4 * ks) * PI_LD]);
  }
  double2 acc = make_double2(c0.x + c1.x, c0.y + c1.y);
  double2* red = reinterpret_cast<double2*>(sm + (size_t)2 * n4 * PI_LD);   // [16 fragments][32 lanes]
  if (half == 1) red[fidx * 32 + lane] = acc;
  __syncthreads();
  if (half == 1) return;
  {
    const double2 r = red[fidx * 32 + lane];
    acc.x += r.x;
    acc.y += r.y;
  }
  // fragment element: row i = i0 + fi8 + fr, columns j0 + fj8 + 2 fk (+1)
  const double* Ls = Ls_all + (size_t)fi * L * L;
  const int i = i0 + fi8 + fr;
  for (int v = 0; v < 2; ++v) {
    const int j = j0 + fj8 + 2 * fk + v;
    if (i >= D || j >= D) continue;
    double s = a.sigma2 * (v == 0 ? acc.x : acc.y);
    if (i < L && j < L) {
      double t0 = 0.0, t1 = 0.0;
      for (int q = 0; q + 1 < L; q += 2) {
        t0 += Ls[i * L + q] * Ls[j * L + q];
        t1 += Ls[i * L + q + 1] * Ls[j * L + q + 1];
      }
      s += t0 + t1;
    }
    P[(size_t)i * a.ldp + j] = s;
  }
}

static void info_attrs() {
  static bool attr = false;
  if (attr) return;
  cudaFuncSetAttribute(k_aform, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024);
  // hybrid states (30 clones + 30 features: D = 232) need 221 KB of tiles: everything the SM has
  cudaFuncSetAttribute(k_chol_prior, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024);
  cudaFuncSetAttribute(k_chol_w_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024);
  cudaFuncSetAttribute(k_pinfo, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
  cudaFuncSetAttribute(k_imu_factor, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
  cudaFuncSetAttribute(k_syrk, cudaFuncAttributeMaxDynamicSharedMemorySize, SY_STAGES * SY_STAGE_DOUBLES * (int)sizeof(double));
  check_launch("info attributes");
  attr = true;
}

static void launch_syrk(const UpdArgs& u, const InfoBufs& ib, int B, const Tile* tiles, cudaStream_t s) {
  dim3 gs(std::max(ib.max_units, 1), B);
  static const int dbg = env_int("ORCVIO_SYRK_DBG", 0);
  if (dbg) {
    if (!g_syrk_dbg_host) {
      cudaMalloc(&g_syrk_dbg_host, (size_t)1024 * SY_DBG_N * sizeof(long long));
      cudaMemcpyToSymbol(g_syrk_dbg, &g_syrk_dbg_host, sizeof(g_syrk_dbg_host));
    }
    cudaMemsetAsync(g_syrk_dbg_host, 0, (size_t)1024 * SY_DBG_N * sizeof(long long), s);
    g_syrk_dbg_units = std::min(1024, std::max(ib.max_units, 1));
  }
  // the parallel slice reduction spins on the other chunks of a pair: only when every CTA of the grid is resident
  int n_sm = 0, dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
  const int spin = ((long long)gs.x * gs.y <= n_sm) ? 1 : 0;
  const size_t smem = (size_t)SY_STAGES * SY_STAGE_DOUBLES * sizeof(double);
  // (SY_GROUP goes in as an argument: folded in as a constant, the reductions specialise and k_syrk spills more)
  k_syrk<<<gs, SY_THREADS, smem, s>>>(u, ib.Amat, u.ldr, ib.part, ib.max_units, ib.cta_budget, SY_GROUP, tiles,
                                       ib.tile_rows, ib.filter_rows, ib.syrk_cnt, spin);
  check_launch("k_syrk");
}

static void launch_pinfo(const UpdArgs& u, const InfoBufs& ib, int nmax, int B, cudaStream_t s) {
  const int Dmax = ORCVIO_LEG + nmax;
  const int g = (Dmax + PT - 1) / PT;
  dim3 g5(g, g + 1, B);                                  // last row of CTAs: the state increment
  const int n4 = (nmax + 3) & ~3;
  k_pinfo<<<g5, PI_THREADS, ((size_t)2 * n4 * PI_LD + 16 * 32 * 2) * sizeof(double), s>>>(u, ib.Ls, ib.filter_rows);
  check_launch("k_pinfo");
}

// Object update, first half (removeLostObjects -> measurementUpdate_msckf with a dense block):
// prior factor, A = Hp L, W = s^2 I + A^T A, Cholesky with F_1 / v carried.  Leaves Y in u.T,
// y in u.yv, dx in u.dx and W_aug's corner r'^T r' untouched in u.S[n][n]:
//   gamma = r'^T (Hp P Hp^T + s^2 I)^-1 r' = (r'^T r' - y^T y) / s^2      (Woodbury).
void launch_info_dense_factor(const UpdArgs& u, const InfoBufs& ib, const double* Hp, int ldh, int rows, int n,
                              cudaStream_t s) {
  info_attrs();
  const int D = ORCVIO_LEG + n;
  const size_t sm_prior = (chol_smem_doubles(n, ORCVIO_LEG) + (size_t)n + 2) * sizeof(double);
  k_chol_prior<<<1, CHOL_THREADS, sm_prior, s>>>(u);
  check_launch("k_chol_prior");
  k_imu_factor<<<1, 256, ((size_t)n * ORCVIO_LEG + ORCVIO_LEG * (ORCVIO_LEG + 1)) * sizeof(double), s>>>(u, ib.Ls);
  check_launch("k_imu_factor");
  k_aform_dense<<<rows, 256, 0, s>>>(Hp, ldh, rows, n, u.T, u.ldt, ib.Amat, u.ldr);
  check_launch("k_aform_dense");
  launch_syrk(u, ib, 1, nullptr, s);
  const size_t sm_w = chol_smem_doubles(n, CS + 1) * sizeof(double);
  dim3 gw((D + CS - 1) / CS, 1);
  k_chol_w_solve<<<gw, CHOL_THREADS, sm_w, s>>>(u);
  check_launch("k_chol_w_solve");
}

// Object update, second half (after the gate passed): state increment, P+.
void launch_info_dense_apply(const UpdArgs& u, const InfoBufs& ib, int n, cudaStream_t s) {
  info_attrs();
  launch_pinfo(u, ib, n, 1, s);
}

// Prior factor on the second stream: it depends only on P, so it overlaps triangulation / Jacobians
// (and, in the end-to-end call, the host's work-list build).  `fork` was recorded on the main stream
// once P was in place; `join` is what the main stream waits for before k_aform.
void launch_info_prior(const UpdArgs& u, const InfoBufs& ib, int max_N, cudaStream_t s2, cudaEvent_t fork,
                       cudaEvent_t join, cudaEvent_t t0, cudaEvent_t t1, int max_E) {
  const int Dmax = ORCVIO_LEG + 6 * max_N + max_E;
  info_attrs();
  cudaStreamWaitEvent(s2, fork, 0);
  if (t0) cudaEventRecord(t0, s2);
  const int nmax = Dmax - ORCVIO_LEG;
  const size_t sm_prior = (chol_smem_doubles(nmax, ORCVIO_LEG) + (size_t)nmax + 2) * sizeof(double);
  k_chol_prior<<<u.n_filters, CHOL_THREADS, sm_prior, s2>>>(u);
  check_launch("k_chol_prior");
  if (t1) cudaEventRecord(t1, s2);
  cudaEventRecord(join, s2);
  // the IMU block's factor: needed by k_pinfo only, so it stays on the side stream behind the join point
  k_imu_factor<<<u.n_filters, 256, ((size_t)nmax * ORCVIO_LEG + ORCVIO_LEG * (ORCVIO_LEG + 1)) * sizeof(double), s2>>>(u, ib.Ls);
  check_launch("k_imu_factor");
  if (ib.ls_done) cudaEventRecord(ib.ls_done, s2);
}

void launch_info_update(const AformArgs& q, const UpdArgs& u, const InfoBufs& ib, int n_tiles, int max_tile_rows,
                        int max_w_blk, int max_N, cudaStream_t s, cudaStream_t s2, cudaEvent_t fork,
                        cudaEvent_t join, cudaEvent_t mid1, cudaEvent_t mid2, int* launches, bool prior_in_flight,
                        cudaEvent_t mid_syrk, cudaEvent_t prior_t0, cudaEvent_t prior_t1, int max_E,
                        const HybArgs* hyb, int max_dense) {
  const int nmax = 6 * max_N + max_E, Dmax = ORCVIO_LEG + nmax;
  const int B = u.n_filters;
  info_attrs();
  if (!prior_in_flight) launch_info_prior(u, ib, max_N, s2, fork, join, prior_t0, prior_t1, max_E);
  cudaStreamWaitEvent(s, join, 0);
  const int lda = u.ldr;
  if (n_tiles > 0) {
    const int rows8 = (std::max(max_tile_rows, 1) + 7) & ~7;
    const int wp = ((6 * max_w_blk + 3) & ~3) + 4;        // >= aform_stride(W) of every tile
    k_aform<<<n_tiles, AF_THREADS, (size_t)rows8 * wp * sizeof(double), s>>>(q, u.T, u.t_stride, u.ldt, ib.Amat, lda,
                                                                           ib.tile_rows);
    check_launch("k_aform");
  }
  if (hyb && max_dense > 0) {      // hybrid mode: the dense rows of the EKF-SLAM features, behind the tiles' rows
    launch_hybrid_aform(*hyb, u.T, u.t_stride, u.ldt, ib.Amat, lda, u.fw, max_dense, s);
    if (launches) *launches += 1;
  }
  if (mid1) cudaEventRecord(mid1, s);
  launch_syrk(u, ib, B, q.tiles, s);
  if (mid_syrk) cudaEventRecord(mid_syrk, s);
  const size_t sm_w = chol_smem_doubles(nmax, CS + 1) * sizeof(double);
  dim3 gw((Dmax + CS - 1) / CS, B);
  // k_chol_w_solve overwrites F_1 (u.T) with Y in place, and k_imu_factor on the side stream still reads the IMU
  // columns of F_1: it must be done first (it is, by tens of microseconds, unless other work delays the side stream)
  if (ib.ls_done) cudaStreamWaitEvent(s, ib.ls_done, 0);
  k_chol_w_solve<<<gw, CHOL_THREADS, sm_w, s>>>(u);
  check_launch("k_chol_w_solve");
  if (mid2) cudaEventRecord(mid2, s);
  launch_pinfo(u, ib, nmax, B, s);
  if (launches) *launches += 3 + (prior_in_flight ? 0 : 2) + (n_tiles > 0 ? 1 : 0);
}

}  // namespace ob

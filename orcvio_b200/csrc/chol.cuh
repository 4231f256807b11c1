// One-CTA blocked Cholesky with carried rows: a left-looking factorisation organised around the pivot chain,
// with FP64 tensor-core (mma.m8n8k4) updates fed straight from the tiled factor.
//
// Used for both factorisations of the whitened-form update (info_kernel.cu): the prior
// P = F F^T (k_chol_prior) and W = C C^T with strips of F_1 / v carried through as extra rows
// (k_chol_w_solve).  The reference does the equivalent work with Eigen's ldlt()
// (src/orcvio.cpp:1690 `S.ldlt().solve(H P)`); on the GPU a 200 x 200 factorisation is a latency
// chain of m dependent pivots, so the routine is organised so that NOTHING but that chain is on the
// critical path:
//
//   * the "tall" matrix [A; X] (m x m lower triangle + nx carried rows) lives in shared memory
//     as 8 x 8 row-major tiles (512 contiguous bytes each).  A tile read as 32 x 16-byte chunks (chunk
//     l = row l/4, columns 2(l%4), 2(l%4)+1) is at once a conflict-free access, the accumulator layout
//     of mma.m8n8k4 and -- with the k index of the MMA permuted to (even columns | odd columns), the same
//     permutation on both operands -- its A / B operand: updates need no staging buffer at all;
//   * warp 0 is the CHAIN warp.  In step q it factors the diagonal tile (q, q) (8-pivot L D L^T elimination, one
//     row per lane, every 8-lane segment redundantly) and publishes the block for the other warps.  Lanes 8..15
//     then solve the rows of tile (q+1, q) in registers: the block's entries are the ones the elimination's
//     shuffles already brought in, nothing is read back from shared memory.  The solved rows reach every lane by
//     shuffles as the operand of the MMA pair that applies the panel to tile (q+1, q+1), and the updated tile is
//     shuffled into row-per-lane form for step q+1 without a store and reload.  It waits for exactly one tile per
//     step, with a whole factorisation of slack;
//   * warp 4 is the FRONTIER warp (same scheduler as the chain warp, which is otherwise kept free of MMA
//     work): in step q it solves tile (q+2, q) and brings tile (q+2, q+1) up to date with panel q -- the tile the
//     chain warp needs one step later -- without waiting for anybody's bulk work;
//   * twelve BULK warps (the warps of the other three schedulers) solve the remaining rows of tile column q
//     (thread per row), bring the rest of tile column q+1 up to date with panel q (one MMA pair per tile) and
//     give tile column q+2 its bulk update with ALL panels 0..q at once (left-looking: the accumulator stays
//     in registers over the whole k loop, one operand chunk per tile and k instead of a load + store of the
//     accumulator per 8 columns).  The hand-offs between the three roles are step counters in shared memory;
//   * the factor is left in the tiles; callers copy what they need out with chol_for_rows().
//
// Measured on B200 (scripts/chol_probe.py, api.latency_probe1): a dependent mma.m8n8k4.f64 costs 26 cycles (16 at
// the issue limit), a 16-byte shared load 48 cycles and FOUR passes of the 128 B / cycle shared-memory pipe even
// when every lane reads the same address -- the worker phases are bound by that pipe (the broadcast loads of the
// diagonal block in the row solve, one operand chunk per MMA pair in the bulk update), not by the tensor pipe.
// Tried and rejected: a 16-row factor in the chain warp (the tile below has to be final a whole factorisation
// earlier: the chain then waits for the workers), FMA instead of MMA for the single-tile updates of the chain and
// frontier warps (more shared-memory passes, slower), 12 accumulators per tile (register spills), an XOR swizzle
// of the tile rows (conflict-free thread-per-row access, but the row solve is bound by the broadcast loads:
// no gain), dropping the fences between the roles (wrong results: they are needed).
//
// `tol != nullptr`: pivots <= tol[k] are exact zeros (semidefinite prior: the IMU pose duplicates
// the newest clone after augmentation and rows 15..21 are exactly zero) -> zero column.
#pragma once
#include "kernels.h"

namespace ob {

constexpr int CHB = 8;
constexpr int CHOL_THREADS = 512;
constexpr int CHOL_BULK_WARPS = 12;                               // warps with (warp & 3) != 0
constexpr int CHOL_BULK_THREADS = CHOL_BULK_WARPS * 32;
constexpr int CHOL_PUB_THREADS = CHOL_BULK_THREADS + 64;          // + chain warp + frontier warp
constexpr int CHOL_MAXM = ORCVIO_LEG + 6 * ORCVIO_MAX_OBS;        // 214
constexpr int CHOL_MAXR = 244;   // rows incl. carried rows

// tile index of (ti, tj), tj <= min(ti, Tm-1); Tm = tile columns = ceil(m / 8)
__device__ __host__ __forceinline__ int chol_tile(int ti, int tj, int Tm) {
  return ti < Tm ? (ti * (ti + 1) >> 1) + tj : (Tm * (Tm + 1) >> 1) + (ti - Tm) * Tm + tj;
}
// element (i, j) of the tall matrix, j <= min(i, m-1)
__device__ __host__ __forceinline__ int chol_at(int i, int j, int Tm) {
  return chol_tile(i >> 3, j >> 3, Tm) * 64 + (i & 7) * 8 + (j & 7);
}
__device__ __host__ __forceinline__ size_t chol_smem_doubles(int m, int nx) {
  const int Tm = (m + 7) >> 3, Tr = (m + nx + 7) >> 3;
  return (size_t)chol_tile(Tr, 0, Tm) * 64;
}

struct CholShared {
  double dblk[2][CHB][CHB];         // factored diagonal block (lower), double-buffered by step parity
  double dinv[2][CHB];              // 1 / diagonal (0 for skipped pivots)
  // step counters (value s+1 = "done for step s"); writer -> reader
  volatile int flag_c2;             // chain -> all: tile (s+1, s) is solved
  volatile int flag_w2;             // frontier -> chain: tile (s+2, s+1) carries every panel <= s
  volatile int flag_w3;             // bulk 0 -> chain: tile (s+2, s+2) carries every panel <= s
  volatile int flag_f1;             // frontier -> bulk: tile (s+2, s) is solved
  volatile int flag_b2;             // bulk 0 -> frontier: tile (s+3, s+1) carries every panel <= s
  volatile int flag_b3;             // bulk 1 -> frontier: tile (s+3, s+2) carries every panel <= s
};

// named barriers: 1 = bulk team; 2 / 3 = "diagonal block of step q published" (chain warp arrives, frontier and
// bulk warps wait), alternating with the parity of q (the chain warp is never two steps ahead of the others)
__device__ __forceinline__ void chol_team_barrier() {
  asm volatile("bar.sync 1, %0;" ::"n"(CHOL_BULK_THREADS) : "memory");
}
__device__ __forceinline__ void chol_pub_arrive(int parity) {
  if (parity) asm volatile("bar.arrive 3, %0;" ::"n"(CHOL_PUB_THREADS) : "memory");
  else asm volatile("bar.arrive 2, %0;" ::"n"(CHOL_PUB_THREADS) : "memory");
}
__device__ __forceinline__ void chol_pub_wait(int parity) {
  if (parity) asm volatile("bar.sync 3, %0;" ::"n"(CHOL_PUB_THREADS) : "memory");
  else asm volatile("bar.sync 2, %0;" ::"n"(CHOL_PUB_THREADS) : "memory");
}
__device__ __forceinline__ void chol_wait_flag(volatile int* f, int v) {
  while (*f < v) {}
  __threadfence_block();
}
// whole warp: everything written by the warp so far is visible before the counter moves
__device__ __forceinline__ void chol_set_flag(volatile int* f, int v) {
  __threadfence_block();
  __syncwarp();
  if ((threadIdx.x & 31) == 0) *f = v;
}
// x <- x L_d^-T for one row held in registers (update form: full ILP across the remaining columns); dl = strictly
// lower part of the factored diagonal block, di = 1 / its diagonal (0 for skipped pivots).  The chain warp and the
// shared-memory row solve below both go through this, so they round alike.
__device__ __forceinline__ void chol_solve_regs(double (&x)[CHB], const double (&dl)[CHB][CHB], const double (&di)[CHB],
                                                int nb) {
#pragma unroll
  for (int c = 0; c < CHB; ++c) {
    if (c >= nb) x[c] = 0.0;
    x[c] *= di[c];
#pragma unroll
    for (int s = c + 1; s < CHB; ++s) x[s] -= x[c] * dl[s][c];
  }
}

// one row of a tile column against the published diagonal block
__device__ __forceinline__ void chol_solve_row(double* __restrict__ xt, const double (*dblk)[CHB], const double* dinv,
                                               int nb) {
  double dl[CHB][CHB], di[CHB];
#pragma unroll
  for (int c = 0; c < CHB; c += 2) {
    const double2 t = *reinterpret_cast<const double2*>(&dinv[c]);
    di[c] = t.x;
    di[c + 1] = t.y;
  }
#pragma unroll
  for (int c = 1; c < CHB; ++c)
#pragma unroll
    for (int s = 0; s < c; s += 2) {
      const double2 t = *reinterpret_cast<const double2*>(&dblk[c][s]);
      dl[c][s] = t.x;
      if (s + 1 < c) dl[c][s + 1] = t.y;
    }
  double x[CHB];
#pragma unroll
  for (int c = 0; c < CHB; c += 2) {
    const double2 t = *reinterpret_cast<const double2*>(xt + c);
    x[c] = t.x;
    x[c + 1] = t.y;
  }
  chol_solve_regs(x, dl, di, nb);
#pragma unroll
  for (int c = 0; c < CHB; c += 2) *reinterpret_cast<double2*>(xt + c) = make_double2(x[c], x[c + 1]);
}

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// 1/x for a normal positive pivot: hardware seed (2^-23) + two Newton steps, no special-case branch.
__device__ __forceinline__ double chol_rcp(double x) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  double e = fma(-x, y, 1.0);
  y = fma(y, e, y);
  e = fma(-x, y, 1.0);
  return fma(y, e, y);
}

// Zero the tiles and the step flags; call before scattering the matrix into `A`.
__device__ __forceinline__ void chol_init(double* __restrict__ A, CholShared& cs, int m, int nx) {
  const int nd2 = (int)(chol_smem_doubles(m, nx) >> 1);
  double2* A2 = reinterpret_cast<double2*>(A);
  for (int e = threadIdx.x; e < nd2; e += blockDim.x) A2[e] = make_double2(0.0, 0.0);
  if (threadIdx.x == 0) {
    cs.flag_c2 = 0; cs.flag_w2 = 0; cs.flag_w3 = 0; cs.flag_f1 = 0; cs.flag_b2 = 0; cs.flag_b3 = 0;
  }
}

// 1/sqrt(x) for a normal positive x: hardware seed (2^-22) + two Newton steps, branch-free.
__device__ __forceinline__ double chol_rsqrt(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double xh = 0.5 * x;
  double e = fma(-xh * y, y, 0.5);
  y = fma(y, e, y);
  e = fma(-xh * y, y, 0.5);
  return fma(y, e, y);
}

__device__ __forceinline__ void chol_cp_async8(double* smem_dst, const double* gsrc) {
  const unsigned int d = (unsigned int)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void chol_cp_async_wait() {
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

// Scatter rows [row_begin, row_end) of the tall matrix into the tiles: element (i, j) comes from the global
// address addr(i, j), j < ncols(i) (ncols(i) = i + 1 for triangle rows, m for carried rows).  Every element is
// one 8-byte cp.async straight into its tile slot, so ALL loads of the CTA are in flight together (one
// memory round trip for the whole matrix instead of one per row batch).  The tiles must have been zeroed
// (chol_init) and made visible (__syncthreads) before; the caller finishes with chol_cp_async_wait() +
// __syncthreads().
template <class Addr>
__device__ __forceinline__ void chol_load_rows(double* __restrict__ A, int m, int row_begin, int row_end, Addr addr) {
  const int Tm = (m + 7) >> 3;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int i = row_begin + warp; i < row_end; i += nw) {
    const int nc = min(i + 1, m);
    const int tbase = chol_tile(i >> 3, 0, Tm) * 64 + (i & 7) * 8;
    for (int j = lane; j < nc; j += 32) chol_cp_async8(A + tbase + (j >> 3) * 64 + (j & 7), addr(i, j));
  }
}

// A: tiled (chol_at) tall matrix: m x m lower triangle followed by nx carried rows.
// On return tile storage holds L (rows < m) and X C^-T (rows >= m).
// PROF: per step q, prof[q][0..3] = chain warp (step start, block published, tile (q+1,q) in hand, tile (q+1,q+1)
// updated), prof[q][4..7] = first bulk warp (block seen, rows solved, column q+1 done, bulk of column q+2 done).
template <bool PROF = false>
__device__ void cta_cholesky(double* __restrict__ A, CholShared& cs, const double* __restrict__ tol, int m, int nx,
                             long long* prof = nullptr) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int mrows = m + nx;
  const int Tm = (m + 7) >> 3, Tr = (mrows + 7) >> 3;
  double2* const A2 = reinterpret_cast<double2*>(A);
  __syncthreads();
  if (warp == 0) {
    // ------------------------------------------------ chain warp
    const int a = lane & 7;                                    // row of the diagonal tile (four redundant copies)
    const bool solver = (lane >> 3) == 1;                      // lanes 8..15: row a of tile (q+1, q)
    double d[CHB];                                             // row a of the diagonal tile; from step 1 on, the
#pragma unroll                                                 // previous step leaves it here (it is never stored)
    for (int b = 0; b < CHB; b += 2) {
      const double2 t = *reinterpret_cast<const double2*>(A + a * 8 + b);
      d[b] = t.x;
      d[b + 1] = t.y;
    }
    for (int q = 0; q < Tm; ++q) {
      const int k0 = q * CHB;
      const int nb = min(CHB, m - k0);
      const bool below = (q + 1 < Tr);
      if (PROF && lane == 0) prof[q * 8 + 0] = clock64();
      double* dt = A + (size_t)chol_tile(q, q, Tm) * 64 + a * 8;
      // columns >= nb do not exist (last, partial block); rows nb..7 of the diagonal tile are then carried rows and
      // are eliminated along with the pivots
#pragma unroll
      for (int b = 0; b < CHB; ++b)
        if (b >= nb) d[b] = 0.0;
      // Unscaled (L D L^T) elimination, branch-free.  The dependent chain per pivot is
      //   shuffle -> reciprocal seed -> 2 FMA (one Newton step) -> multiply -> FMA (second Newton step folded
      //   into w = u / pivot) -> FMA into the next pivot;
      // thresholds are preloaded, rejected pivots are handled by selects.  The 8 rsqrt that turn the
      // result into L = U D^-1/2 run afterwards, in parallel.
      // The shuffles of pivot c bring in column c of rows b > c in its final unscaled form: kept in dl, they give the
      // strictly lower part of the factored block (the same products as the row scaling below) with no further traffic.
      double thr[CHB], ivs[CHB], dl[CHB][CHB];
#pragma unroll
      for (int c = 0; c < CHB; ++c) thr[c] = (tol != nullptr && c < nb) ? tol[k0 + c] : 0.0;
#pragma unroll
      for (int c = 0; c < CHB; ++c) {
        const double pv = __shfl_sync(0xffffffffu, d[c], c, 8);
        const bool ok = pv > thr[c];                            // false for c >= nb (pv == 0)
        const double u = d[c];
        double y0;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y0) : "d"(pv));
        const double e = fma(-pv, y0, 1.0);
        const double y1 = fma(y0, e, y0);                     // 1/pv (1 - e^2)
        const double e2 = e * e;
        const double t = u * y1;
        double w = fma(t, e2, t);                             // u / pv to working precision
        w = ok ? w : 0.0;
        ivs[c] = ok ? pv : 0.0;
#pragma unroll
        for (int b = c + 1; b < CHB; ++b) {
          const double ub = __shfl_sync(0xffffffffu, u, b, 8);
          dl[b][c] = ub;
          d[b] = fma(-w, ub, d[b]);                           // meaningful for rows below row b
        }
      }
#pragma unroll
      for (int c = 0; c < CHB; ++c) {
        const double rs = chol_rsqrt(ivs[c] > 0.0 ? ivs[c] : 1.0);
        ivs[c] = (ivs[c] > 0.0) ? rs : 0.0;
        d[c] *= ivs[c];
      }
      // the block as published in dblk: rows >= nb are zero
#pragma unroll
      for (int c = 0; c < CHB; ++c)
#pragma unroll
        for (int s = c + 1; s < CHB; ++s) dl[s][c] = (s < nb) ? dl[s][c] * ivs[c] : 0.0;
      __syncwarp();   // lanes 8..31 hold redundant copies of the rows: their reads of tile (0, 0) are done before it is rewritten
      if (lane < CHB) {
        const bool tri = (a < nb);                             // triangle row: entries right of the diagonal are zeros
#pragma unroll
        for (int b = 0; b < CHB; b += 2) {
          const double2 t = make_double2((!tri || b <= a) ? d[b] : 0.0, (!tri || b + 1 <= a) ? d[b + 1] : 0.0);
          *reinterpret_cast<double2*>(dt + b) = t;
          *reinterpret_cast<double2*>(&cs.dblk[q & 1][a][b]) = tri ? t : make_double2(0.0, 0.0);
        }
        if (lane == 0) {
#pragma unroll
          for (int b = 0; b < CHB; ++b) cs.dinv[q & 1][b] = ivs[b];
        }
      }
      __syncwarp();
      __threadfence_block();
      chol_pub_arrive(q & 1);                                  // block q is final
      if (PROF && lane == 0) prof[q * 8 + 1] = clock64();
      if (below) {
        // tile (q+1, q): carries panels 0..q-1 once the frontier warp has finished its step q-1
        if (q > 0) chol_wait_flag(&cs.flag_w2, q);
        if (PROF && lane == 0) prof[q * 8 + 2] = clock64();
        double* xt = A + (size_t)chol_tile(q + 1, q, Tm) * 64 + a * 8;
        double x[CHB];
#pragma unroll
        for (int c = 0; c < CHB; c += 2) {
          const double2 t = solver ? *reinterpret_cast<const double2*>(xt + c) : make_double2(0.0, 0.0);
          x[c] = t.x;
          x[c + 1] = t.y;
        }
        if (solver && CHB * (q + 1) + a < mrows) {
          chol_solve_regs(x, dl, ivs, nb);                     // ivs = the published dinv
#pragma unroll
          for (int c = 0; c < CHB; c += 2) *reinterpret_cast<double2*>(xt + c) = make_double2(x[c], x[c + 1]);
        }
        chol_set_flag(&cs.flag_c2, q + 1);
        if (q + 1 < Tm) {
          // tile (q+1, q+1) -= L(q+1, q) L(q+1, q)^T on top of its bulk update (panels < q, bulk step q-1).  The
          // operand chunk of this lane (row lane / 4, columns 2 (lane % 4) + 0, 1) comes from solver lane 8 + lane / 4.
          double2 l = make_double2(0.0, 0.0);
#pragma unroll
          for (int j = 0; j < CHB / 2; ++j) {
            const double lx = __shfl_sync(0xffffffffu, x[2 * j], CHB + (lane >> 2));
            const double ly = __shfl_sync(0xffffffffu, x[2 * j + 1], CHB + (lane >> 2));
            if ((lane & 3) == j) l = make_double2(lx, ly);
          }
          if (q > 0) chol_wait_flag(&cs.flag_w3, q);
          double2 cv = A2[(size_t)chol_tile(q + 1, q + 1, Tm) * 32 + lane];
          dmma884(cv.x, cv.y, -l.x, l.x);
          dmma884(cv.x, cv.y, -l.y, l.y);
          // row a of the updated tile for step q+1: its four chunks are in lanes 4a .. 4a+3
#pragma unroll
          for (int j = 0; j < CHB / 2; ++j) {
            d[2 * j] = __shfl_sync(0xffffffffu, cv.x, 4 * a + j);
            d[2 * j + 1] = __shfl_sync(0xffffffffu, cv.y, 4 * a + j);
          }
        }
      }
      if (PROF && lane == 0) prof[q * 8 + 3] = clock64();
    }
  } else if (warp == 4) {
    // ------------------------------------------------ frontier warp: tile row q+2
    for (int q = 0; q < Tm; ++q) {
      const int nb = min(CHB, m - q * CHB);
      chol_pub_wait(q & 1);
      if (q + 2 >= Tr) continue;
      if (q > 0) chol_wait_flag(&cs.flag_b2, q);               // tile (q+2, q) carries panels 0..q-1
      if (lane < CHB && CHB * (q + 2) + lane < mrows)
        chol_solve_row(A + (size_t)chol_tile(q + 2, q, Tm) * 64 + lane * 8, cs.dblk[q & 1], cs.dinv[q & 1], nb);
      chol_set_flag(&cs.flag_f1, q + 1);
      if (q + 1 < Tm) {
        if (q > 0) chol_wait_flag(&cs.flag_b3, q);             // tile (q+2, q+1) carries panels 0..q-1
        chol_wait_flag(&cs.flag_c2, q + 1);                    // L(q+1, q)
        const double2 bq = A2[(size_t)chol_tile(q + 1, q, Tm) * 32 + lane];
        const double2 av = A2[(size_t)chol_tile(q + 2, q, Tm) * 32 + lane];
        double2* cp = A2 + (size_t)chol_tile(q + 2, q + 1, Tm) * 32 + lane;
        double2 cv = *cp;
        dmma884(cv.x, cv.y, -av.x, bq.x);
        dmma884(cv.x, cv.y, -av.y, bq.y);
        *cp = cv;
        chol_set_flag(&cs.flag_w2, q + 1);
      }
    }
  } else if ((warp & 3) != 0) {
    // ------------------------------------------------ bulk warps
    const int w = (warp >> 2) * 3 + (warp & 3) - 1;             // 0..11
    const int wtid = w * 32 + lane;
    for (int q = 0; q < Tm; ++q) {
      const int nb = min(CHB, m - q * CHB);
      chol_pub_wait(q & 1);
      if (PROF && wtid == 0) prof[q * 8 + 4] = clock64();
      // ---- rows from tile row q+3 on: thread per row
      const int i = CHB * (q + 3) + wtid;
      if (i < mrows)
        chol_solve_row(A + (size_t)chol_tile(i >> 3, q, Tm) * 64 + (i & 7) * 8, cs.dblk[q & 1], cs.dinv[q & 1], nb);
      __threadfence_block();
      chol_team_barrier();
      if (PROF && wtid == 0) prof[q * 8 + 5] = clock64();
      // ---- tile column q+1: the last missing panel (q); tile (q+3, q+1) first -- the frontier warp waits for it
      if (q + 1 < Tm) {
        chol_wait_flag(&cs.flag_c2, q + 1);                    // L(q+1, q)
        const double2 bq = A2[(size_t)chol_tile(q + 1, q, Tm) * 32 + lane];
        for (int ti = q + 3 + w; ti < Tr; ti += CHOL_BULK_WARPS) {
          const double2 av = A2[(size_t)chol_tile(ti, q, Tm) * 32 + lane];
          double2* cp = A2 + (size_t)chol_tile(ti, q + 1, Tm) * 32 + lane;
          double2 cv = *cp;
          dmma884(cv.x, cv.y, -av.x, bq.x);
          dmma884(cv.x, cv.y, -av.y, bq.y);
          *cp = cv;
          if (w == 0 && ti == q + 3) chol_set_flag(&cs.flag_b2, q + 1);
        }
        if (w == 0 && q + 3 >= Tr) chol_set_flag(&cs.flag_b2, q + 1);
      }
      if (PROF && wtid == 0) prof[q * 8 + 6] = clock64();
      // ---- tile column q+2: bulk update with panels 0..q (left-looking; up to two tiles per pass and warp, two
      // accumulators per tile so that the dependent MMA chain is a quarter of the k loop).  Warp 0 takes only tile
      // (q+2, q+2), which the chain warp waits for, and warp 1 only tile (q+3, q+2), which the frontier warp waits
      // for; the other tiles go to warps 2..11.
      if (q + 2 < Tm) {
        const int tc = q + 2;
        constexpr int NP = CHOL_BULK_WARPS - 2;
        chol_wait_flag(&cs.flag_f1, q + 1);                    // L(q+2, q): the B operand of the last k step
        const double2* pb = A2 + (size_t)chol_tile(tc, 0, Tm) * 32 + lane;
        for (int t1 = tc + w; t1 < Tr; t1 += (w < 2 ? Tr : 2 * NP)) {
          const int t2 = w < 2 ? Tr : t1 + NP;
          double2* cp1 = A2 + (size_t)chol_tile(t1, tc, Tm) * 32 + lane;
          const double2* pa1 = A2 + (size_t)chol_tile(t1, 0, Tm) * 32 + lane;
          double2 c1 = *cp1, e1 = make_double2(0.0, 0.0);
          if (t2 < Tr) {
            double2* cp2 = A2 + (size_t)chol_tile(t2, tc, Tm) * 32 + lane;
            const double2* pa2 = A2 + (size_t)chol_tile(t2, 0, Tm) * 32 + lane;
            double2 c2 = *cp2, e2 = make_double2(0.0, 0.0);
            int k = 0;
            for (; k + 1 <= q; k += 2) {
              const double2 b0 = pb[k * 32], b1 = pb[k * 32 + 32];
              const double2 x0 = pa1[k * 32], x1 = pa1[k * 32 + 32];
              const double2 y0 = pa2[k * 32], y1 = pa2[k * 32 + 32];
              dmma884(c1.x, c1.y, -x0.x, b0.x);
              dmma884(e1.x, e1.y, -x1.x, b1.x);
              dmma884(c2.x, c2.y, -y0.x, b0.x);
              dmma884(e2.x, e2.y, -y1.x, b1.x);
              dmma884(c1.x, c1.y, -x0.y, b0.y);
              dmma884(e1.x, e1.y, -x1.y, b1.y);
              dmma884(c2.x, c2.y, -y0.y, b0.y);
              dmma884(e2.x, e2.y, -y1.y, b1.y);
            }
            if (k <= q) {
              const double2 b0 = pb[k * 32];
              const double2 x0 = pa1[k * 32];
              const double2 y0 = pa2[k * 32];
              dmma884(c1.x, c1.y, -x0.x, b0.x);
              dmma884(c2.x, c2.y, -y0.x, b0.x);
              dmma884(c1.x, c1.y, -x0.y, b0.y);
              dmma884(c2.x, c2.y, -y0.y, b0.y);
            }
            c2.x += e2.x; c2.y += e2.y;
            *cp2 = c2;
          } else {
            int k = 0;
            for (; k + 1 <= q; k += 2) {
              const double2 b0 = pb[k * 32], b1 = pb[k * 32 + 32];
              const double2 x0 = pa1[k * 32], x1 = pa1[k * 32 + 32];
              dmma884(c1.x, c1.y, -x0.x, b0.x);
              dmma884(e1.x, e1.y, -x1.x, b1.x);
              dmma884(c1.x, c1.y, -x0.y, b0.y);
              dmma884(e1.x, e1.y, -x1.y, b1.y);
            }
            if (k <= q) {
              const double2 b0 = pb[k * 32];
              const double2 x0 = pa1[k * 32];
              dmma884(c1.x, c1.y, -x0.x, b0.x);
              dmma884(c1.x, c1.y, -x0.y, b0.y);
            }
          }
          c1.x += e1.x; c1.y += e1.y;
          *cp1 = c1;
          if (t1 == tc) chol_set_flag(&cs.flag_w3, q + 1);          // w == 0: the next diagonal tile
          if (t1 == tc + 1) chol_set_flag(&cs.flag_b3, q + 1);      // w == 1: the frontier warp's next tile
        }
        if (w == 1 && tc + 1 >= Tr) chol_set_flag(&cs.flag_b3, q + 1);
      }
      if (PROF && wtid == 0) prof[q * 8 + 7] = clock64();
      __threadfence_block();
      chol_team_barrier();
    }
  }
  __syncthreads();
}

// Calls f(i, k, value) for every stored entry with row_begin <= i < m + nx, k <= min(i, m-1).
// Thread mapping: a warp covers 8 rows x 4 columns per step (32-byte global segments when the
// caller's output is contiguous in i, mild bank conflicts on the tile reads).
template <class F>
__device__ __forceinline__ void chol_for_rows(const double* __restrict__ A, int m, int nx, int row_begin, F f) {
  const int Tm = (m + 7) >> 3;
  const int mrows = m + nx;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const int r = lane >> 2, cq = lane & 3;                    // row in tile, column quarter (2 columns)
  const int t_begin = row_begin >> 3, Tr = (mrows + 7) >> 3;
  // flat loop over (row block, tile column)
  int t = warp;
  for (int ti = t_begin; ti < Tr; ++ti) {
    const int ncol = min(ti + 1, Tm);
    for (; t < ncol; t += nw) {
      const double* tp = A + (size_t)chol_tile(ti, t, Tm) * 64 + r * 8 + cq * 2;
      const double2 v = *reinterpret_cast<const double2*>(tp);
      const int i = ti * 8 + r, k = t * 8 + cq * 2;
      if (i >= row_begin && i < mrows) {
        if (k <= min(i, m - 1)) f(i, k, v.x);
        if (k + 1 <= min(i, m - 1)) f(i, k + 1, v.y);
      }
    }
    t -= ncol;
  }
}

}  // namespace ob

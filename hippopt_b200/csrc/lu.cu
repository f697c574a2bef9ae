// lu.cu -- batched dense LU with partial pivoting for the stage blocks of the KKT sweep (SURVEY.md 8(f) f2).
//
// What it replaces: the sparse symmetric indefinite factorisation IPOPT calls once per iteration (MUMPS
// [ext], reached from /root/reference/src/hippopt/base/opti_solver.py:479).  hippopt_b200/kkt.py orders the
// Newton system by stage, which leaves one dense (n_k + m_E,k)-square block (337 for the kinodynamic OCP)
// per knot and instance; this file factors and solves those blocks, one CTA per matrix.
//
// The blocks are too large for shared memory (908 KB) and too small for one-matrix-per-launch BLAS
// (cuSOLVER through torch.linalg: ~1 TFLOP/s on 256 blocks of 337^2 on B200).  Here a CTA
//   * factors the current 16-column panel with its rows held in REGISTERS (thread t owns rows t, t+256,
//     t+512): two barriers per column (pivot search, pivot-row exchange);
//   * applies the panel's 16 interchanges to a trailing column as ONE gather (the composed permutation
//     touches <= 32 rows), then U12 = L11^{-1} A12 in registers;
//   * updates the trailing matrix A22 -= L21 U12 on the fp64 tensor cores (mma.sync m8n8k4), L21 and U12
//     from shared memory, the A22 fragments read and written in place in global memory.
// The substitution (lu_solve_staged_kernel) stages half panels of the factor in shared memory with
// cp.async beside the triangular solve and updates the other rows with the same MMAs.
//
// Storage: column-major n x n, leading dimension n (a symmetric matrix can be passed as is).
// Pivoting: rows are interchanged inside the panel and in the trailing columns, NOT in the columns to
// the left (LINPACK-style across panels, LAPACK-style inside one), and lu_solve applies the interchanges
// panel by panel in the same order; piv[j] is the row (>= j) exchanged with row j.
#include <cstdint>

#include "hb_math.cuh"  // dmma_m8n8k4

namespace hb {

constexpr int LU_NB = 16;
// B200, 148 blocks of 337^2 (one wave): 256 threads 0.98 ms, 512 threads (128 registers, spills) 1.22 ms
constexpr int LU_THREADS = 256;

__host__ __device__ inline int lu_ldp(int n) { return (n + 3) & ~3; }
// dynamic shared memory of the factor kernel: panel + U strip (+ slack: the last vector loads of a tile may
// run past the strip; what they read is never stored)
__host__ __device__ inline size_t lu_factor_smem(int n) { return ((size_t)2 * LU_NB * lu_ldp(n) + 256) * sizeof(double); }

// RPT = panel rows per thread: n <= RPT * LU_THREADS
// MB = CTAs per SM the register allocation is tuned for.  Measured on B200 (blocks of 337^2): 148 blocks
// 0.93 ms at MB = 1 (232 registers) vs 1.06 ms at MB = 2 (128 registers, 416 B of spills); 296 blocks 1.85 ms
// vs 1.53 ms -- the host picks MB = 2 when the batch exceeds one CTA per SM.
template <int RPT, int MB>
__global__ void __launch_bounds__(LU_THREADS, MB) lu_factor_kernel(double* __restrict__ Aall, int* __restrict__ pivall,
                                                               int* __restrict__ infoall, int n) {
  extern __shared__ __align__(16) double lu_sm[];
  double* A = Aall + (size_t)blockIdx.x * n * n;
  int* piv = pivall + (size_t)blockIdx.x * n;
  const int tid = threadIdx.x;
  constexpr int nt = LU_THREADS;
  const int ldp = lu_ldp(n);     // shared-memory stride, a multiple of 4 doubles (16-byte vector loads)
  double* P = lu_sm;             // factored panel, column c at P + c * ldp, local row i = global row j0 + i
  double* U = P + LU_NB * ldp;   // U strip: row k at U + k * ldp, entry jj = global column j0 + nbw + jj
  __shared__ double red_v[nt / 32];
  __shared__ int red_i[nt / 32];
  __shared__ double rowbuf[2][LU_NB];
  __shared__ int s_piv[LU_NB];
  __shared__ int aff_dst[2 * LU_NB], aff_src[2 * LU_NB], aff_n;
  __shared__ int s_info;
  if (tid == 0) s_info = 0;
  for (int j0 = 0; j0 < n; j0 += LU_NB) {
    const int nbw = min(LU_NB, n - j0);
    const int m = n - j0;
    // ---- panel rows into registers: slot s of this thread is local row tid + s * nt
    double row[RPT][LU_NB];
#pragma unroll
    for (int s = 0; s < RPT; ++s) {
      const int i = tid + s * nt;
#pragma unroll
      for (int c = 0; c < LU_NB; ++c) row[s][c] = (i < m && c < nbw) ? A[(size_t)(j0 + c) * n + j0 + i] : 0.0;
    }
#pragma unroll
    for (int c = 0; c < LU_NB; ++c) {
      if (c < nbw) {  // uniform
        // pivot search over local rows >= c
        double bv = -1.0;
        int bi = c;
#pragma unroll
        for (int s = 0; s < RPT; ++s) {
          const int i = tid + s * nt;
          const double v = fabs(row[s][c]);
          if (i >= c && i < m && v > bv) {
            bv = v;
            bi = i;
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {  // ties go to the lowest row: independent of the schedule
          const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
          const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
          if (ov > bv || (ov == bv && oi < bi)) {
            bv = ov;
            bi = oi;
          }
        }
        if ((tid & 31) == 0) {
          red_v[tid >> 5] = bv;
          red_i[tid >> 5] = bi;
        }
        __syncthreads();
        bv = red_v[0];
        bi = red_i[0];
#pragma unroll
        for (int w = 1; w < nt / 32; ++w)
          if (red_v[w] > bv || (red_v[w] == bv && red_i[w] < bi)) {
            bv = red_v[w];
            bi = red_i[w];
          }
        if (tid == 0) {
          s_piv[c] = bi;
          piv[j0 + c] = j0 + bi;
          if (!(bv > 0.0) && s_info == 0) s_info = j0 + c + 1;  // exactly singular (or NaN) pivot column
        }
        // exchange rows c and bi through shared memory (their owners publish them)
#pragma unroll
        for (int s = 0; s < RPT; ++s) {
          const int i = tid + s * nt;
          if (i == c)
#pragma unroll
            for (int cc = 0; cc < LU_NB; ++cc) rowbuf[0][cc] = row[s][cc];
          if (i == bi)
#pragma unroll
            for (int cc = 0; cc < LU_NB; ++cc) rowbuf[1][cc] = row[s][cc];
        }
        __syncthreads();
#pragma unroll
        for (int s = 0; s < RPT; ++s) {
          const int i = tid + s * nt;
          if (i == c && bi != c)
#pragma unroll
            for (int cc = 0; cc < LU_NB; ++cc) row[s][cc] = rowbuf[1][cc];
          else if (i == bi && bi != c)
#pragma unroll
            for (int cc = 0; cc < LU_NB; ++cc) row[s][cc] = rowbuf[0][cc];
        }
        const double pv = rowbuf[1][c];
        const double inv = pv != 0.0 ? 1.0 / pv : 0.0;
#pragma unroll
        for (int s = 0; s < RPT; ++s) {
          const int i = tid + s * nt;
          if (i > c && i < m) {
            const double l = row[s][c] * inv;
            row[s][c] = l;
#pragma unroll
            for (int cc = c + 1; cc < LU_NB; ++cc) row[s][cc] -= l * rowbuf[1][cc];
          }
        }
      }
    }
    // ---- panel back to global memory and into shared memory (L11 / L21 for the trailing phases)
#pragma unroll
    for (int s = 0; s < RPT; ++s) {
      const int i = tid + s * nt;
      if (i < m)
#pragma unroll
        for (int c = 0; c < LU_NB; ++c)
          if (c < nbw) {
            A[(size_t)(j0 + c) * n + j0 + i] = row[s][c];
            P[c * ldp + i] = row[s][c];
          }
    }
    const int nrem = n - j0 - nbw;  // trailing columns (and rows below the panel's square)
    if (nrem <= 0) break;
    // ---- the panel's interchanges composed into one gather: new[aff_dst[t]] = old[aff_src[t]]
    // (warp 0, entry t of the list on lane t: a serial version on one thread kept the other 255 waiting for
    // ~2.5 us per panel)
    if (tid < 32) {
      int row_l = tid < nbw ? tid : -1, content_l = row_l, cnt = nbw;
      for (int c = 0; c < nbw; ++c) {
        const int r = s_piv[c];  // s_piv writes are ordered by the barriers of the column loop
        const unsigned hit = __ballot_sync(0xffffffffu, tid < cnt && row_l == r);
        int pos;
        if (hit) {
          pos = __ffs(hit) - 1;
        } else {
          pos = cnt++;
          if (tid == pos) row_l = content_l = r;
        }
        const int at_c = __shfl_sync(0xffffffffu, content_l, c), at_pos = __shfl_sync(0xffffffffu, content_l, pos);
        if (tid == c) content_l = at_pos;
        else if (tid == pos) content_l = at_c;
      }
      if (tid < cnt) {
        aff_dst[tid] = row_l;
        aff_src[tid] = content_l;
      }
      if (tid == 0) aff_n = cnt;
    }
    __syncthreads();
    // ---- trailing columns: interchanges, then U12 = L11^{-1} A12 (one thread per column)
    for (int jj = tid; jj < nrem; jj += nt) {
      double* col = A + (size_t)(j0 + nbw + jj) * n + j0;
      const int na = aff_n;
      double vals[2 * LU_NB];
#pragma unroll
      for (int t = 0; t < 2 * LU_NB; ++t) vals[t] = t < na ? col[aff_src[t]] : 0.0;
#pragma unroll
      for (int t = LU_NB; t < 2 * LU_NB; ++t)
        if (t < na) col[aff_dst[t]] = vals[t];
      if (nbw < LU_NB) {  // last, narrow panel: entries nbw..na-1 are pivot rows as well
#pragma unroll
        for (int t = 0; t < LU_NB; ++t)
          if (t >= nbw && t < na) col[aff_dst[t]] = vals[t];
      }
      // rows 0..nbw-1 of the strip are vals[0..nbw-1] (aff_dst[t] = t for t < nbw)
#pragma unroll
      for (int k = 0; k < LU_NB; ++k)
#pragma unroll
        for (int i = k + 1; i < LU_NB; ++i)
          if (i < nbw) vals[i] -= P[k * ldp + i] * vals[k];
#pragma unroll
      for (int k = 0; k < LU_NB; ++k)
        if (k < nbw) {
          col[k] = vals[k];
          U[k * ldp + jj] = vals[k];
        }
    }
    __syncthreads();
    // ---- trailing update A22 -= L21 U12 on the fp64 tensor cores: warp tile 32 rows x 16 columns = 4 x 2 m8n8k4
    // accumulators, A fragments from L21 (negated), B fragments from the U strip, C fragments read from / written to
    // A22 in place (a fragment's 8 rows of one column are 64 contiguous bytes), requested before the products so that
    // their L2 latency overlaps them (with FMA tiles: 0.98 ms vs 1.98 ms without).  32 MMAs per 24 shared-memory
    // loads against 16 multiply-adds per 6 loads in 4 x 4 FMA register tiles; same time (1.44 ms per 296 blocks of
    // 337^2: the update streams A22), fewer issue slots.
    {
      const int lane = tid & 31, w = tid >> 5, g = lane >> 2, t4 = lane & 3;
      const double* L21 = P + nbw;  // local row i of L21 = panel row nbw + i
      double* A22 = A + (size_t)(j0 + nbw) * n + j0 + nbw;
      const int n_rt = (nrem + 31) >> 5, n_ct = (nrem + 15) >> 4;
      for (int tile = w; tile < n_rt * n_ct; tile += nt / 32) {
        const int rb = (tile % n_rt) * 32, cb = (tile / n_rt) * 16;
        double c[4][2][2];
#pragma unroll
        for (int bq = 0; bq < 2; ++bq)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int col = cb + 8 * bq + 2 * t4 + e;
            const double* cp = A22 + (size_t)col * n + rb + g;
#pragma unroll
            for (int a = 0; a < 4; ++a) c[a][bq][e] = (col < nrem && rb + 8 * a + g < nrem) ? cp[8 * a] : 0.0;
          }
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const int k = 4 * kk + t4;
          // rows / columns past nrem read whatever the panel / strip hold (inside the shared-memory block); the
          // accumulators they feed are never stored
          double af[4], bf[2];
#pragma unroll
          for (int a = 0; a < 4; ++a) af[a] = k < nbw ? -L21[k * ldp + rb + 8 * a + g] : 0.0;
#pragma unroll
          for (int bq = 0; bq < 2; ++bq) bf[bq] = k < nbw ? U[k * ldp + cb + 8 * bq + g] : 0.0;
#pragma unroll
          for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int bq = 0; bq < 2; ++bq) dmma_m8n8k4(c[a][bq][0], c[a][bq][1], af[a], bf[bq]);
        }
#pragma unroll
        for (int bq = 0; bq < 2; ++bq)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int col = cb + 8 * bq + 2 * t4 + e;
            double* cp = A22 + (size_t)col * n + rb + g;
#pragma unroll
            for (int a = 0; a < 4; ++a)
              if (col < nrem && rb + 8 * a + g < nrem) cp[8 * a] = c[a][bq][e];
          }
      }
    }
    __syncthreads();
  }
  __syncthreads();
  if (tid == 0) infoall[blockIdx.x] = s_info;
}

// ---------------------------------------------------------------------------------------------------------------
// Solve with the factors: B (n x nrhs, row-major, i.e. right-hand side c of row i at B[i * nrhs + c]) is overwritten
// by the solution, the right-hand sides of a CTA kept in shared memory for the whole forward and backward substitution.
// The factor columns of a step (rows below the panel going forward, above it going back) are STAGED in shared memory
// with cp.async WHILE warp 0 applies the interchanges and solves the triangle -- neither depends on the other -- and the
// diagonal block and pivots of the NEXT step travel with them; the update then reads only shared memory.  The round-1
// substitution read the factor from L2 in its row updates (4 panel columns at a time, FMA register tiles, the triangle
// on one warp while seven waited): 17 800 cycles per panel step on B200, 15 % of them arithmetic, and 1.18 ms against
// this kernel's 0.93 ms per stage of 296 blocks of 337^2 with 88 right-hand sides.
__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gsrc) {
  const unsigned sdst = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sdst), "l"(gsrc));
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
  const unsigned sdst = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(sdst), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// stride of a staged column: >= the rows outside a panel, and = 8 mod 16 so that the A-fragment reads of the
// tensor-core update (4 consecutive k x 8 consecutive rows per warp) hit every bank pair exactly twice
__host__ __device__ inline int lu_staged_ps(int n) {
  const int m = n > 8 ? n - 8 : 1;  // rows outside a half panel (LU_SNB = 8 columns)
  return ((m + 7) & ~15) + 8;
}
__host__ __device__ inline size_t lu_staged_smem(int n, int ct) {
  // right-hand sides b[n][8 ct] + staged half panel P[8][ps]
  return ((size_t)n * (8 * ct) + (size_t)8 * lu_staged_ps(n) + 2) * sizeof(double);
}

// CT = 8-column tiles of right-hand sides per CTA: 4 (32 columns, two CTAs per SM for the 337-blocks) or 3 where 32
// columns no longer fit (api.cu::lu_plan).
// * The rows outside the panel are updated on the TENSOR CORES: b[rows][:] += (-P) Y with m8n8k4 fp64 MMAs, 8 x fewer
//   instructions than 4 x 6 register tiles of fused multiply-adds and a third of their shared-memory reads.
// * With the update that cheap, the triangle of the panel -- one warp, one right-hand side per lane, the other seven
//   warps waiting -- was 40 % of the kernel (ncu).  The substitution therefore walks HALF panels (LU_SNB = 8 columns:
//   valid because the factor kernel interchanges LAPACK-style inside a 16-column panel; the panel's 16 interchanges are
//   applied on its first half): 28 instead of 120 dependent multiply-adds per step, warp 0 takes no part in the staging,
//   and the reciprocals of U's diagonal are computed one step ahead by an otherwise idle warp (the fp64 divisions of the
//   backward sweep were the longest dependent chain).
constexpr int LU_SNB = 8;

template <int CT>
__global__ void __launch_bounds__(LU_THREADS, 2) lu_solve_staged_kernel(const double* __restrict__ LUall,
                                                                        const int* __restrict__ pivall,
                                                                        double* __restrict__ Ball, int n, int nrhs, int n_chunks) {
  constexpr int RC = 8 * CT;
  constexpr int nt = LU_THREADS;
  constexpr int ldb = RC;
  extern __shared__ __align__(16) double lu_sm[];
  // the column chunks of one matrix are neighbours in launch order: they run at the same time and share the factor in
  // L2 (with the matrix index fastest they ran waves apart and each streamed it from DRAM: 943 MB per launch of 296)
  const size_t mat = blockIdx.x / n_chunks;
  const double* A = LUall + mat * n * n;
  const int* piv = pivall + mat * n;
  double* Bg = Ball + mat * n * nrhs;
  const int c0 = (blockIdx.x % n_chunks) * RC;
  const int nc = min(RC, nrhs - c0);
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int ps = lu_staged_ps(n);
  double* b = lu_sm;                     // b[i * ldb + c]; columns >= nc are zero
  double* P = lu_sm + (size_t)n * ldb;   // P[k * ps + i] = A[r0 + i, j0 + k]
  __shared__ double tri[2][LU_SNB][LU_SNB + 1];  // tri[s & 1][k][i] = A[j0 + i, j0 + k] of step s
  __shared__ double rinv[2][LU_SNB];             // backward steps: 1 / U[j0 + k, j0 + k]
  __shared__ int s_piv[2][LU_NB];
  const int S = (n + LU_SNB - 1) / LU_SNB;  // steps 0 .. S-1 forward, S .. 2S-1 backward (half panels aligned from the end)
  auto panel_of = [&](int s, int& j0, int& nbw) {
    if (s < S) {
      j0 = LU_SNB * s;
      nbw = min(LU_SNB, n - j0);
    } else {
      const int j1 = n - LU_SNB * (s - S);
      j0 = max(0, j1 - LU_SNB);
      nbw = j1 - j0;
    }
  };
  // diagonal block of step s into buffer s & 1 (threads t0 .. t0 + 63), pivots of a full panel (threads t0 + 64 .. + 79)
  auto fetch_tri = [&](int s, int t0) {
    int j0, nbw;
    panel_of(s, j0, nbw);
    const int t = tid - t0;
    if (t >= 0 && t < LU_SNB * LU_SNB) {
      const int k = t >> 3, i = t & 7;
      if (k < nbw && i < nbw) cp_async8(&tri[s & 1][k][i], &A[(size_t)(j0 + k) * n + j0 + i]);
      else tri[s & 1][k][i] = 0.0;
    }
    if (s < S && (j0 % LU_NB) == 0 && t >= 64 && t < 64 + LU_NB && j0 + t - 64 < n)
      cp_async4(&s_piv[s & 1][t - 64], &piv[j0 + t - 64]);
  };
  fetch_tri(0, 0);
  cp_async_commit();
  for (int e = tid; e < n * RC; e += nt) {
    const int i = e / RC, c = e - i * RC;
    b[i * ldb + c] = c < nc ? Bg[(size_t)i * nrhs + c0 + c] : 0.0;
  }
  cp_async_wait_all();
  __syncthreads();
  for (int s = 0; s < 2 * S; ++s) {
    int j0, nbw;
    panel_of(s, j0, nbw);
    const bool fwd = s < S;
    const int r0 = fwd ? j0 + nbw : 0, r1 = fwd ? n : j0;
    const int m = r1 - r0;
    if (w > 0) {
      // ---- warps 1..7 stage the step's factor columns and the next step's diagonal block
      for (int k = 0; k < nbw; ++k) {
        const double* src = A + (size_t)(j0 + k) * n + r0;
        double* dst = P + (size_t)k * ps;
        for (int i = tid - 32; i < m; i += nt - 32) cp_async8(dst + i, src + i);
      }
      if (s + 1 < 2 * S) fetch_tri(s + 1, 32);
      cp_async_commit();
      cp_async_wait_all();
    } else if (lane < RC) {
      // ---- warp 0 meanwhile: interchanges and the triangle of this half panel, one right-hand side per lane
      const double(*T)[LU_SNB + 1] = tri[s & 1];
      if (fwd) {
        if ((j0 % LU_NB) == 0) {
          const int np = min(LU_NB, n - j0);
          for (int c = 0; c < np; ++c) {
            const int r = s_piv[s & 1][c];
            if (r != j0 + c) {
              const double t = b[(j0 + c) * ldb + lane];
              b[(j0 + c) * ldb + lane] = b[r * ldb + lane];
              b[r * ldb + lane] = t;
            }
          }
        }
        double y[LU_SNB];
#pragma unroll
        for (int k = 0; k < LU_SNB; ++k) y[k] = k < nbw ? b[(j0 + k) * ldb + lane] : 0.0;
#pragma unroll
        for (int k = 0; k < LU_SNB; ++k)
#pragma unroll
          for (int i = k + 1; i < LU_SNB; ++i) y[i] -= T[k][i] * y[k];  // entries outside the block are zero
#pragma unroll
        for (int k = 0; k < LU_SNB; ++k)
          if (k < nbw) b[(j0 + k) * ldb + lane] = y[k];
      } else {
        double xv[LU_SNB];
#pragma unroll
        for (int k = 0; k < LU_SNB; ++k) xv[k] = k < nbw ? b[(j0 + k) * ldb + lane] : 0.0;
#pragma unroll
        for (int k = LU_SNB - 1; k >= 0; --k)
          if (k < nbw) {
            xv[k] = xv[k] * rinv[s & 1][k];
#pragma unroll
            for (int i = 0; i < k; ++i) xv[i] -= T[k][i] * xv[k];
          }
#pragma unroll
        for (int k = 0; k < LU_SNB; ++k)
          if (k < nbw) b[(j0 + k) * ldb + lane] = xv[k];
      }
    }
    __syncthreads();
    // ---- reciprocals of the next backward step's diagonal (its block landed with this step's copies)
    if (w == 7 && lane < LU_SNB && s + 1 >= S && s + 1 < 2 * S) {
      const double d = tri[(s + 1) & 1][lane][lane];
      rinv[(s + 1) & 1][lane] = 1.0 / d;  // a zero pivot keeps its IEEE consequences (inf / NaN: the caller's failed-solve path)
    }
    // ---- rows outside the panel on the tensor cores: an 8-row tile per warp and trip, all CT column tiles
    {
      const int g = lane >> 2, t4 = lane & 3;
      double yb[CT][LU_SNB / 4];  // B fragments: Y[k][col], k = 4 kk + t4, col = 8 ct + g
#pragma unroll
      for (int ct = 0; ct < CT; ++ct)
#pragma unroll
        for (int kk = 0; kk < LU_SNB / 4; ++kk) {
          const int k = 4 * kk + t4;
          yb[ct][kk] = k < nbw ? b[(j0 + k) * ldb + 8 * ct + g] : 0.0;
        }
      const int n_rt = (m + 7) >> 3;
      for (int rt = w; rt < n_rt; rt += nt / 32) {
        const int i = rt * 8 + g;  // row inside the staged columns
        const bool valid = i < m;
        double a[LU_SNB / 4];
#pragma unroll
        for (int kk = 0; kk < LU_SNB / 4; ++kk) {
          const int k = 4 * kk + t4;
          a[kk] = (valid && k < nbw) ? -P[(size_t)k * ps + i] : 0.0;
        }
        double2* crow = reinterpret_cast<double2*>(b + (size_t)(r0 + (valid ? i : 0)) * ldb + 2 * t4);
#pragma unroll
        for (int ct = 0; ct < CT; ++ct) {
          double2 c = valid ? crow[4 * ct] : make_double2(0.0, 0.0);  // rows past the end are neither read nor written
#pragma unroll
          for (int kk = 0; kk < LU_SNB / 4; ++kk) dmma_m8n8k4(c.x, c.y, a[kk], yb[ct][kk]);
          if (valid) crow[4 * ct] = c;
        }
      }
    }
    __syncthreads();
  }
  for (int e = tid; e < n * nc; e += nt) {
    const int i = e / nc, c = e - i * nc;
    Bg[(size_t)i * nrhs + c0 + c] = b[i * ldb + c];
  }
}

}  // namespace hb

// ---------------------------------------------------------------------------------------------------------------
// Sparse products with the CCS value arrays of jac_g / hess_l for the interior-point driver (ipsolver.SparseOps):
//   y[b][o] = sum_{q = ptr[o]}^{ptr[o+1]-1} w[q] * vals[b][entry[q]] * x[b][idx[q]]
// One thread per (instance, output element) walks its entries in a fixed order: no atomics, so every residual of
// the solver is reproducible run to run (the index_add_ formulation was not: VERDICT round 1).
namespace hb {
__global__ void ccs_group_mul_kernel(const double* __restrict__ vals, const int* __restrict__ ptr,
                                     const int* __restrict__ entry, const int* __restrict__ idx,
                                     const double* __restrict__ w, const double* __restrict__ x, double* __restrict__ y,
                                     int n_out, int n_in, long nnz, long batch) {
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= batch * n_out) return;
  const long b = t / n_out;
  const int o = (int)(t % n_out);
  const double* vb = vals + b * nnz;
  const double* xb = x + b * n_in;
  double acc = 0.0;
  for (int q = ptr[o]; q < ptr[o + 1]; ++q) {
    const double v = vb[entry[q]] * xb[idx[q]];
    acc += w ? w[q] * v : v;
  }
  y[t] = acc;
}
}  // namespace hb

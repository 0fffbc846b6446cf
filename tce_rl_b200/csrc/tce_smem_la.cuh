// Small dense linear algebra on shared-memory matrices (fp64), executed cooperatively by one CTA.
// Building blocks of the trust-region projection kernels (n <= 64: Dp = 63 / 36 / 28 / 12).
// Every routine is called by ALL threads of the CTA and ends with __syncthreads().
#pragma once
#include "tce_common.cuh"

struct Mat {            // strided view; a transpose is a stride swap
  double *p;
  int rs, cs;
  __device__ __forceinline__ double &operator()(int i, int j) const { return p[i * rs + j * cs]; }
  __device__ __forceinline__ Mat T() const { return Mat{p, cs, rs}; }
};

enum { TRI_FULL = 0, TRI_LOWER = 1, TRI_UPPER = 2 };

__device__ __forceinline__ float la_rsqrt_approx(float x) {   // bare MUFU: no denormal fix-up code around it
  float y;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float la_rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}


// D += A B for one 8x8x4 fp64 tile on the tensor cores (SASS DMMA.8x8x4).  Lane l holds A(l / 4, l % 4),
// B(l % 4, l / 4) and D(l / 4, 2 (l % 4) + {0, 1}).
__device__ __forceinline__ void la_dmma(double (&d)[2], double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
      : "+d"(d[0]), "+d"(d[1]) : "d"(a), "d"(b));
}

// C = beta * C + alpha * A B (m x n x k, all <= 64) on the fp64 tensor cores: each warp owns a 16 x 16 block of
// C as 2 x 2 DMMA tiles, so per k step of 4 it loads two A and two B fragments (one LDS.64 each) for four DMMA
// (1024 FMA); the scalar 4x4-tile version issued 8 shared-memory wavefronts per 16 DFMA per lane and ran the
// fp64 pipe at about half its rate.  Tile rows (and columns) are INTERLEAVED: fragment row g of tile t is row
// 4 (g % 4) + g / 4 + 2 t of the block, so that a half-warp's four rows lie 4 apart; with the odd leading
// dimensions of the callers' buffers the 16 addresses of every fragment load then fall in 16 distinct 8-byte
// banks, for A and B, transposed or not.  Each output is summed in ascending k with one rounded FMA per product,
// the same arithmetic as a scalar loop (scripts/ubench/gemm.cu checks this bit for bit).
// a_tri / b_tri describe the structure of A and B and only clip the k range: the unused triangle of a
// triangular operand MUST hold zeros.  Fragment elements outside [0, m) x [0, k) of A and [0, k) x [0, n) of B
// are never read (they may be another buffer, or C itself in la_chol).  c_tri is a hint that only that triangle
// of C is read afterwards; all of the m x n C is written.
__device__ inline void la_gemm(Mat C, Mat A, Mat B, int m, int n, int k, int a_tri, int b_tri, int c_tri,
                               double alpha, double beta) {
  (void)c_tri;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = (int)(blockDim.x >> 5);
  const int g = lane >> 2, q = lane & 3, pg = 4 * (g & 3) + (g >> 2);
  const int TN = (n + 15) >> 4, nblk = ((m + 15) >> 4) * TN;
  for (int t = warp; t < nblk; t += nwarp) {
    const int r0 = (t / TN) << 4, c0 = (t - (t / TN) * TN) << 4;
    int lo = 0, hi = k;                                  // multiples of 16, or k
    if (a_tri == TRI_LOWER) hi = min(hi, r0 + 16);
    if (a_tri == TRI_UPPER) lo = max(lo, r0);
    if (b_tri == TRI_LOWER) lo = max(lo, c0);
    if (b_tri == TRI_UPPER) hi = min(hi, c0 + 16);
    const int ra = r0 + pg, cb = c0 + pg;
    const bool va0 = ra < m, va1 = ra + 2 < m, vb0 = cb < n, vb1 = cb + 2 < n;
    const double *pa0 = &A(va0 ? ra : 0, 0), *pa1 = &A(va1 ? ra + 2 : 0, 0);
    const double *pb0 = &B(0, vb0 ? cb : 0), *pb1 = &B(0, vb1 ? cb + 2 : 0);
    double d[2][2][2] = {};
#pragma unroll 2
    for (int k0 = lo; k0 < hi; k0 += 4) {
      const int kk = k0 + q;
      const bool vk = kk < hi;
      const double a0 = (vk && va0) ? pa0[kk * A.cs] : 0.0, a1 = (vk && va1) ? pa1[kk * A.cs] : 0.0;
      const double b0 = (vk && vb0) ? pb0[kk * B.rs] : 0.0, b1 = (vk && vb1) ? pb1[kk * B.rs] : 0.0;
      la_dmma(d[0][0], a0, b0);
      la_dmma(d[0][1], a0, b1);
      la_dmma(d[1][0], a1, b0);
      la_dmma(d[1][1], a1, b1);
    }
#pragma unroll
    for (int ti = 0; ti < 2; ++ti) {
      const int i = ra + 2 * ti;
#pragma unroll
      for (int tj = 0; tj < 2; ++tj) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int f = 2 * q + e, j = c0 + 4 * (f & 3) + (f >> 2) + 2 * tj;
          const double v = d[ti][tj][e];
          if (i < m && j < n) C(i, j) = beta == 0.0 ? alpha * v : fma(beta, C(i, j), alpha * v);
        }
      }
    }
  }
  __syncthreads();
}

constexpr int LA_NB = 8;                              // block size of the blocked triangular routines
constexpr int LA_DINV_DOUBLES = 8 * LA_NB * LA_NB;    // scratch for the inverted diagonal blocks (n <= 64)

// dinv[bk][i][j] = inverse of the bk-th LA_NB x LA_NB diagonal block of the lower-triangular L (zeros above
// the diagonal).  One warp per block, lane j < 8 builds column j.
__device__ inline void la_diag_block_inverses(Mat L, double *dinv, int n) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = (int)(blockDim.x >> 5);
  const int nblk = (n + LA_NB - 1) / LA_NB;
  for (int bk = warp; bk < nblk; bk += nwarp) {
    if (lane < LA_NB) {
      const int r0 = bk * LA_NB, j = lane;
      double x[LA_NB];
#pragma unroll
      for (int i = 0; i < LA_NB; ++i) {
        const int gi = r0 + i;
        double v = (i == j) ? 1.0 : 0.0;
        if (gi < n) {
#pragma unroll
          for (int q = 0; q < i; ++q) v = fma(-L(gi, r0 + q), x[q], v);     // x[q] = 0 for q < j
          v = (i >= j) ? v / L(gi, gi) : 0.0;
        } else {
          v = 0.0;
        }
        x[i] = v;
        dinv[(bk * LA_NB + i) * LA_NB + j] = v;
      }
    }
  }
  __syncthreads();
}

// X <- L^-1 for a lower-triangular L (n <= 64, X must not alias L; dinv: LA_DINV_DOUBLES doubles of scratch).
// Recursive doubling instead of forward substitution: the 8x8 diagonal blocks are inverted directly, then
// blocks of width w = 8, 16, 32 are merged pairwise,
//   [A1 0; C A2]^-1 = [A1^-1 0; -A2^-1 C A1^-1  A2^-1],
// two small products per level with every output element on its own thread: 3 levels x 3 barriers
// (scripts/ubench/gemm.cu gives the cycles), where the blocked substitution needs 8 dependent block rows (~25k
// cycles with n right-hand sides).  A solve with n right-hand sides is then ONE triangular GEMM.  For the factors met here (covariance factors,
// condition ~1e2) the explicit inverse loses nothing measurable in fp64.  Needs blockDim.x >= 256.
__device__ inline void la_tri_inverse(Mat L, Mat X, double *dinv, int n) {
  la_diag_block_inverses(L, dinv, n);
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, j = e - i * n;
    X(i, j) = (i >> 3) == (j >> 3) ? dinv[((i >> 3) * LA_NB + (i & 7)) * LA_NB + (j & 7)] : 0.0;
  }
  __syncthreads();
  for (int lw = 3; (1 << lw) < n; ++lw) {
    const int w = 1 << lw, npair = (n + 2 * w - 1) >> (lw + 1), nout = npair << (2 * lw);
    double v[4];
    // T = C A1^-1 into the (still zero) block below the diagonal: T(i, j) = sum_{k >= j} L(i, k) A1inv(k, j)
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int o = threadIdx.x + u * (int)blockDim.x;
      v[u] = 0.0;
      if (o < nout) {
        const int pr = o >> (2 * lw), rem = o & ((1 << (2 * lw)) - 1), ii = rem >> lw, jj = rem & (w - 1);
        const int c0 = pr << (lw + 1), i = c0 + w + ii, j = c0 + jj;
        if (i < n) {
          // k runs over the WHOLE block (A1inv(k, j) = 0 for k < j, exact zeros that leave the sums unchanged): the
          // lanes of a warp then read L(i, k) as a broadcast and A1inv(k, .) as a row.  Starting at k = j would give
          // each lane its own k: a diagonal walk through X with a 4-way bank conflict on every load.
          double a0 = 0.0, a1 = 0.0;                                  // even k, odd k
          for (int k = 0; k < w; k += 2) { a0 = fma(L(i, c0 + k), X(c0 + k, j), a0); a1 = fma(L(i, c0 + k + 1), X(c0 + k + 1, j), a1); }
          v[u] = a0 + a1;
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int o = threadIdx.x + u * (int)blockDim.x;
      if (o < nout) {
        const int pr = o >> (2 * lw), rem = o & ((1 << (2 * lw)) - 1), ii = rem >> lw, jj = rem & (w - 1);
        const int c0 = pr << (lw + 1), i = c0 + w + ii, j = c0 + jj;
        if (i < n) X(i, j) = v[u];
      }
    }
    __syncthreads();
    // block <- -A2^-1 T (in place: every output is formed in a register before anything is overwritten)
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int o = threadIdx.x + u * (int)blockDim.x;
      v[u] = 0.0;
      if (o < nout) {
        const int pr = o >> (2 * lw), rem = o & ((1 << (2 * lw)) - 1), ii = rem >> lw, jj = rem & (w - 1);
        const int c0 = pr << (lw + 1), r0 = c0 + w, i = r0 + ii, j = c0 + jj;
        if (i < n) {
          double a0 = 0.0, a1 = 0.0;
          int k = 0;
          for (; k + 1 <= ii; k += 2) { a0 = fma(X(i, r0 + k), X(r0 + k, j), a0); a1 = fma(X(i, r0 + k + 1), X(r0 + k + 1, j), a1); }
          if (k <= ii) a0 = fma(X(i, r0 + k), X(r0 + k, j), a0);
          v[u] = -(a0 + a1);
        }
      }
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int o = threadIdx.x + u * (int)blockDim.x;
      if (o < nout) {
        const int pr = o >> (2 * lw), rem = o & ((1 << (2 * lw)) - 1), ii = rem >> lw, jj = rem & (w - 1);
        const int c0 = pr << (lw + 1), i = c0 + w + ii, j = c0 + jj;
        if (i < n) X(i, j) = v[u];
      }
    }
    __syncthreads();
  }
}

// X <- L^-1 X, L lower triangular n x n, X n x ncols, dinv from la_diag_block_inverses(L).  Four lanes
// share one column (split-k over the already solved rows), one barrier per block row.
// x_lower: X(i, c) = 0 for i < c on entry (and on exit), those entries are skipped.
__device__ inline void la_trsm_lower(Mat L, const double *dinv, Mat X, int n, int ncols, bool x_lower) {
  constexpr int SUB = 4;
  const int sub = threadIdx.x % SUB;
  const unsigned gmask = ((1u << SUB) - 1u) << ((threadIdx.x & 31) & ~(SUB - 1));
  const int ncols_pad = ((ncols + 7) / 8) * 8;          // keep whole warps in the loop (shuffles below)
  for (int r0 = 0; r0 < n; r0 += LA_NB) {
    const int bk = r0 / LA_NB;
    for (int cc = threadIdx.x / SUB; cc < ncols_pad; cc += (int)blockDim.x / SUB) {
      const bool live = cc < ncols && !(x_lower && cc >= r0 + LA_NB);    // else structurally zero / padding
      const int c = cc < ncols ? cc : ncols - 1;
      double acc[LA_NB];
#pragma unroll
      for (int i = 0; i < LA_NB; ++i) acc[i] = 0.0;
      if (live) {
        const int q_lo = x_lower ? (c / SUB) * SUB : 0;       // aligned so that the SUB lanes partition it
        for (int q = q_lo + sub; q < r0; q += SUB) {
          const double xq = X(q, c);
#pragma unroll
          for (int i = 0; i < LA_NB; ++i) acc[i] = fma(L(min(r0 + i, n - 1), q), xq, acc[i]);
        }
      }
#pragma unroll
      for (int i = 0; i < LA_NB; ++i) {
        acc[i] += __shfl_xor_sync(gmask, acc[i], 1);
        acc[i] += __shfl_xor_sync(gmask, acc[i], 2);
      }
      if (live && sub == 0) {
        double x[LA_NB];
#pragma unroll
        for (int i = 0; i < LA_NB; ++i) x[i] = (r0 + i < n) ? X(r0 + i, c) - acc[i] : 0.0;
#pragma unroll
        for (int i = 0; i < LA_NB; ++i) {
          if (r0 + i < n) {
            double y = 0.0;
#pragma unroll
            for (int q = 0; q <= i; ++q) y = fma(dinv[(bk * LA_NB + i) * LA_NB + q], x[q], y);
            if (!(x_lower && r0 + i < c)) X(r0 + i, c) = y;
          }
        }
      }
    }
    __syncthreads();
  }
}

// X <- L^-T X (back substitution with the transpose of the lower-triangular L)
__device__ inline void la_trsm_lower_t(Mat L, const double *dinv, Mat X, int n, int ncols) {
  constexpr int SUB = 4;
  const int sub = threadIdx.x % SUB;
  const unsigned gmask = ((1u << SUB) - 1u) << ((threadIdx.x & 31) & ~(SUB - 1));
  const int nblk = (n + LA_NB - 1) / LA_NB;
  const int ncols_pad = ((ncols + 7) / 8) * 8;
  for (int bk = nblk - 1; bk >= 0; --bk) {
    const int r0 = bk * LA_NB, r1 = min(r0 + LA_NB, n);
    for (int cc = threadIdx.x / SUB; cc < ncols_pad; cc += (int)blockDim.x / SUB) {
      const bool live = cc < ncols;
      const int c = live ? cc : ncols - 1;
      double acc[LA_NB];
#pragma unroll
      for (int i = 0; i < LA_NB; ++i) acc[i] = 0.0;
      if (live) {
        for (int q = r1 + sub; q < n; q += SUB) {
          const double xq = X(q, c);
#pragma unroll
          for (int i = 0; i < LA_NB; ++i) acc[i] = fma(L(q, min(r0 + i, n - 1)), xq, acc[i]);
        }
      }
#pragma unroll
      for (int i = 0; i < LA_NB; ++i) {
        acc[i] += __shfl_xor_sync(gmask, acc[i], 1);
        acc[i] += __shfl_xor_sync(gmask, acc[i], 2);
      }
      if (live && sub == 0) {
        double x[LA_NB];
#pragma unroll
        for (int i = 0; i < LA_NB; ++i) x[i] = (r0 + i < n) ? X(r0 + i, c) - acc[i] : 0.0;
#pragma unroll
        for (int i = 0; i < LA_NB; ++i) {
          if (r0 + i < n) {
            double y = 0.0;                                   // (D^-1)^T : y_i = sum_{q >= i} dinv[q][i] x_q
#pragma unroll
            for (int q = i; q < LA_NB; ++q) y = fma(dinv[(bk * LA_NB + q) * LA_NB + i], x[q], y);
            X(r0 + i, c) = y;
          }
        }
      }
    }
    __syncthreads();
  }
}

// in-place blocked Cholesky of the lower triangle of A (n <= 64; the upper triangle is scratch on exit); *bad
// (shared int, pre-set to 0) receives the 1-based index of the first non-positive pivot.  Per block of 8
// columns: warp 0 factors the whole panel (rows r0..n-1) in REGISTERS -- lane l holds rows l and l + 32, pivots
// and multipliers travel by shuffle, one rsqrt per column -- then everybody applies the rank-8 update to the
// trailing matrix with la_gemm (k = 8).  Two barriers per 8 columns.
__device__ inline void la_chol(Mat A, int n, int *bad) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r0 = 0; r0 < n; r0 += LA_NB) {
    const int nb = min(LA_NB, n - r0);
    if (warp == 0) {
      double p[2][LA_NB];
#pragma unroll
      for (int s = 0; s < 2; ++s)
#pragma unroll
        for (int c = 0; c < LA_NB; ++c) {
          const int row = lane + 32 * s;
          p[s][c] = (row >= r0 && row < n && c < nb) ? A(row, r0 + c) : 0.0;
        }
#pragma unroll
      for (int j = 0; j < LA_NB; ++j) {
        if (j < nb) {                                               // uniform
          const int col = r0 + j;
          const double djj = __shfl_sync(0xffffffffu, col >= 32 ? p[1][j] : p[0][j], col & 31);
          if (lane == 0 && !(djj > 0.0) && *bad == 0) *bad = col + 1;
          // 1/sqrt: fp32 MUFU seed + two fp64 Newton steps (1e-7 -> 1e-14 -> rounding); the library rsqrt(double)
          // is a ~40-instruction subroutine on the critical path of every column
          double inv = (double)la_rsqrt_approx((float)djj);
          inv = inv * fma(-0.5 * djj, inv * inv, 1.5);
          inv = inv * fma(-0.5 * djj, inv * inv, 1.5);
#pragma unroll
          for (int s = 0; s < 2; ++s) p[s][j] = (lane + 32 * s == col) ? djj * inv : p[s][j] * inv;
#pragma unroll
          for (int c = j + 1; c < LA_NB; ++c) {
            const int rc = r0 + c;                                  // L(rc, col) sits in lane rc % 32
            const double lcj = __shfl_sync(0xffffffffu, rc >= 32 ? p[1][j] : p[0][j], rc & 31);
            p[0][c] = fma(-p[0][j], lcj, p[0][c]);
            p[1][c] = fma(-p[1][j], lcj, p[1][c]);
          }
        }
      }
#pragma unroll
      for (int s = 0; s < 2; ++s)
#pragma unroll
        for (int c = 0; c < LA_NB; ++c) {
          const int row = lane + 32 * s;
          if (row >= r0 && row < n && c < nb) A(row, r0 + c) = p[s][c];
        }
    }
    __syncthreads();
    const int t0 = r0 + nb, mrem = n - t0;
    if (mrem > 0) {                                                 // A22 -= L21 L21^T (barrier inside)
      const Mat L21{&A(t0, r0), A.rs, A.cs};
      la_gemm(Mat{&A(t0, t0), A.rs, A.cs}, L21, L21.T(), mrem, mrem, nb, TRI_FULL, TRI_FULL, TRI_LOWER, -1.0, 1.0);
    }
  }
}

// One-sided (Hestenes) Jacobi: rotate the columns of W (n x n, n <= 64) until they are orthogonal; on exit
// lam_j = |W_j|^2.  A single CTA is bound by instruction issue and by the SM's one-shuffle-per-clock unit, not
// by fp64 latency (DFMA: 8.5 cycles dependent, scripts/ubench/lat.cu), so the matrix lives in REGISTERS for
// the whole iteration: warp w holds rows 16w..16w+15, lane t holds the two columns (P_t, Q_t) of pair slot t, and
// a step is
//   16 DFMA (partial dot) -> one 4-way combine through shared memory (ONE named barrier over the active warps)
//   -> the rotation (computed redundantly and bit-identically by every warp) -> 64 fp64 ops to apply it
//   -> ONE shuffle per register of Q.
// Pair ordering (recursive halving): with the P columns X and the Q columns Y of a segment of `w` lanes,
// w steps that ring-shift Q inside the segment (__shfl_sync with width = w, no selects) meet all X x Y pairs;
// then the halves trade a column set (lower lanes keep P and receive the upper lanes' P as Q, upper lanes
// keep Q and receive the lower lanes' Q as P) and the same is done at width w/2 inside X and inside Y.
// 32 + 16 + ... + 1 = 63 steps meet all 2016 pairs while only Q moves.  Column ids travel with the data;
// any arrangement is a valid start for the next sweep.  Everything that only steers convergence (norms,
// thresholds, the rotation angle) is fp32; the dot product, the normalisation of (c, s) and the rotation
// itself are fp64.  scratch: LA_JACOBI_SCRATCH doubles.  All threads of the CTA must call this.
constexpr int LA_JACOBI_ROWS = 16;                    // rows per thread: 4 warps hold a 64 x 64 matrix
constexpr int LA_JACOBI_WARPS = 64 / LA_JACOBI_ROWS;
constexpr int LA_JACOBI_SCRATCH = 2 * 8 * 32;
#ifdef JAC_PROF
__device__ unsigned int g_jac_prof[8];
#define JP(i) do { const unsigned int _t = clock(); if (threadIdx.x == 0) jp[i] += _t - jt; jt = _t; } while (0)
#else
#define JP(i)
#endif

#ifdef TCE_PROFILE
__device__ float g_jac_diag[8];       // diagnostics of the last call (block 0): max cos^2 met in sweep 0..7
#endif

__device__ __forceinline__ void la_named_barrier(int nthreads) {
  asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory");
}

__device__ __forceinline__ double la_combine(const double *col) {   // fixed-order sum of the warps' partials
  double v = 0.0;
  if (LA_JACOBI_WARPS == 4) v = (col[0] + col[32]) + (col[64] + col[96]);
  else v = ((col[0] + col[32]) + (col[64] + col[96])) + ((col[128] + col[160]) + (col[192] + col[224]));
  return v;
}

// A sweep is the last one when every pair it visited had cos^2 <= LA_JACOBI_TOL2 (cos <= 3.2e-4).  What such a sweep
// leaves behind was measured on the warm-started box-pushing problem (eigenvalues clustered around 1, gaps ~1e-3, so
// rotation angles are NOT small and the textbook c^2 estimate does not apply): cosines <= 2e-5, i.e. a relative error
// of <= 1e-5 in f(N) = U f(lam) U^T -- one order below the 1e-4 parity bound of the projected parameters.  (1e-8
// forced a second, purely confirming sweep in every epoch of an update: 57 k cycles.)  What the KL projection then
// carries (tests/test_gpu_kl_spectra.py, clustered / wide / extreme spectra, n = 1..64, against an fp64 reference;
// B200): Sigma_proj within 1e-5 of max|Sigma|; the fp32 factor within 6e-6 of its max (2 clusters, gaps 1e-4, n = 7);
// the scalars that are sums over lam (kl0, the KL shape / volume parts) within 1e-6 relative -- lam_j = |U~_j|^2 are
// the diagonal of Q^T N Q, so the residual enters them in second order, largest on clusters with gaps of 1e-6.
constexpr float LA_JACOBI_TOL2 = 1e-7f;

struct LaNoIdle { __device__ void operator()(int, int) const {} };

// idle(t, nt): executed by the nt threads of the warps that hold no rows (t = 0..nt-1) while the others iterate;
// it must not touch W, lam or scratch and must not synchronise.
template <typename Idle = LaNoIdle>
__device__ inline int la_jacobi_onesided(Mat W, double *lam, double *scratch, int n, Idle idle = Idle()) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nw = (n + LA_JACOBI_ROWS - 1) / LA_JACOBI_ROWS, nbar = nw * 32;   // warps that hold rows
  int w0 = 1;                                          // pair slots: power of two >= ceil(n / 2), <= 32
  while (2 * w0 < n) w0 <<= 1;
  int sweeps = 0;
  for (int i = threadIdx.x; i < LA_JACOBI_SCRATCH; i += blockDim.x) scratch[i] = 0.0;   // warps >= nw add 0
  __syncthreads();
  if (warp < nw) {
    double *mine = scratch + warp * 32 + lane;         // this thread's partial; its lane's column of partials
    const double *col = scratch + lane;
    int idp = lane, idq = w0 + lane;                   // column ids (>= n or lane >= w0: zero padding)
    if (lane >= w0) idp = idq = n;
    double xp[LA_JACOBI_ROWS], xq[LA_JACOBI_ROWS];
#pragma unroll
    for (int i = 0; i < LA_JACOBI_ROWS; ++i) {
      const int r = warp * LA_JACOBI_ROWS + i;
      xp[i] = (idp < n && r < n) ? W(r, idp) : 0.0;
      xq[i] = (idq < n && r < n) ? W(r, idq) : 0.0;
    }
    double ap, aq;
    bool done = false;
    for (;;) {
      // exact squared norms (once per sweep: bounds the drift of the closed-form fp32 updates)
      double sp = 0.0, sq = 0.0;
#pragma unroll
      for (int i = 0; i < LA_JACOBI_ROWS; ++i) { sp = fma(xp[i], xp[i], sp); sq = fma(xq[i], xq[i], sq); }
      mine[0] = sp;
      mine[256] = sq;
      la_named_barrier(nbar);
      ap = la_combine(col);
      aq = la_combine(col + 256);
      la_named_barrier(nbar);                          // the step buffers alias these partial sums
      if (done || sweeps == 40) break;
      float a = (float)ap, b = (float)aq;
      int big = 0;      // some pair was still correlated above the tolerance when it was visited in this sweep
#ifdef TCE_PROFILE
      float cmax2 = 0.f;
#endif
      int buf = 0;                                     // double buffered partials: one barrier per step
#ifdef JAC_PROF
      unsigned int jp[5] = {0, 0, 0, 0, 0}, jt = clock();
#endif
#pragma unroll 1
      for (int w = w0; w >= 1; w >>= 1) {
#pragma unroll 1
        for (int k = 0; k < w; ++k, buf ^= 256) {
          JP(4);
          double g0 = 0.0, g1 = 0.0;
#pragma unroll
          for (int i = 0; i < LA_JACOBI_ROWS; i += 2) { g0 = fma(xp[i], xq[i], g0); g1 = fma(xp[i + 1], xq[i + 1], g1); }
          mine[buf] = g0 + g1;
          JP(0);
          la_named_barrier(nbar);
          JP(1);
          const float g = (float)la_combine(col + buf);
#ifdef JAC_PROF
          if (g == 123.456f) jp[0]++;
#endif
          JP(2);
          double c = 1.0, sn = 0.0;
          float na = a, nb = b;
          const float g2 = g * g, ab = a * b;
          if (g2 > LA_JACOBI_TOL2 * ab) big = 1;
#ifdef TCE_PROFILE
          if (ab > 0.f) cmax2 = fmaxf(cmax2, g2 / ab);
#endif
          if (g2 > 1e-24f * ab) {
            // tan(theta) = 2g / (d + sgn(d) sqrt(d^2 + 4 g^2)), d = b - a: three MUFU ops, no IEEE fix-ups
            const float d = b - a, s4 = fmaf(d, d, 4.0f * g2);
            const float r = s4 * la_rsqrt_approx(s4);
            const float tf = 2.0f * g * la_rcp_approx(d + copysignf(r, d));
            const float c0 = la_rsqrt_approx(fmaf(tf, tf, 1.0f));
            const double t = (double)tf, hh = fma(t, t, 1.0);
            c = (double)c0;
            c = c * fma(-0.5 * hh, c * c, 1.5);        // one Newton step: c^2 (1 + t^2) = 1 to ~1e-14
            sn = c * t;
            const float sf = c0 * tf, cs2 = 2.0f * c0 * sf * g;   // |c x - s y|^2, |s x + c y|^2 (fp32)
            na = c0 * c0 * a + sf * sf * b - cs2;
            nb = sf * sf * a + c0 * c0 * b + cs2;
          }
          a = na;
#ifdef JAC_PROF
          if (sn == 123.456) jp[0]++;
#endif
          JP(3);
          // rotate, then ring-shift Q inside the segment (not after the last step of a level: Q then stays
          // shifted by w - 1, which is as good a start for the next level; a shift by 0 keeps the code branch-free)
          const int src = lane + (k + 1 < w ? 1 : 0);
#pragma unroll
          for (int i = 0; i < LA_JACOBI_ROWS; ++i) {
            const double np = fma(c, xp[i], -sn * xq[i]), nq = fma(sn, xp[i], c * xq[i]);
            xp[i] = np;
            xq[i] = __shfl_sync(0xffffffffu, nq, src, w);
          }
          b = __shfl_sync(0xffffffffu, nb, src, w);
        }
        idq = __shfl_sync(0xffffffffu, idq, lane + w - 1, w);
        if (w > 1) {                                   // trade column sets between the halves of the segment
          const int hw = w >> 1;
          const bool upper = (lane & hw) != 0;
#pragma unroll
          for (int i = 0; i < LA_JACOBI_ROWS; ++i) {
            const double got = __shfl_xor_sync(0xffffffffu, upper ? xp[i] : xq[i], hw);
            if (upper) xp[i] = got; else xq[i] = got;
          }
          const float fgot = __shfl_xor_sync(0xffffffffu, upper ? a : b, hw);
          const int igot = __shfl_xor_sync(0xffffffffu, upper ? idp : idq, hw);
          if (upper) { a = fgot; idp = igot; } else { b = fgot; idq = igot; }
        }
      }
#ifdef JAC_PROF
      if (threadIdx.x == 0 && blockIdx.x == 0) for (int i = 0; i < 5; ++i) g_jac_prof[i] = jp[i];
#endif
#ifdef TCE_PROFILE
      if (blockIdx.x == 0 && warp == 0 && sweeps < 8) {
        float m = cmax2;
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (lane == 0) g_jac_diag[sweeps] = m;
      }
#endif
      ++sweeps;
      la_named_barrier(nbar);                          // the last step's buffer is the next norm buffer
      // a sweep that only met cosines <= sqrt(LA_JACOBI_TOL2) is the last one (see the constant)
      done = !__any_sync(0xffffffffu, big);            // identical in every warp (same data, same code)
    }
#pragma unroll
    for (int i = 0; i < LA_JACOBI_ROWS; ++i) {
      const int r = warp * LA_JACOBI_ROWS + i;
      if (idp < n && r < n) W(r, idp) = xp[i];
      if (idq < n && r < n) W(r, idq) = xq[i];
    }
    if (warp == 0) {
      if (idp < n) lam[idp] = ap;
      if (idq < n) lam[idq] = aq;
    }
  } else {
    idle((int)threadIdx.x - nbar, (int)blockDim.x - nbar);
  }
  __syncthreads();
  return sweeps;
}

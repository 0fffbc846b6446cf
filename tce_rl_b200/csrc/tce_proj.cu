// (4a) Differentiable trust-region projections (KL / Frobenius / W2) and the Gaussian distances they use.
// Replaces the trust_region_projections layers instantiated at mprl/rl/projection/__init__.py:19-40 and
// called at mprl/rl/agent/temporal_correlated_agent.py:530-533,561-567 (math: SURVEY App. B / App. F;
// Otto et al., ICLR 2021), including the C++ cpp_projection (ITPAL) KL covariance projection, which the
// reference runs on the CPU through numpy.  One CTA per matrix; all matrices live in shared memory in fp64
// (bounds such as cov_bound = 5e-4 are differences of O(n) quantities -- fp32 cannot resolve them).
#include <cuda_pipeline.h>
#include <math.h>

#include "tce_bulk.cuh"
#include "tce_smem_la.cuh"

// Profiling scaffolding, compiled in with -DTCE_PROFILE only (TCE_PROFILE=1 python -m tce_rl_b200._build --force):
// SM-clock stamps of block 0 / thread 0 of the last KL forward [0..15] and covariance-space backward [16..31] kernel.
#ifdef TCE_PROFILE
__device__ long long g_kl_prof[32];
#define KL_STAMP(i) do { if (blockIdx.x == 0 && threadIdx.x == 0) g_kl_prof[i] = clock64(); } while (0)
#define KL_PROF_SET(i, v) do { if (blockIdx.x == 0 && threadIdx.x == 0) g_kl_prof[i] = (v); } while (0)
#else
#define KL_STAMP(i) do { } while (0)
#define KL_PROF_SET(i, v) do { } while (0)
#endif

namespace {

constexpr int PJ_THREADS = 512;
constexpr int KL_THREADS = 512;   // 128 registers per thread: the register-resident Jacobi
constexpr double LOG_2PI = 1.8378770664093453;
constexpr int KL_SC = 16;     // scalars saved per matrix by the KL projection: eta, active, kl0, fingerprint, alpha, ent_active,
                              // alpha^2, [7] trust-region shape part, [8] trust-region volume part (KL(new || out)),
                              // [9] entropy of the output, [10] / [11] shape / volume part of KL(new || old),
                              // [12] / [13] shape / volume part of KL(out || old), (2 spare)

__device__ inline int pad_even(int n) { return (n + 1) & ~1; }

// Stream `count` contiguous global elements through `sink(e, value)` with FOUR loads in flight per thread: a
// plain `for (e...) smem[f(e)] = src[e]` loop is not unrolled (runtime trip count, index arithmetic in the
// body) and pays one full memory latency per iteration -- 4 to 16 dependent round trips per matrix.
template <typename T, typename Sink>
__device__ __forceinline__ void batched_load(const T *__restrict__ src, int count, Sink sink) {
  const int step = (int)blockDim.x;
  for (int e0 = threadIdx.x; e0 < count; e0 += 4 * step) {
    T v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = (e0 + u * step < count) ? src[e0 + u * step] : T(0);
#pragma unroll
    for (int u = 0; u < 4; ++u) if (e0 + u * step < count) sink(e0 + u * step, v[u]);
  }
}

__device__ inline void zero_padding(Mat M, int n, int m) {           // row / column n of an odd-sized problem
  if (m > n) for (int t = threadIdx.x; t < m; t += blockDim.x) { M(n, t) = 0.0; M(t, n) = 0.0; }
}

// load the lower triangle of a dense fp32 [n,n] matrix into an fp64 shared buffer (m x LD, zero elsewhere)
__device__ inline void load_lower_d(Mat M, const float *__restrict__ src, int n, int m) {
  batched_load(src, n * n, [&](int e, float v) {
    const int i = e / n, j = e - i * n;
    M(i, j) = j <= i ? (double)v : 0.0;
  });
  zero_padding(M, n, m);
  __syncthreads();
}
__device__ inline void load_full_d(Mat M, const double *__restrict__ src, int n, int m) {
  batched_load(src, n * n, [&](int e, double v) {
    const int i = e / n, j = e - i * n;
    M(i, j) = v;
  });
  zero_padding(M, n, m);
  __syncthreads();
}
__device__ inline void store_lower_f(float *__restrict__ dst, Mat M, int n, double scale) {
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, j = e % n;
    dst[e] = j <= i ? (float)(scale * M(i, j)) : 0.f;
  }
}
__device__ inline double block_sum(double v, double *red) {   // red: >= 32 doubles of shared scratch
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
  __syncthreads();
  return t;
}

// grad_A (sym) of a Cholesky factor P with upstream G (lower): Sbar = sym(P^-T Phi(P^T G) P^-1)
// P in bP, G in bG; result in bM (full symmetric); bP and bG are destroyed.  P^-1 by recursive doubling and
// two GEMMs instead of two triangular solves with n right-hand sides.
__device__ inline void chol_backward(Mat bP, Mat bG, Mat bM, double *inv_diag, int n) {
  // M = Phi(P^T G)  (lower, halved diagonal, zero above)
  la_gemm(bM, bP.T(), bG, n, n, n, TRI_UPPER, TRI_LOWER, TRI_FULL, 1.0, 0.0);
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, j = e % n;
    if (j > i) bM(i, j) = 0.0; else if (i == j) bM(i, j) *= 0.5;
  }
  __syncthreads();
  la_tri_inverse(bP, bG, inv_diag, n);                                              // bG = P^-1 (G is consumed)
  la_gemm(bP, bM, bG, n, n, n, TRI_LOWER, TRI_LOWER, TRI_FULL, 1.0, 0.0);           // Phi P^-1 (P is consumed)
  la_gemm(bM, bG.T(), bP, n, n, n, TRI_UPPER, TRI_FULL, TRI_FULL, 1.0, 0.0);        // X = P^-T Phi P^-1
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, j = e % n;
    if (j < i) { const double s = 0.5 * (bM(i, j) + bM(j, i)); bG(i, j) = s; }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, j = e % n;
    if (j < i) { bM(i, j) = bG(i, j); bM(j, i) = bG(i, j); }
  }
  __syncthreads();
}

// =====================================================================================================
// Gaussian distances: per episode maha / trace / logdets / entropy, and their gradient w.r.t. (mean, L)
// =====================================================================================================
// fwd: out[b] = {maha, tr(Sigma_o^-1 Sigma), logdet Sigma, logdet Sigma_o, entropy(L)}
// bwd: given gout[b][5] -> grad_mean[b] (n), grad_L[b] (n x n lower)
//   d maha / d mean = 2 Sigma_o^-1 (mean - mean_o) ; d tr / d L = 2 Sigma_o^-1 L ; d logdet / d L_ii = 2 / L_ii ;
//   d entropy / d L_ii = 1 / L_ii
__global__ void __launch_bounds__(PJ_THREADS)
gauss_kl_kernel(const float *__restrict__ mean, const float *__restrict__ L, long long ldb_L,
                const float *__restrict__ mean_o, const float *__restrict__ L_o, long long ldb_Lo,
                double *__restrict__ out, const double *__restrict__ gout, float *__restrict__ grad_mean,
                float *__restrict__ grad_L, int n, int mean_only) {
  extern __shared__ double sd[];
  const int m = pad_even(n), LD = m + 1;
  Mat Lo{sd, LD, 1}, W{sd + m * LD, LD, 1};
  double *inv_diag = sd + 2 * m * LD, *red = inv_diag + LA_DINV_DOUBLES;
  const long long b = blockIdx.x;
  load_lower_d(Lo, L_o + b * ldb_Lo, n, m);
  // W = [L | diff] : n x (n+1)
  for (int e = threadIdx.x; e < m * m; e += blockDim.x) {
    const int i = e / m, j = e % m;
    W(i, j) = (i < n && j <= i && !mean_only) ? (double)L[b * ldb_L + (size_t)i * n + j] : 0.0;
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x) W(i, m) = (double)mean[b * n + i] - (double)mean_o[b * n + i];
  __syncthreads();
  double ld = 0.0, ldo = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) { ld += mean_only ? 0.0 : log(W(i, i)); ldo += log(Lo(i, i)); }
  ld = block_sum(ld, red);
  ldo = block_sum(ldo, red);
  la_diag_block_inverses(Lo, inv_diag, n);
  const bool backward = gout != nullptr;
  double g_tr = 0.0, g_ld = 0.0, g_ent = 0.0, g_maha = 0.0;
  if (backward) {
    g_maha = gout[b * 5 + 0]; g_tr = gout[b * 5 + 1]; g_ld = gout[b * 5 + 2]; g_ent = gout[b * 5 + 4];
    // dlogdet/dL_ii and dentropy/dL_ii need the ORIGINAL diagonal: stash it before the solves
    for (int i = threadIdx.x; i < n; i += blockDim.x) red[64 + i] = mean_only ? 1.0 : W(i, i);
    __syncthreads();
  }
  // mean column first (plain column), then the lower-triangular block
  la_trsm_lower(Lo, inv_diag, Mat{W.p + m, LD, 1}, n, 1, false);
  if (!mean_only) la_trsm_lower(Lo, inv_diag, W, n, n, true);
  if (!backward) {
    double fro = 0.0, maha = 0.0;
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) { const double v = W(e / n, e % n); fro = fma(v, v, fro); }
    for (int i = threadIdx.x; i < n; i += blockDim.x) { const double v = W(i, m); maha = fma(v, v, maha); }
    fro = block_sum(fro, red);
    maha = block_sum(maha, red);
    if (threadIdx.x == 0) {
      double *o = out + b * 5;
      o[0] = maha; o[1] = fro; o[2] = 2.0 * ld; o[3] = 2.0 * ldo; o[4] = 0.5 * n * (1.0 + LOG_2PI) + ld;
    }
    return;
  }
  // Sigma_o^-1 [L | diff] = L_o^-T W
  la_trsm_lower_t(Lo, inv_diag, Mat{W.p + m, LD, 1}, n, 1);
  if (!mean_only) la_trsm_lower_t(Lo, inv_diag, W, n, n);
  if (grad_mean)
    for (int i = threadIdx.x; i < n; i += blockDim.x) grad_mean[b * n + i] = (float)(2.0 * g_maha * W(i, m));
  if (grad_L && !mean_only) {
    float *gl = grad_L + (size_t)b * n * n;
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
      const int i = e / n, j = e % n;
      double v = 0.0;
      if (j <= i) v = 2.0 * g_tr * W(i, j);
      if (i == j) v += (2.0 * g_ld + g_ent) / red[64 + i];
      gl[e] = (float)v;
    }
  }
}

// =====================================================================================================
// Mahalanobis distance |L_o^-1 (mean - mean_o)|^2 and its gradient 2 g Sigma_o^-1 (mean - mean_o).
// Called several times per epoch on the whole batch: light kernel, one 128-thread CTA per episode, L_o staged
// as fp32 (odd row stride -> conflict-free column access), the two triangular vector solves run in fp64 on
// warp 0 (column oriented: after z_j is known every lane updates its rows).
// =====================================================================================================
__global__ void __launch_bounds__(128)
maha_kernel(const float *__restrict__ mean, const float *__restrict__ mean_o, const float *__restrict__ L_o,
            long long ldb_Lo, const double *__restrict__ gout, double *__restrict__ out,
            float *__restrict__ grad_mean, float *__restrict__ grad_L, int n) {
  extern __shared__ double smd[];
  const int LD = n | 1;
  double *bv = smd, *inv = smd + n, *zv = smd + 2 * n;
  float *sL = reinterpret_cast<float *>(smd + 3 * n);
  const long long b = blockIdx.x;
  const float *Lo = L_o + b * ldb_Lo;
  {
    const int warp = threadIdx.x >> 5, lane_ = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int i = warp; i < n; i += nw)                       // lower triangle only, no index divisions
      for (int j = lane_; j <= i; j += 32) sL[i * LD + j] = Lo[(size_t)i * n + j];
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    bv[i] = (double)mean[b * n + i] - (double)mean_o[b * n + i];
    inv[i] = 1.0 / (double)Lo[(size_t)i * n + i];
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    double maha = 0.0;
    for (int j = 0; j < n; ++j) {                       // z = L_o^-1 diff
      const double zj = bv[j] * inv[j];
      __syncwarp();
      for (int i = j + 1 + lane; i < n; i += 32) bv[i] = fma(-(double)sL[i * LD + j], zj, bv[i]);
      if (lane == 0) { bv[j] = zj; zv[j] = zj; }
      maha = fma(zj, zj, maha);
      __syncwarp();
    }
    if (out && lane == 0) out[b] = maha;
    if (gout) {
      const double g2 = 2.0 * gout[b];
      for (int i = n - 1; i >= 0; --i) {                  // u = L_o^-T z
        const double ui = bv[i] * inv[i];
        __syncwarp();
        for (int k = lane; k < i; k += 32) bv[k] = fma(-(double)sL[i * LD + k], ui, bv[k]);
        if (lane == 0) bv[i] = ui;
        __syncwarp();
      }
      if (grad_mean)
        for (int i = lane; i < n; i += 32) grad_mean[b * n + i] = (float)(g2 * bv[i]);
    }
  }
  if (!gout || !grad_L) return;
  // d maha / d L_o = -2 tril(u z^T)   (d(L^-1) = -L^-1 dL L^-1)
  __syncthreads();
  const double g2 = 2.0 * gout[b];
  float *gl = grad_L + (size_t)b * n * n;
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, j = e - i * n;
    gl[e] = j <= i ? (float)(-g2 * bv[i] * zv[j]) : 0.f;
  }
}

// n <= 64: ONE WARP per episode (four episodes per 128-thread CTA, every warp busy -- the kernel above keeps three of its
// four warps idle during the solves).  Lane l owns rows l and l + 32 of the system: right-hand side, solution and the
// inverted diagonal live in registers; per step the owner lane broadcasts z_j with a shuffle and every lane updates its
// two rows with the column entries it fetched from shared memory one step ahead: ~45 cycles per step instead of ~150.
//
// BULK (odd n, contiguous factors, B a multiple of MW_WARPS): the dense factors of the CTA's MW_WARPS episodes are one
// 16-byte-aligned block of 4 n^2 floats, requested by ONE bulk asynchronous copy (mbarrier completion) instead of
// ~2 n four-byte copies per lane; row stride n is odd, so the column accesses of the forward solve stay conflict free.
// One buffer per CTA, three CTAs per SM: the copies of two CTAs are in flight while the third solves.
constexpr int MW_WARPS = 4;
template <bool BULK>
__global__ void __launch_bounds__(MW_WARPS * 32)
maha_warp_kernel(const float *__restrict__ mean, const float *__restrict__ mean_o, const float *__restrict__ L_o,
                 long long ldb_Lo, const double *__restrict__ gout, double *__restrict__ out,
                 float *__restrict__ grad_mean, float *__restrict__ grad_L, int n, long long B) {
  extern __shared__ __align__(128) unsigned char mw_raw[];
  __shared__ __align__(8) uint64_t bar;
  const int LD = BULK ? n : (n | 1), warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t mat_bytes = BULK ? (size_t)n * n * sizeof(float) : (((size_t)n * LD * sizeof(float) + 15) & ~(size_t)15);
  const size_t per_warp = mat_bytes + (BULK ? 0 : 2 * 64 * sizeof(double));
  float *sL = reinterpret_cast<float *>(mw_raw + warp * per_warp);
  double *sz = reinterpret_cast<double *>(mw_raw + (BULK ? MW_WARPS * mat_bytes + warp * 2 * 64 * sizeof(double)
                                                         : warp * per_warp + mat_bytes));
  double *su = sz + 64;
  const unsigned full = 0xffffffffu;
  uint32_t parity = 0;
  if (BULK) {
    if (threadIdx.x == 0) mbar_init(&bar, 1);
    __syncthreads();
  }
  for (long long b = (long long)blockIdx.x * MW_WARPS + warp; b < B; b += (long long)gridDim.x * MW_WARPS) {
    const float *Lo = L_o + b * ldb_Lo;
    const int r0 = lane, r1 = lane + 32;
    double b0, b1;
    if (BULK) {                         // (B is a multiple of MW_WARPS: all warps of a CTA run the same iterations)
      __syncthreads();                  // the previous iteration's reads of the buffer are done
      if (threadIdx.x == 0) {
        const uint32_t bytes = (uint32_t)(MW_WARPS * mat_bytes);
        mbar_arrive_expect_tx(&bar, bytes);
        bulk_copy_g2s(mw_raw, L_o + (b - warp) * ldb_Lo, bytes, &bar);
      }
      b0 = r0 < n ? (double)mean[b * n + r0] - (double)mean_o[b * n + r0] : 0.0;
      b1 = r1 < n ? (double)mean[b * n + r1] - (double)mean_o[b * n + r1] : 0.0;
      mbar_wait(&bar, parity);
      parity ^= 1;
    } else {
      __syncwarp();
      // lower triangle, row by row (lanes = consecutive columns), as asynchronous global -> shared copies: all ~2 n
      // requests of a lane are in flight at once (staging through registers four rows at a time made this a chain of
      // n / 4 memory round trips, 3/4 of the kernel's time)
      for (int i = 0; i < n; ++i) {
        if (lane <= i) __pipeline_memcpy_async(sL + i * LD + lane, Lo + (size_t)i * n + lane, sizeof(float));
        if (lane + 32 <= i) __pipeline_memcpy_async(sL + i * LD + lane + 32, Lo + (size_t)i * n + lane + 32, sizeof(float));
      }
      __pipeline_commit();
      b0 = r0 < n ? (double)mean[b * n + r0] - (double)mean_o[b * n + r0] : 0.0;
      b1 = r1 < n ? (double)mean[b * n + r1] - (double)mean_o[b * n + r1] : 0.0;
      __pipeline_wait_prior(0);
      __syncwarp();
    }
    const double inv0 = r0 < n ? 1.0 / (double)sL[r0 * LD + r0] : 0.0, inv1 = r1 < n ? 1.0 / (double)sL[r1 * LD + r1] : 0.0;
    double z0 = 0.0, z1 = 0.0, maha = 0.0;
    // z = L_o^-1 diff (column oriented)
    float c0 = (r0 > 0 && r0 < n) ? sL[r0 * LD] : 0.f, c1 = r1 < n ? sL[r1 * LD] : 0.f;
    for (int j = 0; j < n; ++j) {
      const double mine = (j < 32 ? b0 * inv0 : b1 * inv1);
      const double zj = __shfl_sync(full, mine, j & 31);
      const float n0 = (j + 1 < n && r0 > j + 1 && r0 < n) ? sL[r0 * LD + j + 1] : 0.f;      // next column, fetched ahead
      const float n1 = (j + 1 < n && r1 > j + 1 && r1 < n) ? sL[r1 * LD + j + 1] : 0.f;
      if (r0 > j) b0 = fma(-(double)c0, zj, b0);
      if (r1 > j) b1 = fma(-(double)c1, zj, b1);
      if (lane == (j & 31)) { if (j < 32) z0 = zj; else z1 = zj; }
      maha = fma(zj, zj, maha);
      c0 = n0; c1 = n1;
    }
    if (out && lane == 0) out[b] = maha;
    if (!gout) continue;
    const double g2 = 2.0 * gout[b];
    // u = L_o^-T z: after u_i is known every lane k < i subtracts L_o[i][k] u_i from its rows (row i of L: consecutive lanes)
    b0 = z0; b1 = z1;
    for (int i = n - 1; i >= 0; --i) {
      const double mine = (i < 32 ? b0 * inv0 : b1 * inv1);
      const double ui = __shfl_sync(full, mine, i & 31);
      const float l0 = r0 < i ? sL[i * LD + r0] : 0.f, l1 = r1 < i ? sL[i * LD + r1] : 0.f;
      if (lane == (i & 31)) { if (i < 32) b0 = ui; else b1 = ui; }
      if (r0 < i) b0 = fma(-(double)l0, ui, b0);
      if (r1 < i) b1 = fma(-(double)l1, ui, b1);
    }
    if (grad_mean) {
      if (r0 < n) grad_mean[b * n + r0] = (float)(g2 * b0);
      if (r1 < n) grad_mean[b * n + r1] = (float)(g2 * b1);
    }
    if (grad_L) {                       // d maha / d L_o = -2 tril(u z^T)   (d(L^-1) = -L^-1 dL L^-1)
      if (r0 < n) { sz[r0] = z0; su[r0] = b0; }
      if (r1 < n) { sz[r1] = z1; su[r1] = b1; }
      __syncwarp();
      float *gl = grad_L + (size_t)b * n * n;
      for (int i = 0; i < n; ++i) {
        const double ui = -g2 * su[i];
        for (int j = lane; j < n; j += 32) gl[(size_t)i * n + j] = j <= i ? (float)(ui * sz[j]) : 0.f;
      }
    }
  }
}

// Shared-covariance variants (non-contextual policy: every episode has the same L_o).  L_o^-1 is formed once
// (tri_inverse_kernel, fp64) and the two triangular solves per episode become dense matrix-vector products
// without a dependent chain: one warp per episode, Linv staged once per CTA (row stride n | 1).
__global__ void __launch_bounds__(256)
tri_inverse_kernel(const float *__restrict__ L, long long ldb, double *__restrict__ Linv, int n) {
  extern __shared__ double sd[];
  const int m = pad_even(n), LD = m + 1, MS = m * LD;
  Mat A{sd, LD, 1}, X{sd + MS, LD, 1};
  double *dinv = sd + 2 * MS;
  const long long b = blockIdx.x;
  load_lower_d(A, L + b * ldb, n, m);
  la_tri_inverse(A, X, dinv, n);
  double *out = Linv + (size_t)b * n * n;
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, j = e - i * n;
    out[e] = j <= i ? X(i, j) : 0.0;
  }
}

__global__ void __launch_bounds__(256)
maha_shared_kernel(const float *__restrict__ mean, const float *__restrict__ mean_o, const double *__restrict__ Linv,
                   const double *__restrict__ gout, double *__restrict__ out, float *__restrict__ grad_mean,
                   long long B, int n) {
  extern __shared__ double smd[];
  const int LD = n | 1, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  double *sA = smd, *dv = smd + (size_t)n * LD + (size_t)warp * 2 * n, *zv = dv + n;
  batched_load(Linv, n * n, [&](int e, double v) {
    const int i = e / n, j = e - i * n;
    sA[i * LD + j] = v;
  });
  __syncthreads();
  for (long long b = (long long)blockIdx.x * nw + warp; b < B; b += (long long)gridDim.x * nw) {
#pragma unroll 1
    for (int i = lane; i < n; i += 32) dv[i] = (double)mean[b * n + i] - (double)mean_o[b * n + i];
    __syncwarp();
    // compact loops (`#pragma unroll 1`): the kernel is a chain of memory latencies (Linv staging, the episode's
    // means, the result), not pipe bound; unrolling only grew the code
    double maha = 0.0;
#pragma unroll 1
    for (int i = lane; i < n; i += 32) {                 // z = Linv d (rows of different lanes: stride LD is odd)
      double z0 = 0.0, z1 = 0.0, z2 = 0.0, z3 = 0.0;      // four chains: eight shared-memory loads in flight
      const double *row = sA + i * LD;
      int j = 0;
#pragma unroll 1
      for (; j + 3 <= i; j += 4) {
        z0 = fma(row[j], dv[j], z0); z1 = fma(row[j + 1], dv[j + 1], z1);
        z2 = fma(row[j + 2], dv[j + 2], z2); z3 = fma(row[j + 3], dv[j + 3], z3);
      }
      for (; j <= i; ++j) z0 = fma(row[j], dv[j], z0);
      const double z = (z0 + z1) + (z2 + z3);
      zv[i] = z;
      maha = fma(z, z, maha);
    }
    maha = warp_sum(maha);
    if (out && lane == 0) out[b] = maha;
    if (grad_mean) {                                     // grad = 2 g Linv^T z (columns: consecutive lanes)
      __syncwarp();
      const double g2 = gout ? 2.0 * gout[b] : 2.0;      // gout == NULL: d maha / d mean, saved for the backward
#pragma unroll 1
      for (int j = lane; j < n; j += 32) {
        double u0 = 0.0, u1 = 0.0, u2 = 0.0, u3 = 0.0;
        const double *colp = sA + j;
        int i = j;
#pragma unroll 1
        for (; i + 3 < n; i += 4) {
          u0 = fma(colp[i * LD], zv[i], u0); u1 = fma(colp[(i + 1) * LD], zv[i + 1], u1);
          u2 = fma(colp[(i + 2) * LD], zv[i + 2], u2); u3 = fma(colp[(i + 3) * LD], zv[i + 3], u3);
        }
        for (; i < n; ++i) u0 = fma(colp[i * LD], zv[i], u0);
        u0 += u2; u1 += u3;
        grad_mean[b * n + j] = (float)(g2 * (u0 + u1));
      }
    }
    __syncwarp();
  }
}


// =====================================================================================================
// mean projection (closed form) -- elementwise, one warp per episode
// =====================================================================================================
__global__ void proj_mean_fwd_kernel(const float *__restrict__ mean, const float *__restrict__ mean_o,
                                     const double *__restrict__ mean_part, double eps, float *__restrict__ out,
                                     long long B, int n) {
  const long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  const double mp = mean_part[b];
  const bool active = mp > eps;
  const double om = active ? fabs(sqrt(mp / eps) - 1.0) : 0.0;
  const double a = 1.0 / (1.0 + om + 1e-16);
  for (int i = lane; i < n; i += 32) {
    const double x = mean[b * n + i];
    out[b * n + i] = active ? (float)((x + om * (double)mean_o[b * n + i]) * a) : (float)x;
  }
}
// g [B,n] -> grad_mean [B,n], grad_mean_part [B]
__global__ void proj_mean_bwd_kernel(const float *__restrict__ mean, const float *__restrict__ mean_o,
                                     const double *__restrict__ mean_part, double eps, const float *__restrict__ g,
                                     float *__restrict__ grad_mean, double *__restrict__ grad_part, long long B, int n) {
  const long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  const double mp = mean_part[b];
  const bool active = mp > eps;
  if (!active) {
    for (int i = lane; i < n; i += 32) grad_mean[b * n + i] = g[b * n + i];
    if (lane == 0) grad_part[b] = 0.0;
    return;
  }
  const double om = sqrt(mp / eps) - 1.0;       // > 0 when active
  const double a = 1.0 / (1.0 + om + 1e-16);
  double dot = 0.0;
  for (int i = lane; i < n; i += 32) {
    const double x = mean[b * n + i], xo = mean_o[b * n + i], gi = g[b * n + i];
    const double proj = (x + om * xo) * a;
    dot = fma(gi, a * (xo - proj), dot);
    grad_mean[b * n + i] = (float)(gi * a);
  }
  dot = warp_sum(dot);
  if (lane == 0) grad_part[b] = dot / (2.0 * sqrt(mp * eps));
}

// =====================================================================================================
// entropy projection: L <- L * exp((beta - H(L)) / n) where H(L) < beta (or always, equality variant)
// =====================================================================================================
__global__ void __launch_bounds__(256)
proj_entropy_kernel(const float *__restrict__ L, const double *__restrict__ beta, long long ldb_beta, int equality,
                    const float *__restrict__ gout, float *__restrict__ out, double *__restrict__ ent_out, int n) {
  __shared__ double red[40];
  const long long b = blockIdx.x;
  const float *Lb = L + (size_t)b * n * n;
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += log((double)Lb[(size_t)i * n + i]);
  s = block_sum(s, red);
  const double H = 0.5 * n * (1.0 + LOG_2PI) + s, bt = beta[b * ldb_beta];
  const bool active = equality || (H < bt);
  const double alpha = active ? exp((bt - H) / n) : 1.0;
  float *ob = out + (size_t)b * n * n;
  if (!gout) {                                   // forward
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) ob[e] = (e % n <= e / n) ? (float)(alpha * Lb[e]) : 0.f;
    if (ent_out && threadIdx.x == 0) ent_out[b] = H;
    return;
  }
  // backward: out = alpha(L) L ; d alpha / d L_ii = -alpha / (n L_ii)
  const float *gb = gout + (size_t)b * n * n;
  double dot = 0.0;
  if (active)
    for (int e = threadIdx.x; e < n * n; e += blockDim.x)
      if (e % n <= e / n) dot = fma((double)gb[e], (double)Lb[e], dot);
  dot = block_sum(dot, red);
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, j = e % n;
    double v = 0.0;
    if (j <= i) v = alpha * gb[e];
    if (i == j && active) v -= dot * alpha / (n * (double)Lb[e]);
    ob[e] = (float)v;
  }
}

// =====================================================================================================
// KL covariance projection (exact dual solve on the generalised eigenvalues, SURVEY App. B.4)
// =====================================================================================================
// Warp-cooperative evaluation of KL_cov(eta) = 1/2 sum_i g((lam_i + eta) / (1 + eta)), g(r) = 1/r - 1 + ln r,
// and of d/d eta (every lane of the calling warp participates).
__device__ inline double kl_of_eta(const double *lam, int n, double eta, double *dfd_eta) {
  // with s = lam + eta, r = s / (1 + eta):  g(r) = (1+eta)/s - 1 + ln s - ln(1+eta),
  // d g / d eta = -(lam - 1)^2 / ((1+eta) s^2)  -- one division and one logarithm per eigenvalue
  double f = 0.0, df = 0.0;
  const double ope = 1.0 + eta, iope = 1.0 / ope, lope = log(ope);
  for (int i = threadIdx.x & 31; i < n; i += 32) {
    const double s = lam[i] + eta, is = 1.0 / s, d = lam[i] - 1.0;
    f += fma(ope, is, -1.0) + (log(s) - lope);
    df -= d * d * is * is * iope;
  }
  f = warp_sum(f); df = warp_sum(df);
  if (dfd_eta) *dfd_eta = 0.5 * df;
  return 0.5 * f;
}

// Root of KL_cov(eta) = eps (monotone decreasing in eta).  All warps of the CTA evaluate candidates in
// parallel (two grid-refinement rounds), warp 0 polishes with safeguarded Newton steps.  cand: >= 36 doubles.
// eta0 > 0: the root found for the previous L~ of the same update (warm start) -- Newton from there first and
// fall back to the bracketing search only if it leaves the positive axis or does not settle in 6 steps.
__device__ inline double kl_solve_eta(const double *lam, int n, double eps, double *cand, double eta0) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = (int)(blockDim.x >> 5);
  if (eta0 > 0.0) {                                   // uniform over the CTA
    if (warp == 0) {
      double eta = eta0;
      bool ok = false;
      for (int it = 0; it < 6 && !ok; ++it) {       // quadratic: 2-3 steps from the previous epoch's root
        double df;
        const double f = kl_of_eta(lam, n, eta, &df) - eps;
        const double nxt = eta - f / df;
        if (!(df < 0.0) || !(nxt > 0.0) || !(nxt < 1e300)) break;
        ok = fabs(nxt - eta) <= 1e-9 * fmax(1.0, fabs(eta));      // error after this step ~ (1e-9)^2: rounding level
        eta = nxt;
      }
      if (lane == 0) { cand[34] = ok ? 1.0 : 0.0; cand[35] = eta; }
    }
    __syncthreads();
    const bool ok = cand[34] != 0.0;
    const double eta = cand[35];
    __syncthreads();
    if (ok) return eta;
  }
  // round 1: geometric grid eta_w = 2^(w - 10), w = 0..31  (1e-3 .. 2.1e6); a root above the grid is bracketed by
  // doubling from there (rare: the new standard deviations ~100x below the old ones), then two refinement rounds
  double lo = 0.0, hi = ldexp(1.0, 32 - 10);
  for (int round = 0; round < 3; ++round) {
    for (int w = warp; w < 32; w += nwarp) {
      const double e = round == 0 ? ldexp(1.0, w - 10) : lo + (hi - lo) * (double)(w + 1) / 33.0;
      const double f = kl_of_eta(lam, n, e, nullptr);
      if (lane == 0) cand[w] = f;
    }
    __syncthreads();
    if (threadIdx.x == 0) {            // f decreasing: last candidate with f > eps brackets from below
      double nlo = lo, nhi = hi;
      for (int w = 0; w < 32; ++w) {
        const double e = round == 0 ? ldexp(1.0, w - 10) : lo + (hi - lo) * (double)(w + 1) / 33.0;
        if (cand[w] > eps) nlo = e; else { nhi = e; break; }
      }
      cand[32] = nlo; cand[33] = nhi;
    }
    __syncthreads();
    if (round == 0 && cand[31] > eps) {      // f(2^21) > eps (uniform over the CTA): hi = 2^22 is not known to bound
      if (warp == 0) {
        double l = ldexp(1.0, 21), h = 2.0 * l;
        for (int it = 0; it < 1000 && kl_of_eta(lam, n, h, nullptr) > eps; ++it) { l = h; h *= 2.0; }
        if (lane == 0) { cand[32] = l; cand[33] = h; }
      }
      __syncthreads();
    }
    lo = cand[32]; hi = cand[33];
    __syncthreads();
  }
  if (warp == 0) {
    double eta = 0.5 * (lo + hi);
    for (int it = 0; it < 5; ++it) {              // bracket is ~1e-3 wide: Newton converges in 3-4 steps
      double df;
      const double f = kl_of_eta(lam, n, eta, &df) - eps;
      if (f > 0.0) lo = eta; else hi = eta;
      double nxt = (df != 0.0) ? eta - f / df : 0.5 * (lo + hi);
      if (!(nxt > lo && nxt < hi)) nxt = 0.5 * (lo + hi);
      const bool done = fabs(nxt - eta) <= 4e-16 * fmax(1.0, fabs(eta)) || hi - lo <= 4e-16 * fmax(1.0, hi);
      eta = nxt;
      if (done) break;
    }
    if (lane == 0) cand[32] = eta;
  }
  __syncthreads();
  const double eta = cand[32];
  __syncthreads();
  return eta;
}

// -----------------------------------------------------------------------------------------------------
// Diagonal KL projection (std_only policies).  With lam_i = (s_old,i / s_i)^2 the dual is the same scalar function
// kl_of_eta, and the projected variance is elementwise: s_old,i^2 (1 + eta) / (lam_i + eta)  -- no eigen-solve, so
// equal standard deviations (a fresh policy) are not a degenerate case.  One warp per episode.
// -----------------------------------------------------------------------------------------------------
constexpr int KD_WARPS = 4;
constexpr int KD_SC = 4;      // state per episode: eta, KL step active, alpha, entropy control active

// Root of KL_cov(eta) = eps for one warp (kl_of_eta hands every lane the same value, so the control flow is
// warp-uniform): bracket by doubling, then Newton steps safeguarded by bisection.
__device__ inline double kl_solve_eta_warp(const double *lam, int n, double eps) {
  double lo = 0.0, hi = 1.0;
  for (int it = 0; it < 1000 && kl_of_eta(lam, n, hi, nullptr) > eps; ++it) { lo = hi; hi *= 2.0; }
  double eta = 0.5 * (lo + hi);
  for (int it = 0; it < 200; ++it) {
    double df;
    const double f = kl_of_eta(lam, n, eta, &df) - eps;
    if (f > 0.0) lo = eta; else hi = eta;
    double nxt = (df < 0.0) ? eta - f / df : 0.5 * (lo + hi);
    if (!(nxt > lo && nxt < hi)) nxt = 0.5 * (lo + hi);
    const bool done = fabs(nxt - eta) <= 4e-16 * fmax(1.0, eta) || hi - lo <= 4e-16 * fmax(1.0, hi);
    eta = nxt;
    if (done) break;
  }
  return eta;
}

// Forward (gout == NULL): out = alpha * s_proj and the state {eta, active, alpha, entropy active}.
// Backward: out = d loss / d s from gout = d loss / d out; implicit differentiation of eta,
// d eta / d lam_j = -(d KL / d lam_j) / (d KL / d eta), and the alpha term of the entropy control.
__global__ void __launch_bounds__(KD_WARPS * 32)
proj_kl_diag_kernel(const float *__restrict__ s, long long ldb_s, long long inc_s, const float *__restrict__ so,
                    long long ldb_so, long long inc_so, double eps, const double *__restrict__ beta, long long ldb_beta,
                    int equality, const float *__restrict__ gout, long long ldb_g, long long inc_g,
                    float *__restrict__ out, long long ldb_o, long long inc_o, double *__restrict__ state,
                    int32_t *__restrict__ info, long long B, int n) {
  extern __shared__ double kd_lam[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long b = (long long)blockIdx.x * KD_WARPS + warp;
  if (b >= B) return;                                   // warp-uniform, no CTA barrier below
  double *lam = kd_lam + warp * n;
  const float *sb = s + b * ldb_s, *sob = so + b * ldb_so;
  int bad = 0;
  for (int i = lane; i < n; i += 32) {
    const double v = sb[i * inc_s], vo = sob[i * inc_so];
    if (!(v > 0.0) || !(vo > 0.0) || !(v < INFINITY) || !(vo < INFINITY)) bad = 1;
    const double r = vo / v;
    lam[i] = r * r;
  }
  bad = __any_sync(0xffffffffu, bad);
  __syncwarp();
  double *sc = state + b * KD_SC;
  float *ob = out + b * ldb_o;
  if (!gout) {
    const bool active = !bad && kl_of_eta(lam, n, 0.0, nullptr) > eps;
    const double eta = active ? kl_solve_eta_warp(lam, n, eps) : 0.0;
    double ls = 0.0;
    for (int i = lane; i < n; i += 32)
      ls += active ? log((double)sob[i * inc_so]) + 0.5 * log((1.0 + eta) / (lam[i] + eta)) : log((double)sb[i * inc_s]);
    ls = warp_sum(ls);
    const double H = 0.5 * n * (1.0 + LOG_2PI) + ls;
    const double bt = beta ? beta[b * ldb_beta] : 0.0;
    const bool ent = beta != nullptr && (equality || H < bt);
    const double alpha = ent ? exp((bt - H) / n) : 1.0;
    for (int i = lane; i < n; i += 32) {
      const double p = active ? (double)sob[i * inc_so] * sqrt((1.0 + eta) / (lam[i] + eta)) : (double)sb[i * inc_s];
      ob[i * inc_o] = (float)(alpha * p);
    }
    if (lane == 0) {
      sc[0] = eta; sc[1] = active ? 1.0 : 0.0; sc[2] = alpha; sc[3] = ent ? 1.0 : 0.0;
      if (info) info[b] = bad;
    }
    return;
  }
  const double eta = sc[0], alpha = sc[2];
  const bool active = sc[1] != 0.0, ent = sc[3] != 0.0;
  const float *gb = gout + b * ldb_g;
  // entropy control: out = alpha(p) p with d alpha / d p_j = -alpha / (n p_j)
  double dot = 0.0;
  for (int i = lane; i < n; i += 32) {
    const double p = active ? (double)sob[i * inc_so] * sqrt((1.0 + eta) / (lam[i] + eta)) : (double)sb[i * inc_s];
    dot = fma((double)gb[i * inc_g], p, dot);
  }
  dot = ent ? warp_sum(dot) : 0.0;
  if (!active) {
    for (int i = lane; i < n; i += 32) {
      const double p = sb[i * inc_s];
      ob[i * inc_o] = (float)(alpha * gb[i * inc_g] - alpha * dot / (n * p));
    }
    return;
  }
  // p_i = s_old,i sqrt((1+eta)/(lam_i+eta)):  d p_i / d lam_i = -p_i / (2 (lam_i+eta)),
  // d p_i / d eta = p_i (lam_i - 1) / (2 (1+eta) (lam_i+eta));  d KL / d lam_j = (lam_j - 1) / (2 (lam_j+eta)^2)
  double geta = 0.0;
  for (int i = lane; i < n; i += 32) {
    const double l = lam[i], p = (double)sob[i * inc_so] * sqrt((1.0 + eta) / (l + eta));
    const double gp = alpha * gb[i * inc_g] - alpha * dot / (n * p);
    geta += gp * p * (l - 1.0) / (2.0 * (1.0 + eta) * (l + eta));
  }
  geta = warp_sum(geta);
  double dfde;
  kl_of_eta(lam, n, eta, &dfde);
  for (int i = lane; i < n; i += 32) {
    const double l = lam[i], p = (double)sob[i * inc_so] * sqrt((1.0 + eta) / (l + eta));
    const double gp = alpha * gb[i * inc_g] - alpha * dot / (n * p);
    const double glam = -gp * p / (2.0 * (l + eta)) - geta * (l - 1.0) / (2.0 * (l + eta) * (l + eta) * dfde);
    ob[i * inc_o] = (float)(glam * (-2.0 * l / (double)sb[i * inc_s]));     // d lam_i / d s_i = -2 lam_i / s_i
  }
}

// Forward.  With W = Lt^-1 Lo, one-sided Jacobi rotates the columns of W into U~ = W Q (orthogonal columns,
// |U~_j|^2 = lam_j = eigenvalues of W^T W); then M := Lo Q = Lt U~ and
//   Sigma_proj = Lo Q diag((1+eta)/(lam+eta)) Q^T Lo^T = M D M^T ,   proj_L = chol(Sigma_proj).
// `save` = { M, U~, Lt^-1, Sigma_proj [n,n each], lam [n], {eta, active, kl0, fingerprint(Lo), alpha, ent_active, alpha^2, -} }:
// state for the backward AND a
// warm start for the next call with the same Lo (the 50 epochs of one update_policy): starting Jacobi from
// Lt^-1 M_prev = W Q_prev is an orthogonal change of basis of the same problem, so 2-3 sweeps suffice.
// sum NV values over the CTA at once (scratch: >= 32 * NV + NV doubles); every thread receives all sums in v[]
template <int NV>
__device__ inline void block_sum_n(double (&v)[NV], double *scratch) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (int)(blockDim.x >> 5);
#pragma unroll
  for (int k = 0; k < NV; ++k) v[k] = warp_sum(v[k]);
  __syncthreads();
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < NV; ++k) scratch[warp * NV + k] = v[k];
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double t = 0.0;
    for (int w = 0; w < nw; ++w) t += scratch[w * NV + threadIdx.x];
    scratch[32 * NV + threadIdx.x] = t;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < NV; ++k) v[k] = scratch[32 * NV + k];
  __syncthreads();
}

// dense row-major [n, n] global <- shared matrix, one row per warp pass (no index divisions, coalesced rows)
__device__ __forceinline__ void store_full_rows(double *__restrict__ dst, Mat M, int n, int t, int nt) {
  const int w = t >> 5, lane = t & 31, nw = nt >> 5;
  for (int i = w; i < n; i += nw)
    for (int j = lane; j < n; j += 32) dst[(size_t)i * n + j] = M(i, j);
}

__global__ void __launch_bounds__(KL_THREADS)
proj_kl_cov_fwd_kernel(const float *__restrict__ L, const float *__restrict__ L_o, double eps_cov,
                       float *__restrict__ proj_L, double *__restrict__ save_M, double *__restrict__ save_U,
                       double *__restrict__ save_Li, double *__restrict__ save_Sig, double *__restrict__ save_lam,
                       double *__restrict__ save_sc, int32_t *__restrict__ info, int n, int warm_start,
                       const double *__restrict__ beta,
                       long long ldb_beta, int entropy_eq, float *__restrict__ out_L, int split,
                       const float *__restrict__ vec, long long ldb_vec, float min_std, float *__restrict__ L_built,
                       int compact) {
  extern __shared__ double sd[];
  const int m = pad_even(n), LD = m + 1, MS = m * LD;
  // Four buffers: b0 = Lt throughout, b3 = Lo -> W -> U~.  `compact` (batches: two CTAs of 256 threads per SM instead of
  // one of 512, so that one matrix's Jacobi phase -- four busy warps -- runs beside another's GEMMs): THREE buffers;
  // Lo is staged where Lt^-1 goes next, W = Lt^-1 (basis) overwrites Lt, and the warps that idle during the Jacobi
  // iteration fetch Lt again into the buffer the start basis has left (bL: where Lt is once U~ exists).
  Mat b0{sd, LD, 1}, b1{sd + MS, LD, 1}, b2{sd + 2 * MS, LD, 1}, b3{compact ? sd : sd + 3 * MS, LD, 1};
  Mat bLo = compact ? b2 : b3, bL = compact ? b1 : b0, bS = compact ? b0 : b1;       // bS: Sigma of an identity step
  double *dinv = sd + (compact ? 3 : 4) * MS, *lam = dinv + LA_DINV_DOUBLES, *nrm = lam + m,
         *red = nrm + LA_JACOBI_SCRATCH;                                                               // red: >= 48
  __shared__ int s_bad;
  const long long b = blockIdx.x;
  const size_t off = (size_t)b * n * n;
  // `vec` != NULL: the policy head is fused in -- Lt is built from the covariance vector (softplus(v_i) + min_std on the
  // diagonal, strictly-lower entries row-major behind the first n: abstract_policy.py:166-187) and also written to
  // L_built for the kernels that read the factor later.
  const float *Lt = vec ? L_built + off : L + off, *Lo = L_o + off;
  const float *vb = vec ? vec + b * ldb_vec : nullptr;
  if (threadIdx.x == 0) s_bad = 0;
  KL_STAMP(0);
  // All three input matrices are requested before anything is consumed (EIGHT global loads in flight per thread: the
  // kernel starts with cold caches and every dependent round trip costs ~2 k cycles): Lt -> b0, Lo -> b3 (with its
  // fingerprint: position weighted sum, deterministic order; guards the warm start), and -- speculatively -- the
  // previous call's M = Lo Q_prev -> b1.
  double fp = 0.0;
  {
    const int total = n * n, step = (int)blockDim.x;
    for (int e0 = threadIdx.x; e0 < total; e0 += 4 * step) {
      float vt[4], vo[4];
      double vm[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = e0 + u * step;
        if (vb) {
          const int i = e / n, j = e - i * n;
          vt[u] = (e < total && j <= i) ? (j == i ? vb[i] : vb[n + i * (i - 1) / 2 + j]) : 0.f;
        } else {
          vt[u] = e < total ? Lt[e] : 0.f;
        }
        vo[u] = e < total ? Lo[e] : 0.f;
        vm[u] = (e < total && warm_start) ? save_M[off + e] : 0.0;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = e0 + u * step;
        if (e < total) {
          const int i = e / n, j = e - i * n;
          if (vb) {
            if (i == j) vt[u] = (vt[u] > 20.f ? vt[u] : log1pf(expf(vt[u]))) + min_std;     // head_fwd_kernel's softplus
            L_built[off + e] = j <= i ? vt[u] : 0.f;
          }
          b0(i, j) = j <= i ? (double)vt[u] : 0.0;
          bLo(i, j) = j <= i ? (double)vo[u] : 0.0;
          b1(i, j) = vm[u];
          fp = fma((double)(e % 251 + 1), (double)vo[u], fp);
        }
      }
    }
    zero_padding(b0, n, m);
    zero_padding(b1, n, m);
    zero_padding(bLo, n, m);
  }
  fp = block_sum(fp, red);
  const bool warm = warm_start && save_sc[b * KL_SC + 3] == fp;
  if (!warm) {                                                                      // cold: b1 = Lo (lower)
    for (int e = threadIdx.x; e < m * m; e += blockDim.x) b1(e / m, e % m) = bLo(e / m, e % m);
    __syncthreads();
  }
  KL_STAMP(1);
  la_tri_inverse(b0, b2, dinv, n);                                                 // Lt^-1 (kept for the backward)
  KL_STAMP(10);
  zero_padding(b3, n, m);
  la_gemm(b3, b2, b1, n, n, n, TRI_LOWER, warm ? TRI_FULL : TRI_LOWER, TRI_FULL, 1.0, 0.0);   // W (or W Q_prev)
  KL_STAMP(11);
  KL_STAMP(2);
  // the warps that hold no rows of the register-resident iteration write Lt^-1 to the state meanwhile
  auto refetch_Lt = [&](int t, int nt) {              // compact: Lt (fp32 in HBM / L2; exact in fp64) -> bL, padding zeroed
    for (int e = t; e < m * m; e += nt) {
      const int i = e / m, j = e - i * m;
      bL(i, j) = (i < n && j <= i) ? (double)Lt[(size_t)i * n + j] : 0.0;
    }
  };
  const int sweeps = la_jacobi_onesided(b3, lam, nrm, n, [&](int t, int nt) {
    if (nt >= 32) {
      store_full_rows(save_Li + off, b2, n, t, nt);
      if (compact) refetch_Lt(t, nt);
    }
  });                                                                               // b3 = U~
  if ((int)blockDim.x - 32 * ((n + LA_JACOBI_ROWS - 1) / LA_JACOBI_ROWS) < 32) {    // (no idle warp: all of them do it now)
    store_full_rows(save_Li + off, b2, n, threadIdx.x, blockDim.x);
    if (compact) refetch_Lt(threadIdx.x, blockDim.x);
    __syncthreads();
  }
  KL_STAMP(3);
  const double kl0 = [&] {
    double v = 0.0;
    if (threadIdx.x < 32) v = kl_of_eta(lam, n, 0.0, nullptr);
    if (threadIdx.x == 0) red[40] = v;
    __syncthreads();
    v = red[40];
    __syncthreads();
    return v;
  }();
  const bool active = kl0 > eps_cov;
  const double eta = active ? kl_solve_eta(lam, n, eps_cov, red, warm && save_sc[b * KL_SC + 1] != 0.0 ? save_sc[b * KL_SC + 0] : 0.0) : 0.0;
  KL_STAMP(4);
  la_gemm(b2, bL, b3, n, n, n, TRI_LOWER, TRI_FULL, TRI_FULL, 1.0, 0.0);           // M = Lt U~
  if (threadIdx.x == 0) {
    save_sc[b * KL_SC + 0] = eta; save_sc[b * KL_SC + 1] = active ? 1.0 : 0.0; save_sc[b * KL_SC + 2] = kl0; save_sc[b * KL_SC + 3] = fp;
    save_sc[b * KL_SC + 4] = 1.0; save_sc[b * KL_SC + 5] = 0.0;    // alpha, ent_active, alpha^2: overwritten by the fused
    save_sc[b * KL_SC + 6] = 1.0;                                  // entropy control
    KL_PROF_SET(15, sweeps);
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    save_lam[b * n + i] = lam[i];
    nrm[i] = active ? sqrt((1.0 + eta) / (lam[i] + eta)) : 1.0;                     // sqrt(D_ii): column scale of M
  }
  store_full_rows(save_M + off, b2, n, threadIdx.x, blockDim.x);
  store_full_rows(save_U + off, b3, n, threadIdx.x, blockDim.x);                   // U~ = Lt^-1 M for the backward
  __syncthreads();
  KL_STAMP(5);
  float *out = proj_L + off;
  // Everything that is a sum over the eigenvalues, in ONE reduction:
  //  * fused entropy control (optional, `beta` != NULL): out_L = alpha * proj_L with alpha = exp((beta - H(proj_L)) / n)
  //    where H < beta (or always: equality variant), as proj_entropy_kernel.  `half_logdet(i)`: the i-th term of
  //    1/2 logdet of the projected covariance (log of the Cholesky diagonal, or its closed form 1/2 logdet(Sigma_o) +
  //    1/2 sum log((1+eta)/(lam+eta)) when the factor is not formed here: `split`)
  //  * covariance part of KL(N(., Sigma) || N(., Sigma_out)), Sigma = Lt Lt^T the UNPROJECTED covariance and
  //    Sigma_out = alpha^2 Sigma_proj the layer's output -- the covariance term of the trust-region regression loss
  //    (get_trust_region_loss, temporal_correlated_agent.py:561-567) -- in closed form on the eigen-system:
  //      tr(Sigma_out^-1 Sigma) = alpha^-2 sum_i 1 / (D_ii lam_i),  logdet Sigma_out - logdet Sigma = 2 n ln alpha + sum_i ln(D_ii lam_i)
  //    with D_ii = (1 + eta) / (lam_i + eta)  (identity step: D_ii lam_i = 1).  -> save_sc[7] (1/2 (tr - n)), save_sc[8]
  //  * the logging decompositions of temporal_correlated_agent.py:641-686 in the same closed form (no extra kernels):
  //      KL(new || old):  tr(Sigma_o^-1 Sigma) = sum_i 1 / lam_i,  logdet Sigma_o - logdet Sigma = sum_i ln lam_i
  //      KL(out || old):  tr(Sigma_o^-1 Sigma_out) = alpha^2 sum_i D_ii,  logdet Sigma_o - logdet Sigma_out = -2 n ln alpha - sum_i ln D_ii
  //    (identity step: D_ii = 1 / lam_i).  -> save_sc[10..13];  save_sc[9] = entropy of the output
  auto tail_scalars = [&](auto half_logdet, bool act) -> double {
    double v[7] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};              // sl, tr, ld, il, ll, sd, ldd
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const double li = lam[i], dii = act ? (1.0 + eta) / (li + eta) : 1.0 / li;
      const double llog = log(li), dlog = log(dii);
      const double dl = act ? dii * li : 1.0;                       // D_ii lam_i
      v[0] += half_logdet(i, dlog);
      v[1] += 1.0 / dl;
      v[2] += act ? dlog + llog : 0.0;
      v[3] += 1.0 / li;
      v[4] += llog;
      v[5] += dii;
      v[6] += dlog;
    }
    block_sum_n<7>(v, nrm + 64);
    const double H = 0.5 * n * (1.0 + LOG_2PI) + v[0];
    double alpha = 1.0, Hout = H;
    bool ent_active = false;
    if (beta) {
      const double bt = beta[b * ldb_beta];
      ent_active = entropy_eq || (H < bt);
      alpha = ent_active ? exp((bt - H) / n) : 1.0;
      Hout = ent_active ? bt : H;                                   // H + n ln alpha
    }
    if (threadIdx.x == 0) {
      double *sc = save_sc + b * KL_SC;
      if (beta) { sc[4] = alpha; sc[5] = ent_active ? 1.0 : 0.0; sc[6] = alpha * alpha; }
      const double la = log(alpha);
      sc[7] = 0.5 * (v[1] / (alpha * alpha) - (double)n);           // "shape" part  1/2 (tr - n)
      sc[8] = 0.5 * (2.0 * n * la + v[2]);                          // "volume" part 1/2 (logdet_t - logdet)
      sc[9] = Hout;
      sc[10] = 0.5 * (v[3] - (double)n);
      sc[11] = 0.5 * v[4];
      sc[12] = 0.5 * (alpha * alpha * v[5] - (double)n);
      sc[13] = -(double)n * la - 0.5 * v[6];
    }
    return alpha;
  };
  // Sigma of the (pre-entropy) result goes to the state as well: with ONE covariance for the batch the
  // likelihood's stage 1 takes alpha^2 * Sigma from there instead of re-forming L L^T per episode.
  if (!active) {                                                                    // identity
    la_gemm(bS, bL, bL.T(), n, n, n, TRI_LOWER, TRI_UPPER, TRI_FULL, 1.0, 0.0);      // Sigma = Lt Lt^T
    store_full_rows(save_Sig + off, bS, n, threadIdx.x, blockDim.x);
    const double alpha = tail_scalars([&](int i, double) { return log(bL(i, i)); }, false);
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
      const float v = (e % n <= e / n) ? (float)bL(e / n, e % n) : 0.f;          // Lt (fp32 values, exact in fp64)
      out[e] = v;
      if (out_L) out_L[off + e] = (float)(alpha * (double)v);
    }
    if (info && threadIdx.x == 0) info[b] = 0;
    return;
  }
  {                                                                                 // M sqrt(D)
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (int)(blockDim.x >> 5);
    for (int i = w; i < n; i += nw)
      for (int j = lane; j < n; j += 32) b2(i, j) *= nrm[j];
  }
  __syncthreads();
  KL_STAMP(6);
  la_gemm(b1, b2, b2.T(), n, n, n, TRI_FULL, TRI_FULL, TRI_LOWER, 1.0, 0.0);       // Sigma_proj (all of it is written)
  store_full_rows(save_Sig + off, b1, n, threadIdx.x, blockDim.x);
  if (split) {        // the factor is formed by kl_chol_kernel; consumers of Sigma (likelihood stage 1) need not wait
    tail_scalars([&](int i, double dlog) { return log((double)Lo[(size_t)i * n + i]) + 0.5 * dlog; }, true);
    KL_STAMP(7); KL_STAMP(8); KL_STAMP(9);
    return;
  }
  __syncthreads();                                                                  // ... before chol overwrites it
  KL_STAMP(7);
  la_chol(b1, n, &s_bad);
  KL_STAMP(8);
  const double alpha = tail_scalars([&](int i, double) { return log(b1(i, i)); }, true);
  store_lower_f(out, b1, n, 1.0);
  if (out_L) store_lower_f(out_L + off, b1, n, alpha);
  if (info && threadIdx.x == 0) info[b] = s_bad;
  KL_STAMP(9);
}

// Second half of a `split` forward: proj_L = chol(Sigma_proj) from the state, out_L = alpha * proj_L.
__global__ void __launch_bounds__(KL_THREADS)
kl_chol_kernel(const double *__restrict__ save_Sig, const double *__restrict__ save_sc, float *__restrict__ proj_L,
               float *__restrict__ out_L, double *__restrict__ out_inv, int32_t *__restrict__ info, int n) {
  extern __shared__ double sd[];
  const int m = pad_even(n), LD = m + 1, MS = m * LD;
  Mat b0{sd, LD, 1}, b1{sd + MS, LD, 1};
  double *dinv = sd + 2 * MS;
  __shared__ int s_bad;
  const long long b = blockIdx.x;
  const size_t off = (size_t)b * n * n;
  const double alpha = save_sc[b * KL_SC + 4];
  if (save_sc[b * KL_SC + 1] == 0.0) {                // inactive projection: the first half wrote the identity result
    if (!out_inv) return;
    load_lower_d(b0, proj_L + off, n, m);             // proj_L = Lt
  } else {
    if (threadIdx.x == 0) s_bad = 0;
    load_full_d(b0, save_Sig + off, n, m);
    la_chol(b0, n, &s_bad);
    store_lower_f(proj_L + off, b0, n, 1.0);
    if (out_L) store_lower_f(out_L + off, b0, n, alpha);
    if (info && threadIdx.x == 0) info[b] = s_bad;
  }
  if (out_inv) {                                      // (alpha P)^-1, fp64 lower: the trust-region loss's Mahalanobis term
    __syncthreads();
    la_tri_inverse(b0, b1, dinv, n);
    const double ia = 1.0 / alpha;
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
      const int i = e / n, j = e - i * n;
      out_inv[off + e] = j <= i ? ia * b1(i, j) : 0.0;
    }
  }
}

// Backward (implicit differentiation of eta*, no eigen-derivative singularities).  With P = proj_L, G the
// upstream gradient, Phi = Phi(P^T G) (lower triangle, halved diagonal) the Cholesky adjoint is
// Sbar = sym(P^-T Phi P^-1); only M^T Sbar M is needed, so with Y = P^-1 M
//   Ft = sym(Y^T Phi Y) ;  rho_i = 1/(lam_i + eta) ;
//   Nt_ij = -(1+eta) rho_i rho_j Ft_ij - delta_ij etabar (df/dlam_i) / (df/deta) ,
//   etabar = sum_i Ft_ii (rho_i - (1+eta) rho_i^2) ;  grad_Lt = -2 tril(Lt^-T U~ Nt U~^T)
// with U~ = Lt^-1 M and Lt^-1 saved by the forward.  No triangular solves: P^-1 by recursive doubling
// (la_tri_inverse), everything else is fp64 tensor-core GEMMs (la_gemm) on four shared buffers.
__global__ void __launch_bounds__(KL_THREADS)
proj_kl_cov_bwd_kernel(const float *__restrict__ L, const float *__restrict__ proj_L, const float *__restrict__ gout,
                       const double *__restrict__ save_M, const double *__restrict__ save_U,
                       const double *__restrict__ save_Li, const double *__restrict__ save_lam,
                       const double *__restrict__ save_sc, float *__restrict__ grad_L, int n, int fused_entropy,
                       const double *__restrict__ out_inv, double tr_coeff, int compact) {
  extern __shared__ double sd[];
  const int m = pad_even(n), LD = m + 1, MS = m * LD;
  Mat b0{sd, LD, 1}, b1{sd + MS, LD, 1}, b2{sd + 2 * MS, LD, 1}, b3{sd + 3 * MS, LD, 1};     // b3: not with `compact`
  double *dinv = sd + (compact ? 3 : 4) * MS, *lam = dinv + LA_DINV_DOUBLES, *rho = lam + m, *red = rho + m;
  const long long b = blockIdx.x;
  const size_t off = (size_t)b * n * n;
  float *gl = grad_L + off;
  (void)L;
  const double eta = save_sc[b * KL_SC + 0];
  const bool kl_active = save_sc[b * KL_SC + 1] != 0.0;
  // tr_coeff != 0: the gradient of the trust-region regression term tr_coeff * KL_cov(N(Lt Lt^T) || N(Sigma_out DETACHED))
  // is added (see proj_kl_cov_bwd_sigma_kernel); identity KL step: Sigma_out = alpha^2 Lt Lt^T -> tr_coeff (1 / alpha^2 - 1) / Lt_ii
  if (!kl_active && !fused_entropy) {                                              // identity (alpha = 1: no trust-region term)
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) gl[e] = (e % n <= e / n) ? gout[off + e] : 0.f;
    return;
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x) { lam[i] = save_lam[b * n + i]; rho[i] = 1.0 / (lam[i] + eta); }
  load_lower_d(b0, proj_L + off, n, m);                                            // P
  load_lower_d(b1, gout + off, n, m);                                              // G
  if (fused_entropy) {               // G <- adjoint of out_L = alpha(P) P  (proj_entropy_kernel, backward branch)
    const double alpha = save_sc[b * KL_SC + 4];
    const bool ent_active = save_sc[b * KL_SC + 5] != 0.0;
    double dot = 0.0;
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
      const int i = e / n, j = e - i * n;
      if (j <= i) dot = fma(b1(i, j), b0(i, j), dot);
    }
    dot = block_sum(dot, red);
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
      const int i = e / n, j = e - i * n;
      if (j > i) continue;
      double v = alpha * b1(i, j);
      if (i == j && ent_active) v -= dot * alpha / (n * b0(i, i));
      b1(i, j) = v;
    }
    __syncthreads();
    if (!kl_active) {                                                              // identity KL step
      if (tr_coeff != 0.0) {
        const double a2 = alpha * alpha;
        for (int i = threadIdx.x; i < n; i += blockDim.x) b1(i, i) += tr_coeff * (1.0 / a2 - 1.0) / (double)L[off + (size_t)i * n + i];
        __syncthreads();
      }
      store_lower_f(gl, b1, n, 1.0);
      return;
    }
  }
  la_gemm(b2, b0.T(), b1, n, n, n, TRI_UPPER, TRI_LOWER, TRI_FULL, 1.0, 0.0);      // P^T G
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, j = e - i * n;
    if (j > i) b2(i, j) = 0.0; else if (i == j) b2(i, j) *= 0.5;                   // Phi
  }
  // `compact` (batches: two CTAs of 256 threads per SM, three buffers): F' = M^T (P^-T Phi P^-1) M with the products
  // ordered so that never more than two operands and one result are alive; bF = where F' ends up, bN = where Nt goes
  Mat bF = compact ? b2 : b1, bN = compact ? b1 : b2, bT = compact ? b2 : b3;
  auto load_out_inv = [&](Mat X) {   // (alpha P)^-1 is already known (the trust-region loss inverts the layer's output)
    const double alpha = fused_entropy ? save_sc[b * KL_SC + 4] : 1.0;
    batched_load(out_inv + off, n * n, [&](int e, double v) {
      const int i = e / n, j = e - i * n;
      X(i, j) = j <= i ? alpha * v : 0.0;
    });
    zero_padding(X, n, m);
    __syncthreads();
  };
  if (compact) {
    __syncthreads();                                                               // Phi complete, G consumed
    if (out_inv) load_out_inv(b1); else la_tri_inverse(b0, b1, dinv, n);           // P^-1 (over G)
    la_gemm(b0, b2, b1, n, n, n, TRI_LOWER, TRI_LOWER, TRI_LOWER, 1.0, 0.0);       // Phi P^-1 (over P; lower x lower)
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {                        // (its strict upper triangle is zero)
      const int i = e / n, j = e - i * n;
      if (j > i) b0(i, j) = 0.0;
    }
    __syncthreads();
    la_gemm(b2, b1.T(), b0, n, n, n, TRI_UPPER, TRI_LOWER, TRI_FULL, 1.0, 0.0);    // S' = P^-T Phi P^-1 (over Phi)
    load_full_d(b0, save_M + off, n, m);                                           // M
    la_gemm(b1, b2, b0, n, n, n, TRI_FULL, TRI_FULL, TRI_FULL, 1.0, 0.0);          // S' M
    la_gemm(b2, b0.T(), b1, n, n, n, TRI_FULL, TRI_FULL, TRI_FULL, 1.0, 0.0);      // F' = M^T S' M ; Ft = sym(F')
  } else {
    load_full_d(b1, save_M + off, n, m);                                           // M (G is consumed)
    if (out_inv) load_out_inv(b3); else la_tri_inverse(b0, b3, dinv, n);           // P^-1
    la_gemm(b0, b3, b1, n, n, n, TRI_LOWER, TRI_FULL, TRI_FULL, 1.0, 0.0);         // Y = P^-1 M (P is consumed)
    la_gemm(b3, b2, b0, n, n, n, TRI_LOWER, TRI_FULL, TRI_FULL, 1.0, 0.0);         // Phi Y
    la_gemm(b1, b0.T(), b3, n, n, n, TRI_FULL, TRI_FULL, TRI_FULL, 1.0, 0.0);      // F' = Y^T Phi Y ; Ft = sym(F')
  }
  double eb = 0.0, dfe = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    eb += bF(i, i) * (rho[i] - (1.0 + eta) * rho[i] * rho[i]);
    dfe += 2.0 * rho[i] - (1.0 + eta) * rho[i] * rho[i] - 1.0 / (1.0 + eta);
  }
  eb = block_sum(eb, red);
  dfe = 0.5 * block_sum(dfe, red);
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, j = e - i * n;
    double v = -(1.0 + eta) * rho[i] * rho[j] * (0.5 * (bF(i, j) + bF(j, i)));
    if (i == j) v -= eb * (0.5 * (rho[i] - (1.0 + eta) * rho[i] * rho[i])) / dfe;
    if (i == j && tr_coeff != 0.0) {                                               // trust-region term, as in the sigma kernel
      const double a2 = fused_entropy ? save_sc[b * KL_SC + 6] : 1.0;
      v -= 0.5 * tr_coeff / (a2 * (1.0 + eta) * rho[i] * lam[i] * lam[i]);
    }
    bN(i, j) = v;                                                                  // Nt (Phi / S' M is consumed)
  }
  load_full_d(b0, save_U + off, n, m);                                             // U~ (Y / M is consumed)
  la_gemm(bT, b0, bN, n, n, n, TRI_FULL, TRI_FULL, TRI_FULL, 1.0, 0.0);            // U~ Nt (compact: over F', which Nt
  la_gemm(b1, bT, b0.T(), n, n, n, TRI_FULL, TRI_FULL, TRI_FULL, 1.0, 0.0);        // has absorbed) ; U~ Nt U~^T (over F' / Nt)
  Mat bI = compact ? b0 : b2, bG = compact ? b2 : b3;
  load_full_d(bI, save_Li + off, n, m);                                            // Lt^-1 (Nt / U~ is consumed)
  la_gemm(bG, bI.T(), b1, n, n, n, TRI_UPPER, TRI_FULL, TRI_LOWER, 1.0, 0.0);      // Lt^-T (.)
  if (tr_coeff != 0.0) {                                                           // - tr_coeff (Lt^-T)_ii  (scaled by -2 below)
    for (int i = threadIdx.x; i < n; i += blockDim.x) bG(i, i) += 0.5 * tr_coeff / (double)L[off + (size_t)i * n + i];
    __syncthreads();
  }
  store_lower_f(gl, bG, n, -2.0);
}

// Backward in COVARIANCE space: the consumer of the projected covariance (the segment likelihood, which reads
// Sigma_out = alpha^2 Sigma_proj straight from the state) hands back Sbar_out = d loss / d Sigma_out (symmetric, fp64)
// instead of a gradient w.r.t. the Cholesky factor.  Then M^T Sbar_proj M is formed directly:
//   F0 = M^T Sbar_out M ;  fused entropy control (alpha = exp((beta - H) / n), H = const + 1/2 logdet Sigma_proj):
//   Sbar_proj = alpha^2 (Sbar_out - c / n Sigma_proj^-1),  c = <Sbar_out, Sigma_proj> = sum_i D_ii F0_ii,
//   M^T Sigma_proj^-1 M = D^-1,  D = diag((1 + eta) / (lam + eta))   =>   Ft = alpha^2 (F0 - c / n D^-1)
// and the rest is the implicit differentiation of proj_kl_cov_bwd_kernel.  Neither the factor P, nor P^-1, nor the
// Cholesky adjoint appear: 5 GEMMs instead of 7 + a triangular inverse, and the forward need not form P on the
// critical path at all (tce_proj_kl_entropy_fwd_sigma).
// K = Lt^-T U~ : the part of the covariance-space backward that does not depend on the incoming gradient.  Launched
// right after the forward on the covariance stream it runs while the segment likelihood is busy and takes one GEMM and
// one matrix load off the backward's critical path.
__global__ void __launch_bounds__(KL_THREADS)
kl_bwd_prep_kernel(const double *__restrict__ save_U, const double *__restrict__ save_Li, const double *__restrict__ save_sc,
                   double *__restrict__ save_K, int n) {
  extern __shared__ double sd[];
  const int m = pad_even(n), LD = m + 1, MS = m * LD;
  Mat b0{sd, LD, 1}, b1{sd + MS, LD, 1}, b2{sd + 2 * MS, LD, 1};
  const long long b = blockIdx.x;
  const size_t off = (size_t)b * n * n;
  if (save_sc[b * KL_SC + 1] == 0.0) return;                                        // identity step: K is not used
  {
    const int total = n * n, step = (int)blockDim.x;
    for (int e0 = threadIdx.x; e0 < total; e0 += 4 * step) {
      double vu[4], vl[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = e0 + u * step;
        vu[u] = e < total ? save_U[off + e] : 0.0;
        vl[u] = e < total ? save_Li[off + e] : 0.0;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = e0 + u * step;
        if (e < total) { const int i = e / n, j = e - i * n; b0(i, j) = vu[u]; b1(i, j) = vl[u]; }
      }
    }
    zero_padding(b0, n, m);
    zero_padding(b1, n, m);
    __syncthreads();
  }
  la_gemm(b2, b1.T(), b0, n, n, n, TRI_UPPER, TRI_FULL, TRI_FULL, 1.0, 0.0);        // Lt^-T U~
  store_full_rows(save_K + off, b2, n, threadIdx.x, blockDim.x);
}

__global__ void __launch_bounds__(KL_THREADS)
proj_kl_cov_bwd_sigma_kernel(const float *__restrict__ L, const double *__restrict__ gsig,
                             const double *__restrict__ save_M, const double *__restrict__ save_U,
                             const double *__restrict__ save_Li, const double *__restrict__ save_Sig,
                             const double *__restrict__ save_lam, const double *__restrict__ save_sc,
                             const double *__restrict__ save_K, float *__restrict__ grad_L, int n, int fused_entropy,
                             double tr_coeff, const float *__restrict__ vec, long long ldb_vec,
                             float *__restrict__ grad_vec) {
  extern __shared__ double sd[];
  const int m = pad_even(n), LD = m + 1, MS = m * LD;
  Mat b0{sd, LD, 1}, b1{sd + MS, LD, 1}, b2{sd + 2 * MS, LD, 1}, b3{sd + 3 * MS, LD, 1}, b4{sd + 4 * MS, LD, 1},
      b5{sd + 5 * MS, LD, 1};
  double *dinv = sd + 6 * MS, *lam = dinv + LA_DINV_DOUBLES, *rho = lam + m, *red = rho + m;
  const long long b = blockIdx.x;
  const size_t off = (size_t)b * n * n;
  float *gl = grad_L ? grad_L + off : nullptr;
  // grad_vec != NULL: the adjoint of the policy head is fused in (head_bwd_kernel): the gradient is written w.r.t. the
  // covariance vector -- strictly-lower entries copied, diagonal entries times sigmoid(v_i) -- instead of w.r.t. Lt
  const float *vb = grad_vec ? vec + b * ldb_vec : nullptr;
  float *gv = grad_vec ? grad_vec + b * (long long)(n + n * (n - 1) / 2) : nullptr;
  auto emit = [&](int i, int j, double v) {
    if (gv) {
      if (j < i) gv[n + i * (i - 1) / 2 + j] = (float)v;
      else if (j == i) gv[i] = (float)(v / (1.0 + exp(-(double)vb[i])));
    } else {
      gl[(size_t)i * n + j] = (float)v;
    }
  };
  const double eta = save_sc[b * KL_SC + 0];
  const bool kl_active = save_sc[b * KL_SC + 1] != 0.0;
  const double alpha = fused_entropy ? save_sc[b * KL_SC + 4] : 1.0, a2 = alpha * alpha;
  const bool ent_active = fused_entropy && save_sc[b * KL_SC + 5] != 0.0;
  KL_STAMP(16);
  if (!kl_active) {
    // identity KL step: Sigma_proj = Lt Lt^T, grad_Lt = 2 alpha^2 tril(Sbar_out Lt) - (2 alpha^2 c / n) diag(1 / Lt_ii)
    load_full_d(b0, gsig + off, n, m);                                             // Sbar_out
    load_lower_d(b1, L + off, n, m);                                               // Lt
    double c = 0.0;
    if (ent_active) {
      for (int e = threadIdx.x; e < n * n; e += blockDim.x) c = fma(b0(e / n, e % n), save_Sig[off + e], c);
      c = block_sum(c, red);
    }
    la_gemm(b2, b0, b1, n, n, n, TRI_FULL, TRI_LOWER, TRI_LOWER, 1.0, 0.0);
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
      const int i = e / n, j = e - i * n;
      double v = j <= i ? 2.0 * a2 * b2(i, j) : 0.0;
      if (i == j && ent_active) v -= 2.0 * a2 * c / (n * b1(i, i));
      if (i == j) v += tr_coeff * (1.0 / a2 - 1.0) / b1(i, i);      // trust-region term: Sigma_t = alpha^2 Sigma
      emit(i, j, v);
    }
    return;
  }
  // Every matrix the backward needs is requested at once (eight loads in flight per thread): Sbar_out -> b0, M -> b1,
  // U~ -> b4, and K = Lt^-T U~ -> b5 when tce_proj_kl_bwd_prep ran (else Lt^-1 -> b5).
  {
    const double *src3 = save_K ? save_K : save_Li;
    const int total = n * n, step = (int)blockDim.x;
    for (int e0 = threadIdx.x; e0 < total; e0 += 2 * step) {
      double v0[2], v1[2], v2[2], v3[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int e = e0 + u * step;
        const bool ok = e < total;
        v0[u] = ok ? gsig[off + e] : 0.0; v1[u] = ok ? save_M[off + e] : 0.0;
        v2[u] = ok ? save_U[off + e] : 0.0; v3[u] = ok ? src3[off + e] : 0.0;
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int e = e0 + u * step;
        if (e < total) {
          const int i = e / n, j = e - i * n;
          b0(i, j) = v0[u]; b1(i, j) = v1[u]; b4(i, j) = v2[u]; b5(i, j) = v3[u];
        }
      }
    }
    for (int i = threadIdx.x; i < n; i += blockDim.x) { lam[i] = save_lam[b * n + i]; rho[i] = 1.0 / (lam[i] + eta); }
    zero_padding(b0, n, m); zero_padding(b1, n, m); zero_padding(b4, n, m); zero_padding(b5, n, m);
    __syncthreads();
  }
  KL_STAMP(17);
  KL_STAMP(18);
  la_gemm(b2, b0, b1, n, n, n, TRI_FULL, TRI_FULL, TRI_FULL, 1.0, 0.0);            // Sbar_out M
  KL_STAMP(19);
  la_gemm(b3, b1.T(), b2, n, n, n, TRI_FULL, TRI_FULL, TRI_FULL, 1.0, 0.0);        // F0 = M^T Sbar_out M
  KL_STAMP(20);
  // c = <Sbar_out, Sigma_proj> = sum_i D_ii F0_ii (entropy adjoint), etabar, d f / d eta: one reduction
  double v3s[3] = {0.0, 0.0, 0.0};
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    v3s[0] += (1.0 + eta) * rho[i] * b3(i, i);
    v3s[2] += 2.0 * rho[i] - (1.0 + eta) * rho[i] * rho[i] - 1.0 / (1.0 + eta);
  }
  block_sum_n<3>(v3s, red);
  const double c = ent_active ? v3s[0] : 0.0, dfe = 0.5 * v3s[2];
  double eb = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double ft = a2 * (b3(i, i) - (ent_active ? c / (n * (1.0 + eta) * rho[i]) : 0.0));
    eb += ft * (rho[i] - (1.0 + eta) * rho[i] * rho[i]);
  }
  eb = block_sum(eb, red);
  {
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (int)(blockDim.x >> 5);
    for (int i = w; i < n; i += nw)
      for (int j = lane; j < n; j += 32) {
        double ft = a2 * 0.5 * (b3(i, j) + b3(j, i));
        if (i == j && ent_active) ft -= a2 * c / (n * (1.0 + eta) * rho[i]);
        double v = -(1.0 + eta) * rho[i] * rho[j] * ft;
        if (i == j) v -= eb * (0.5 * (rho[i] - (1.0 + eta) * rho[i] * rho[i])) / dfe;
        // trust-region regression term tr_coeff * KL_cov(N(Sigma) || N(Sigma_t)), Sigma_t = alpha^2 Sigma_proj DETACHED:
        // d / d Lt = tr_coeff (Sigma_t^-1 Lt - Lt^-T), Sigma_t^-1 Lt = Lt^-T U~ diag(1 / (alpha^2 lam_i^2 D_ii)) U~^T
        if (i == j) v -= 0.5 * tr_coeff / (a2 * (1.0 + eta) * rho[i] * lam[i] * lam[i]);
        b2(i, j) = v;                                                              // Nt
      }
  }
  __syncthreads();
  KL_STAMP(21);
  KL_STAMP(22);
  if (save_K) {
    la_gemm(b0, b2, b4.T(), n, n, n, TRI_FULL, TRI_FULL, TRI_FULL, 1.0, 0.0);      // Nt U~^T
    KL_STAMP(23);
    la_gemm(b3, b5, b0, n, n, n, TRI_FULL, TRI_FULL, TRI_LOWER, 1.0, 0.0);         // K (Nt U~^T) = Lt^-T U~ Nt U~^T
    KL_STAMP(24);
    KL_STAMP(25);
  } else {
    la_gemm(b3, b4, b2, n, n, n, TRI_FULL, TRI_FULL, TRI_FULL, 1.0, 0.0);          // U~ Nt
    KL_STAMP(23);
    la_gemm(b1, b3, b4.T(), n, n, n, TRI_FULL, TRI_FULL, TRI_FULL, 1.0, 0.0);      // U~ Nt U~^T
    KL_STAMP(24);
    KL_STAMP(25);
    la_gemm(b3, b5.T(), b1, n, n, n, TRI_UPPER, TRI_FULL, TRI_LOWER, 1.0, 0.0);    // Lt^-T (.)
  }
  KL_STAMP(26);
  {
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (int)(blockDim.x >> 5);
    for (int i = w; i < n; i += nw)
      for (int j = lane; j < n; j += 32) {
        double v = j <= i ? -2.0 * b3(i, j) : 0.0;
        if (i == j && tr_coeff != 0.0) v -= tr_coeff / (double)L[off + (size_t)i * n + i];          // - tr_coeff (Lt^-T)_ii
        emit(i, j, v);
      }
  }
  KL_STAMP(27);
}

// =====================================================================================================
// Frobenius covariance projection
// =====================================================================================================
__global__ void __launch_bounds__(PJ_THREADS)
proj_frob_cov_fwd_kernel(const float *__restrict__ L, const float *__restrict__ L_o, long long ldb_Lo, double eps_cov,
                         float *__restrict__ proj_L, double *__restrict__ save_sc, int32_t *__restrict__ info, int n) {
  extern __shared__ double sd[];
  const int m = pad_even(n), LD = m + 1, MS = m * LD;
  Mat b0{sd, LD, 1}, b1{sd + MS, LD, 1}, b2{sd + 2 * MS, LD, 1};
  double *red = sd + 3 * MS;
  __shared__ int s_bad;
  const long long b = blockIdx.x;
  const size_t off = (size_t)b * n * n;
  if (threadIdx.x == 0) s_bad = 0;
  load_lower_d(b0, L + off, n, m);
  la_gemm(b1, b0, b0.T(), n, n, n, TRI_LOWER, TRI_UPPER, TRI_FULL, 1.0, 0.0);     // Sigma
  load_lower_d(b0, L_o + b * ldb_Lo, n, m);
  la_gemm(b2, b0, b0.T(), n, n, n, TRI_LOWER, TRI_UPPER, TRI_FULL, 1.0, 0.0);     // Sigma_o
  double cp = 0.0;
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) { const double d = b2(e / n, e % n) - b1(e / n, e % n); cp = fma(d, d, cp); }
  cp = block_sum(cp, red);
  const bool active = cp > eps_cov;
  const double eta = active ? fabs(sqrt(cp / eps_cov) - 1.0) : 0.0;
  if (save_sc && threadIdx.x == 0) { save_sc[b * 4] = eta; save_sc[b * 4 + 1] = active ? 1.0 : 0.0; save_sc[b * 4 + 2] = cp; save_sc[b * 4 + 3] = 0.0; }
  float *out = proj_L + off;
  if (!active) {
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) out[e] = (e % n <= e / n) ? L[off + e] : 0.f;
    if (info && threadIdx.x == 0) info[b] = 0;
    return;
  }
  const double a = 1.0 / (1.0 + eta + 1e-16);
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) b1(e / n, e % n) = (b1(e / n, e % n) + eta * b2(e / n, e % n)) * a;
  __syncthreads();
  la_chol(b1, n, &s_bad);
  store_lower_f(out, b1, n, 1.0);
  if (info && threadIdx.x == 0) info[b] = s_bad;
}

__global__ void __launch_bounds__(PJ_THREADS)
proj_frob_cov_bwd_kernel(const float *__restrict__ L, const float *__restrict__ L_o, long long ldb_Lo, double eps_cov,
                         const float *__restrict__ proj_L, const float *__restrict__ gout,
                         const double *__restrict__ save_sc, float *__restrict__ grad_L, int n) {
  extern __shared__ double sd[];
  const int m = pad_even(n), LD = m + 1, MS = m * LD;
  Mat b0{sd, LD, 1}, b1{sd + MS, LD, 1}, b2{sd + 2 * MS, LD, 1}, b3{sd + 3 * MS, LD, 1};
  double *inv_diag = sd + 4 * MS, *red = inv_diag + LA_DINV_DOUBLES;
  const long long b = blockIdx.x;
  const size_t off = (size_t)b * n * n;
  float *gl = grad_L + off;
  const double eta = save_sc[b * 4];
  if (save_sc[b * 4 + 1] == 0.0) {
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) gl[e] = (e % n <= e / n) ? gout[off + e] : 0.f;
    return;
  }
  load_lower_d(b0, proj_L + off, n, m);
  load_lower_d(b1, gout + off, n, m);
  chol_backward(b0, b1, b2, inv_diag, n);                                          // b2 = Sbar_new (sym)
  load_lower_d(b1, L + off, n, m);
  la_gemm(b3, b1, b1.T(), n, n, n, TRI_LOWER, TRI_UPPER, TRI_FULL, 1.0, 0.0);     // Sigma
  load_lower_d(b1, L_o + b * ldb_Lo, n, m);
  la_gemm(b0, b1, b1.T(), n, n, n, TRI_LOWER, TRI_UPPER, TRI_FULL, 1.0, 0.0);     // Sigma_o
  double dot = 0.0;
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, j = e % n;
    const double d = b0(i, j) - b3(i, j);
    b0(i, j) = d;                                                                  // Dm = Sigma_o - Sigma
    dot = fma(b2(i, j), d, dot);
  }
  dot = block_sum(dot, red);
  const double a = 1.0 / (1.0 + eta + 1e-16);
  const double cp = save_sc[b * 4 + 2];
  const double eta_bar = a * a * dot, deta_dcp = 1.0 / (2.0 * sqrt(cp * eps_cov));
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, j = e % n;
    b2(i, j) = a * b2(i, j) - 2.0 * eta_bar * deta_dcp * b0(i, j);                 // Sigma_bar
  }
  __syncthreads();
  load_lower_d(b1, L + off, n, m);
  la_gemm(b3, b2, b1, n, n, n, TRI_FULL, TRI_LOWER, TRI_LOWER, 2.0, 0.0);          // grad = 2 Sigma_bar L (lower)
  store_lower_f(gl, b3, n, 1.0);
}

// =====================================================================================================
// W2 (commutative) covariance projection on whatever "square roots" are passed (Cholesky factors in TCE)
// =====================================================================================================
// cov_part: scale_prec ? tr(I + A Sigma A - 2 A R) : tr(Sigma_o + Sigma - 2 S R), A = S^-1, S = L_o, R = L
// mode 0: forward (proj + scalars); mode 1: backward
__global__ void __launch_bounds__(PJ_THREADS)
proj_w2_cov_kernel(const float *__restrict__ L, const float *__restrict__ L_o, long long ldb_Lo, double eps_cov,
                   int scale_prec, const float *__restrict__ gout, float *__restrict__ out, double *__restrict__ save_sc,
                   int n) {
  extern __shared__ double sd[];
  const int m = pad_even(n), LD = m + 1, MS = m * LD;
  Mat R{sd, LD, 1}, S{sd + MS, LD, 1}, A{sd + 2 * MS, LD, 1}, T{sd + 3 * MS, LD, 1}, U{sd + 4 * MS, LD, 1};
  double *inv_diag = sd + 5 * MS, *red = inv_diag + LA_DINV_DOUBLES;
  const long long b = blockIdx.x;
  const size_t off = (size_t)b * n * n;
  load_lower_d(R, L + off, n, m);
  load_lower_d(S, L_o + b * ldb_Lo, n, m);
  double cp;
  if (scale_prec) {
    zero_padding(A, n, m);
    la_tri_inverse(S, A, inv_diag, n);                                             // A = S^-1 (lower)
    la_gemm(T, A, R, n, n, n, TRI_LOWER, TRI_LOWER, TRI_FULL, 1.0, 0.0);           // T = A R (lower)
    la_gemm(U, A.T(), R, n, n, n, TRI_UPPER, TRI_LOWER, TRI_FULL, 1.0, 0.0);       // U = A^T R
    double v = 0.0;
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
      const int i = e / n, j = e % n;
      v = fma(T(i, j), U(i, j), v);
      if (i == j) v += 1.0 - 2.0 * T(i, i);
    }
    cp = block_sum(v, red);
  } else {
    la_gemm(T, S, R, n, n, n, TRI_LOWER, TRI_LOWER, TRI_FULL, 1.0, 0.0);           // S R
    double v = 0.0;
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
      const int i = e / n, j = e % n;
      v += S(i, j) * S(i, j) + R(i, j) * R(i, j);
      if (i == j) v -= 2.0 * T(i, i);
    }
    cp = block_sum(v, red);
  }
  const bool active = cp > eps_cov;
  const double eta = active ? fabs(sqrt(cp / eps_cov) - 1.0) : 0.0;
  const double a = 1.0 / (1.0 + eta + 1e-16);
  float *ob = out + off;
  if (!gout) {
    if (save_sc && threadIdx.x == 0) { save_sc[b * 4] = eta; save_sc[b * 4 + 1] = active ? 1.0 : 0.0; save_sc[b * 4 + 2] = cp; save_sc[b * 4 + 3] = 0.0; }
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
      const int i = e / n, j = e % n;
      ob[e] = j <= i ? (float)(active ? (R(i, j) + eta * S(i, j)) * a : R(i, j)) : 0.f;
    }
    return;
  }
  const float *gb = gout + off;
  if (!active) {
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) ob[e] = (e % n <= e / n) ? gb[e] : 0.f;
    return;
  }
  // eta_bar = <g, a (S - proj)>, proj = (R + eta S) a
  double dot = 0.0;
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, j = e % n;
    if (j <= i) dot = fma((double)gb[e], a * (S(i, j) - (R(i, j) + eta * S(i, j)) * a), dot);
  }
  dot = block_sum(dot, red);
  const double coef = dot / (2.0 * sqrt(cp * eps_cov));
  if (scale_prec) {
    // d cp / d R = A T + A^T U - 2 A^T   (lower part)
    la_gemm(S, A, T, n, n, n, TRI_LOWER, TRI_LOWER, TRI_LOWER, 1.0, 0.0);          // S <- A T (S no longer needed)
    la_gemm(S, A.T(), U, n, n, n, TRI_UPPER, TRI_FULL, TRI_LOWER, 1.0, 1.0);       // += A^T U
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
      const int i = e / n, j = e % n;
      double v = 0.0;
      if (j <= i) v = a * gb[e] + coef * (S(i, j) - 2.0 * A(j, i));
      ob[e] = (float)v;
    }
  } else {
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
      const int i = e / n, j = e % n;
      double v = 0.0;
      if (j <= i) v = a * gb[e] + coef * (2.0 * R(i, j) - 2.0 * S(j, i));
      ob[e] = (float)v;
    }
  }
}

// gradient of the W2 / Frobenius covariance distances themselves (needed by the trust-region loss):
// value only (gval == nullptr) or gradient w.r.t. L scaled by gval[b]
__global__ void __launch_bounds__(PJ_THREADS)
cov_distance_kernel(int kind /*0 frob, 1 w2*/, const float *__restrict__ L, const float *__restrict__ L_o,
                    long long ldb_Lo, int scale_prec, const double *__restrict__ gval, double *__restrict__ val,
                    float *__restrict__ grad_L, int n) {
  extern __shared__ double sd[];
  const int m = pad_even(n), LD = m + 1, MS = m * LD;
  Mat R{sd, LD, 1}, S{sd + MS, LD, 1}, A{sd + 2 * MS, LD, 1}, T{sd + 3 * MS, LD, 1}, U{sd + 4 * MS, LD, 1};
  double *inv_diag = sd + 5 * MS, *red = inv_diag + LA_DINV_DOUBLES;
  const long long b = blockIdx.x;
  const size_t off = (size_t)b * n * n;
  load_lower_d(R, L + off, n, m);
  load_lower_d(S, L_o + b * ldb_Lo, n, m);
  double cp = 0.0;
  if (kind == 0) {
    la_gemm(T, R, R.T(), n, n, n, TRI_LOWER, TRI_UPPER, TRI_FULL, 1.0, 0.0);      // Sigma
    la_gemm(U, S, S.T(), n, n, n, TRI_LOWER, TRI_UPPER, TRI_FULL, 1.0, 0.0);      // Sigma_o
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
      const int i = e / n, j = e % n;
      const double d = U(i, j) - T(i, j);
      U(i, j) = d;
      cp = fma(d, d, cp);
    }
    cp = block_sum(cp, red);
    if (gval) {                                                                    // d/dL = -4 (Sigma_o - Sigma) L
      la_gemm(T, U, R, n, n, n, TRI_FULL, TRI_LOWER, TRI_LOWER, -4.0 * gval[b], 0.0);
      store_lower_f(grad_L + off, T, n, 1.0);
    }
  } else if (scale_prec) {
    zero_padding(A, n, m);
    la_tri_inverse(S, A, inv_diag, n);
    la_gemm(T, A, R, n, n, n, TRI_LOWER, TRI_LOWER, TRI_FULL, 1.0, 0.0);
    la_gemm(U, A.T(), R, n, n, n, TRI_UPPER, TRI_LOWER, TRI_FULL, 1.0, 0.0);
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
      const int i = e / n, j = e % n;
      cp = fma(T(i, j), U(i, j), cp);
      if (i == j) cp += 1.0 - 2.0 * T(i, i);
    }
    cp = block_sum(cp, red);
    if (gval) {
      la_gemm(S, A, T, n, n, n, TRI_LOWER, TRI_LOWER, TRI_LOWER, 1.0, 0.0);
      la_gemm(S, A.T(), U, n, n, n, TRI_UPPER, TRI_FULL, TRI_LOWER, 1.0, 1.0);
      const double g = gval[b];
      for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
        const int i = e / n, j = e % n;
        grad_L[off + e] = j <= i ? (float)(g * (S(i, j) - 2.0 * A(j, i))) : 0.f;
      }
    }
  } else {
    la_gemm(T, S, R, n, n, n, TRI_LOWER, TRI_LOWER, TRI_FULL, 1.0, 0.0);
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
      const int i = e / n, j = e % n;
      cp += S(i, j) * S(i, j) + R(i, j) * R(i, j);
      if (i == j) cp -= 2.0 * T(i, i);
    }
    cp = block_sum(cp, red);
    if (gval) {
      const double g = gval[b];
      for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
        const int i = e / n, j = e % n;
        grad_L[off + e] = j <= i ? (float)(g * (2.0 * R(i, j) - 2.0 * S(j, i))) : 0.f;
      }
    }
  }
  if (val && threadIdx.x == 0) val[b] = cp;
}

size_t pj_smem(int n, int nbuf) {
  const int m = (n + 1) & ~1;
  return sizeof(double) * ((size_t)nbuf * m * (m + 1) + LA_DINV_DOUBLES + 8 * m + 256);
}

// CTA-per-matrix kernels launched for a FEW matrices (shared covariance: B = 1) are latency chains on the
// critical path of the epoch, and batch-sized kernels of parallel graph branches would be co-scheduled onto
// their SMs (issue slots shared with 8-32 busy warps: the unlucky CTA of the batch kernel then finishes 3-5x
// late and so does the chain).  Asking for (almost) all shared memory of the SM keeps the SM exclusive.
size_t pj_smem_exclusive(size_t smem, int64_t B) { return B <= 16 && smem < 200 * 1024 ? 200 * 1024 : smem; }

int num_sms_proj() {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
  }
  return sms;
}

template <typename K>
int set_smem(K kernel, size_t smem) {
  if (smem > 220 * 1024) return TCE_ERR_UNSUPPORTED_SHAPE;
  TCE_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "proj smem attr");
  // same carve-out preference as the likelihood kernels these run beside (no measurable effect either way)
  cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  return TCE_OK;
}

}  // namespace

#define PJ_CHECK_N(n) if ((n) < 1 || (n) > 64) return TCE_ERR_UNSUPPORTED_SHAPE

extern "C" int tce_gauss_stats(const float *mean, const float *L, int64_t ldb_L, const float *mean_o,
                               const float *L_o, int64_t ldb_Lo, double *out, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!mean || !mean_o || !L_o || !out || B < 0) return TCE_ERR_INVALID_ARGUMENT;
  PJ_CHECK_N(n);
  const size_t smem = pj_smem(n, 2);      // NOT exclusive: these run beside the likelihood kernels (trust-region loss,
  int rc = set_smem(gauss_kl_kernel, smem);   // logging) and must fit into the first CTA slot that frees up
  if (rc) return rc;
  gauss_kl_kernel<<<(unsigned)B, PJ_THREADS, smem, (cudaStream_t)stream>>>(mean, L, ldb_L, mean_o, L_o, ldb_Lo, out,
                                                                          nullptr, nullptr, nullptr, n, L ? 0 : 1);
  TCE_CHECK_LAUNCH("gauss_kl_kernel");
  return TCE_OK;
}

extern "C" int tce_gauss_stats_bwd(const float *mean, const float *L, int64_t ldb_L, const float *mean_o,
                                   const float *L_o, int64_t ldb_Lo, const double *grad_out, float *grad_mean,
                                   float *grad_L, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!mean || !mean_o || !L_o || !grad_out || B < 0 || (grad_L && !L)) return TCE_ERR_INVALID_ARGUMENT;
  PJ_CHECK_N(n);
  const size_t smem = pj_smem(n, 2);      // NOT exclusive: these run beside the likelihood kernels (trust-region loss,
  int rc = set_smem(gauss_kl_kernel, smem);   // logging) and must fit into the first CTA slot that frees up
  if (rc) return rc;
  gauss_kl_kernel<<<(unsigned)B, PJ_THREADS, smem, (cudaStream_t)stream>>>(mean, L, ldb_L, mean_o, L_o, ldb_Lo, nullptr,
                                                                          grad_out, grad_mean, grad_L, n, grad_L ? 0 : 1);
  TCE_CHECK_LAUNCH("gauss_kl_kernel(bwd)");
  return TCE_OK;
}

static int maha_launch(const float *mean, const float *mean_o, const float *L_o, int64_t ldb_Lo, const double *grad_out,
                       double *maha, float *grad_mean, float *grad_L, int64_t B, int n, void *stream) {
  if (n <= 64 && B >= 2 * MW_WARPS) {                   // warp per episode (a handful of episodes: the CTA kernel's extra
    cudaStream_t st = (cudaStream_t)stream;             // threads help with the loads)
    int64_t done = 0;
    // contiguous per-episode factors of odd order: whole groups of MW_WARPS episodes through the bulk-copy variant
    if ((n & 1) && ldb_Lo == (int64_t)n * n && B >= 8 * MW_WARPS && ((uintptr_t)L_o & 15) == 0) {
      const size_t smem_b = MW_WARPS * ((size_t)n * n * sizeof(float) + 2 * 64 * sizeof(double));
      if (smem_b > 48 * 1024)
        TCE_CUDA(cudaFuncSetAttribute(maha_warp_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b), "maha attr");
      done = B / MW_WARPS * MW_WARPS;
      long long grid = done / MW_WARPS;
      const long long cap = 3LL * num_sms_proj();
      if (grid > cap) grid = cap;
      maha_warp_kernel<true><<<(unsigned)grid, MW_WARPS * 32, smem_b, st>>>(mean, mean_o, L_o, ldb_Lo, grad_out, maha, grad_mean,
                                                                             grad_L, n, (long long)done);
      TCE_CHECK_LAUNCH("maha_warp_kernel<bulk>");
      if (done == B) return TCE_OK;
    }
    const size_t per_warp = (((size_t)n * (n | 1) * sizeof(float) + 15) & ~(size_t)15) + 2 * 64 * sizeof(double);
    const size_t smem_w = MW_WARPS * per_warp;
    if (smem_w > 48 * 1024)
      TCE_CUDA(cudaFuncSetAttribute(maha_warp_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_w), "maha attr");
    const int64_t rest = B - done;                      // (the tail of a bulk launch: at most MW_WARPS - 1 episodes)
    long long grid = (rest + MW_WARPS - 1) / MW_WARPS;
    const long long cap = 6LL * num_sms_proj();
    if (grid > cap) grid = cap;
    maha_warp_kernel<false><<<(unsigned)grid, MW_WARPS * 32, smem_w, st>>>(
        mean + done * n, mean_o + done * n, L_o + done * ldb_Lo, ldb_Lo, grad_out ? grad_out + done : nullptr,
        maha ? maha + done : nullptr, grad_mean ? grad_mean + done * n : nullptr,
        grad_L ? grad_L + (size_t)done * n * n : nullptr, n, (long long)rest);
    TCE_CHECK_LAUNCH("maha_warp_kernel");
    return TCE_OK;
  }
  const size_t smem = 3 * (size_t)n * sizeof(double) + (size_t)n * (n | 1) * sizeof(float);
  if (smem > 48 * 1024)
    TCE_CUDA(cudaFuncSetAttribute(maha_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "maha attr");
  maha_kernel<<<(unsigned)B, 128, smem, (cudaStream_t)stream>>>(mean, mean_o, L_o, ldb_Lo, grad_out, maha, grad_mean,
                                                               grad_L, n);
  TCE_CHECK_LAUNCH("maha_kernel");
  return TCE_OK;
}

extern "C" int tce_gauss_maha(const float *mean, const float *mean_o, const float *L_o, int64_t ldb_Lo,
                              const double *grad_out, double *maha, float *grad_mean, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!mean || !mean_o || !L_o || B < 0 || n < 1 || n > 128 || (grad_out && !grad_mean) || (!grad_out && !maha))
    return TCE_ERR_INVALID_ARGUMENT;
  return maha_launch(mean, mean_o, L_o, ldb_Lo, grad_out, maha, grad_mean, nullptr, B, n, stream);
}

extern "C" int tce_gauss_maha_bwd_full(const float *mean, const float *mean_o, const float *L_o, int64_t ldb_Lo,
                                       const double *grad_out, float *grad_mean, float *grad_L, int64_t B, int n,
                                       void *stream) {
  if (B == 0) return TCE_OK;
  if (!mean || !mean_o || !L_o || !grad_out || (!grad_mean && !grad_L) || B < 0 || n < 1 || n > 128)
    return TCE_ERR_INVALID_ARGUMENT;
  return maha_launch(mean, mean_o, L_o, ldb_Lo, grad_out, nullptr, grad_mean, grad_L, B, n, stream);
}

extern "C" int tce_tri_inverse(const float *L, int64_t ldb, double *Linv, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!L || !Linv || B < 0) return TCE_ERR_INVALID_ARGUMENT;
  PJ_CHECK_N(n);
  const size_t smem = pj_smem(n, 2);
  int rc = set_smem(tri_inverse_kernel, smem);
  if (rc) return rc;
  tri_inverse_kernel<<<(unsigned)B, 256, smem, (cudaStream_t)stream>>>(L, ldb, Linv, n);
  TCE_CHECK_LAUNCH("tri_inverse_kernel");
  return TCE_OK;
}

extern "C" int tce_gauss_maha_shared(const float *mean, const float *mean_o, const double *Linv, const double *grad_out,
                                     double *maha, float *grad_mean, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!mean || !mean_o || !Linv || B < 0 || n < 1 || n > 128 || (grad_out && !grad_mean) || (!grad_mean && !maha))
    return TCE_ERR_INVALID_ARGUMENT;
  const int nw = 8;
  const size_t smem = sizeof(double) * ((size_t)n * (n | 1) + (size_t)nw * 2 * n);
  int rc = set_smem(maha_shared_kernel, smem);
  if (rc) return rc;
  const long long blocks = (B + nw - 1) / nw;
  maha_shared_kernel<<<(unsigned)(blocks < 148 * 2 ? blocks : 148 * 2), nw * 32, smem, (cudaStream_t)stream>>>(
      mean, mean_o, Linv, grad_out, maha, grad_mean, B, n);
  TCE_CHECK_LAUNCH("maha_shared_kernel");
  return TCE_OK;
}

extern "C" int tce_proj_mean_fwd(const float *mean, const float *mean_o, const double *mean_part, double eps,
                                 float *proj_mean, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!mean || !mean_o || !mean_part || !proj_mean || B < 0 || n < 1 || !(eps > 0)) return TCE_ERR_INVALID_ARGUMENT;
  proj_mean_fwd_kernel<<<(unsigned)((B * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(mean, mean_o, mean_part, eps,
                                                                                          proj_mean, B, n);
  TCE_CHECK_LAUNCH("proj_mean_fwd_kernel");
  return TCE_OK;
}

extern "C" int tce_proj_mean_bwd(const float *mean, const float *mean_o, const double *mean_part, double eps,
                                 const float *grad_out, float *grad_mean, double *grad_mean_part, int64_t B, int n,
                                 void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!mean || !mean_o || !mean_part || !grad_out || !grad_mean || !grad_mean_part || B < 0 || n < 1)
    return TCE_ERR_INVALID_ARGUMENT;
  proj_mean_bwd_kernel<<<(unsigned)((B * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      mean, mean_o, mean_part, eps, grad_out, grad_mean, grad_mean_part, B, n);
  TCE_CHECK_LAUNCH("proj_mean_bwd_kernel");
  return TCE_OK;
}

extern "C" int tce_proj_entropy_fwd(const float *L, const double *beta, int64_t ldb_beta, int equality, float *out,
                                    double *entropy, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!L || !beta || !out || B < 0 || n < 1) return TCE_ERR_INVALID_ARGUMENT;
  proj_entropy_kernel<<<(unsigned)B, 256, 0, (cudaStream_t)stream>>>(L, beta, ldb_beta, equality, nullptr, out, entropy, n);
  TCE_CHECK_LAUNCH("proj_entropy_kernel");
  return TCE_OK;
}

extern "C" int tce_proj_entropy_bwd(const float *L, const double *beta, int64_t ldb_beta, int equality,
                                    const float *grad_out, float *grad_L, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!L || !beta || !grad_out || !grad_L || B < 0 || n < 1) return TCE_ERR_INVALID_ARGUMENT;
  proj_entropy_kernel<<<(unsigned)B, 256, 0, (cudaStream_t)stream>>>(L, beta, ldb_beta, equality, grad_out, grad_L, nullptr, n);
  TCE_CHECK_LAUNCH("proj_entropy_kernel(bwd)");
  return TCE_OK;
}

extern "C" int tce_proj_kl_diag_fwd(const float *s, int64_t ldb_s, int64_t inc_s, const float *s_old, int64_t ldb_so,
                                    int64_t inc_so, double eps_cov, const double *beta, int64_t ldb_beta, int equality,
                                    float *out, int64_t ldb_o, int64_t inc_o, double *state, int32_t *info, int64_t B,
                                    int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!s || !s_old || !out || !state || B < 0 || n < 1 || n > 1024 || !(eps_cov > 0) || ldb_s < 0 || ldb_so < 0 ||
      ldb_beta < 0 || (ldb_o == 0 && B > 1) || ldb_o < 0)
    return TCE_ERR_INVALID_ARGUMENT;
  proj_kl_diag_kernel<<<(unsigned)((B + KD_WARPS - 1) / KD_WARPS), KD_WARPS * 32, KD_WARPS * n * sizeof(double),
                        (cudaStream_t)stream>>>(s, ldb_s, inc_s, s_old, ldb_so, inc_so, eps_cov, beta, ldb_beta, equality,
                                                nullptr, 0, 0, out, ldb_o, inc_o, state, info, B, n);
  TCE_CHECK_LAUNCH("proj_kl_diag_kernel");
  return TCE_OK;
}

extern "C" int tce_proj_kl_diag_bwd(const float *s, int64_t ldb_s, int64_t inc_s, const float *s_old, int64_t ldb_so,
                                    int64_t inc_so, const double *state, const float *grad_out, int64_t ldb_g,
                                    int64_t inc_g, float *grad_s, int64_t ldb_gs, int64_t inc_gs, int64_t B, int n,
                                    void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!s || !s_old || !state || !grad_out || !grad_s || B < 0 || n < 1 || n > 1024 || ldb_s < 0 || ldb_so < 0 ||
      ldb_g < 0 || (ldb_gs == 0 && B > 1) || ldb_gs < 0)
    return TCE_ERR_INVALID_ARGUMENT;
  proj_kl_diag_kernel<<<(unsigned)((B + KD_WARPS - 1) / KD_WARPS), KD_WARPS * 32, KD_WARPS * n * sizeof(double),
                        (cudaStream_t)stream>>>(s, ldb_s, inc_s, s_old, ldb_so, inc_so, 0.0, nullptr, 0, 0, grad_out,
                                                ldb_g, inc_g, grad_s, ldb_gs, inc_gs, const_cast<double *>(state),
                                                nullptr, B, n);
  TCE_CHECK_LAUNCH("proj_kl_diag_kernel(bwd)");
  return TCE_OK;
}

// debugging aid: SM-clock stamps of the phases of the last KL forward kernel (synchronises)
extern "C" int tce_debug_kl_phase_cycles(long long *out32) {
  if (!out32) return TCE_ERR_INVALID_ARGUMENT;
#ifdef TCE_PROFILE
  TCE_CUDA(cudaDeviceSynchronize(), "kl prof sync");
  TCE_CUDA(cudaMemcpyFromSymbol(out32, g_kl_prof, 32 * sizeof(long long)), "kl prof copy");
  float diag[8];
  TCE_CUDA(cudaMemcpyFromSymbol(diag, g_jac_diag, sizeof(diag)), "jacobi diag copy");
  for (int i = 0; i < 3; ++i) out32[12 + i] = (long long)(1e12 * (double)diag[i]);     // max cos^2 met in sweep i, x 1e12
  return TCE_OK;
#else
  return TCE_ERR_UNSUPPORTED_SHAPE;          /* library built without -DTCE_PROFILE */
#endif
}

// {M, U~, Lt^-1, Sigma_proj [B,n,n each], lam [B,n], scalars [B,KL_SC], K = Lt^-T U~ [B,n,n] (tce_proj_kl_bwd_prep)}
extern "C" size_t tce_proj_kl_save_doubles(int64_t B, int n) { return (size_t)B * (5 * (size_t)n * n + n + KL_SC); }

static int kl_fwd_launch(const float *L, const float *L_o, double eps_cov, const double *beta, int64_t ldb_beta,
                         int equality, float *proj_L, float *out_L, double *save, int32_t *info, int warm_start,
                         int64_t B, int n, void *stream, int split = 0, const float *vec = nullptr,
                         int64_t ldb_vec = 0, float min_std = 0.f, float *L_built = nullptr) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if ((!L && !vec) || (vec && !L_built) || !L_o || !proj_L || !save || B < 0 || !(eps_cov > 0))
    return TCE_ERR_INVALID_ARGUMENT;
  PJ_CHECK_N(n);
  // more matrices than SMs: two CTAs of 256 threads per SM on three buffers each (`compact`), else one of 512 on four
  const int compact = B > num_sms_proj();
  const size_t smem = pj_smem_exclusive(pj_smem(n, compact ? 3 : 4) + sizeof(double) * LA_JACOBI_SCRATCH, B);
  int rc = set_smem(proj_kl_cov_fwd_kernel, compact ? pj_smem(n, 4) + sizeof(double) * LA_JACOBI_SCRATCH : smem);
  if (rc) return rc;
  const size_t nn = (size_t)B * n * n;
  double *M = save, *U = M + nn, *Li = U + nn, *Sig = Li + nn, *lam = Sig + nn, *sc = lam + (size_t)B * n;
  proj_kl_cov_fwd_kernel<<<(unsigned)B, compact ? KL_THREADS / 2 : KL_THREADS, smem, (cudaStream_t)stream>>>(
      L, L_o, eps_cov, proj_L, M, U, Li, Sig, lam, sc, info, n, warm_start, beta, (long long)ldb_beta, equality, out_L,
      split, vec, (long long)ldb_vec, min_std, L_built, compact);
  TCE_CHECK_LAUNCH("proj_kl_cov_fwd_kernel");
  return TCE_OK;
}

static int kl_bwd_launch(const float *L, const float *proj_L, const float *grad_out, const double *save, float *grad_L,
                         int64_t B, int n, int fused_entropy, void *stream, const double *out_inv = nullptr,
                         double tr_coeff = 0.0) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!L || !proj_L || !grad_out || !save || !grad_L || B < 0) return TCE_ERR_INVALID_ARGUMENT;
  PJ_CHECK_N(n);
  const int compact = B > num_sms_proj();      // as kl_fwd_launch: two 256-thread CTAs per SM
  const size_t smem = pj_smem_exclusive(pj_smem(n, compact ? 3 : 4), B);
  int rc = set_smem(proj_kl_cov_bwd_kernel, compact ? pj_smem(n, 4) : smem);
  if (rc) return rc;
  const size_t nn = (size_t)B * n * n;
  const double *M = save, *U = M + nn, *Li = U + nn, *lam = Li + 2 * nn, *sc = lam + (size_t)B * n;
  proj_kl_cov_bwd_kernel<<<(unsigned)B, compact ? KL_THREADS / 2 : KL_THREADS, smem, (cudaStream_t)stream>>>(
      L, proj_L, grad_out, M, U, Li, lam, sc, grad_L, n, fused_entropy, out_inv, tr_coeff, compact);
  TCE_CHECK_LAUNCH("proj_kl_cov_bwd_kernel");
  return TCE_OK;
}

extern "C" int tce_proj_kl_cov_fwd(const float *L, const float *L_o, double eps_cov, float *proj_L, double *save,
                                   int32_t *info, int warm_start, int64_t B, int n, void *stream) {
  return kl_fwd_launch(L, L_o, eps_cov, nullptr, 0, 0, proj_L, nullptr, save, info, warm_start, B, n, stream);
}

extern "C" int tce_proj_kl_cov_bwd(const float *L, const float *proj_L, const float *grad_out, const double *save,
                                   float *grad_L, int64_t B, int n, void *stream) {
  return kl_bwd_launch(L, proj_L, grad_out, save, grad_L, B, n, 0, stream);
}

extern "C" int tce_proj_kl_entropy_fwd(const float *L, const float *L_o, double eps_cov, const double *beta,
                                       int64_t ldb_beta, int equality, float *proj_L, float *out_L, double *save,
                                       int32_t *info, int warm_start, int64_t B, int n, void *stream) {
  if (B != 0 && (!beta || !out_L)) return TCE_ERR_INVALID_ARGUMENT;
  return kl_fwd_launch(L, L_o, eps_cov, beta, ldb_beta, equality, proj_L, out_L, save, info, warm_start, B, n, stream);
}

/* The forward in two launches: _sigma writes the state (Sigma_proj, alpha, ...; for an inactive projection also the
 * outputs), _chol forms proj_L = chol(Sigma_proj) and out_L = alpha proj_L from it.  What only needs Sigma (stage 1
 * of the likelihood) can start after the first.                                                           */
extern "C" int tce_proj_kl_entropy_fwd_sigma(const float *L, const float *L_o, double eps_cov, const double *beta,
                                             int64_t ldb_beta, int equality, float *proj_L, float *out_L,
                                             double *save, int32_t *info, int warm_start, int64_t B, int n,
                                             void *stream) {
  if (B != 0 && !out_L) return TCE_ERR_INVALID_ARGUMENT;        /* beta == NULL: no entropy control (bound -inf) */
  return kl_fwd_launch(L, L_o, eps_cov, beta, ldb_beta, equality, proj_L, out_L, save, info, warm_start, B, n, stream,
                       1);
}

/* tce_proj_kl_entropy_fwd_sigma with the policy head fused in: the unprojected factor is built from the covariance
 * vector(s) `vec` (batch stride ldb_vec, 0 = one shared vector) inside the kernel and also written to L_built [B,n,n]. */
extern "C" int tce_proj_kl_entropy_fwd_sigma_vec(const float *vec, int64_t ldb_vec, float min_std, float *L_built,
                                                 const float *L_o, double eps_cov, const double *beta, int64_t ldb_beta,
                                                 int equality, float *proj_L, float *out_L, double *save, int32_t *info,
                                                 int warm_start, int64_t B, int n, void *stream) {
  if (B != 0 && (!out_L || !vec)) return TCE_ERR_INVALID_ARGUMENT;
  return kl_fwd_launch(nullptr, L_o, eps_cov, beta, ldb_beta, equality, proj_L, out_L, save, info, warm_start, B, n, stream,
                       1, vec, ldb_vec, min_std, L_built);
}

extern "C" int tce_proj_kl_entropy_fwd_chol(const double *save, float *proj_L, float *out_L, double *out_inv,
                                            int32_t *info, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!save || !proj_L || B < 0) return TCE_ERR_INVALID_ARGUMENT;
  PJ_CHECK_N(n);
  const size_t smem = pj_smem_exclusive(pj_smem(n, 2), B);
  int rc = set_smem(kl_chol_kernel, smem);
  if (rc) return rc;
  const size_t nn = (size_t)B * n * n;
  const double *Sig = save + 3 * nn, *sc = save + 4 * nn + (size_t)B * n;
  kl_chol_kernel<<<(unsigned)B, KL_THREADS, smem, (cudaStream_t)stream>>>(Sig, sc, proj_L, out_L, out_inv, info, n);
  TCE_CHECK_LAUNCH("kl_chol_kernel");
  return TCE_OK;
}

extern "C" int tce_proj_kl_entropy_bwd(const float *L, const float *proj_L, const float *grad_out, const double *save,
                                       float *grad_L, int64_t B, int n, void *stream) {
  return kl_bwd_launch(L, proj_L, grad_out, save, grad_L, B, n, 1, stream);
}

/* tce_proj_kl_entropy_bwd + the gradient of tr_coeff * KL_cov(N(L L^T) || N(Sigma_out detached)) (trust-region loss). */
extern "C" int tce_proj_kl_entropy_bwd_tr(const float *L, const float *proj_L, const float *grad_out, const double *save,
                                          double tr_coeff, float *grad_L, int64_t B, int n, void *stream) {
  return kl_bwd_launch(L, proj_L, grad_out, save, grad_L, B, n, 1, stream, nullptr, tr_coeff);
}

/* Backward of tce_proj_kl_cov_fwd (fused_entropy = 0) / tce_proj_kl_entropy_fwd* (fused_entropy = 1) given the gradient
 * w.r.t. the OUTPUT COVARIANCE Sigma_out = alpha^2 Sigma_proj [B,n,n] (symmetric, fp64) instead of w.r.t. its factor.  */
static int kl_bwd_sigma_launch(const float *L, const double *grad_sigma, const double *save, int fused_entropy,
                               double tr_coeff, float *grad_L, int64_t B, int n, void *stream, int use_K,
                               const float *vec = nullptr, int64_t ldb_vec = 0, float *grad_vec = nullptr) {
  if (B == 0) return TCE_OK;
  if (!L || !grad_sigma || !save || (!grad_L && !grad_vec) || (grad_vec && !vec) || B < 0) return TCE_ERR_INVALID_ARGUMENT;
  PJ_CHECK_N(n);
  const size_t smem = pj_smem_exclusive(pj_smem(n, 6), B);
  int rc = set_smem(proj_kl_cov_bwd_sigma_kernel, smem);
  if (rc) return rc;
  const size_t nn = (size_t)B * n * n;
  const double *M = save, *U = M + nn, *Li = U + nn, *Sig = Li + nn, *lam = Sig + nn, *sc = lam + (size_t)B * n;
  const double *K = use_K ? sc + (size_t)B * KL_SC : nullptr;
  proj_kl_cov_bwd_sigma_kernel<<<(unsigned)B, KL_THREADS, smem, (cudaStream_t)stream>>>(L, grad_sigma, M, U, Li, Sig, lam,
                                                                                       sc, K, grad_L, n, fused_entropy, tr_coeff,
                                                                                       vec, (long long)ldb_vec, grad_vec);
  TCE_CHECK_LAUNCH("proj_kl_cov_bwd_sigma_kernel");
  return TCE_OK;
}

extern "C" int tce_proj_kl_bwd_sigma(const float *L, const double *grad_sigma, const double *save, int fused_entropy,
                                     double tr_coeff, float *grad_L, int64_t B, int n, void *stream) {
  return kl_bwd_sigma_launch(L, grad_sigma, save, fused_entropy, tr_coeff, grad_L, B, n, stream, 0);
}

/* K = Lt^-T U~ into the state (needs only the forward's outputs); then tce_proj_kl_bwd_sigma_k is tce_proj_kl_bwd_sigma
 * with one GEMM and one load less on its critical path.  The pair must see the state of the SAME forward.      */
extern "C" int tce_proj_kl_bwd_prep(double *save, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;
  if (!save || B < 0) return TCE_ERR_INVALID_ARGUMENT;
  PJ_CHECK_N(n);
  const size_t smem = pj_smem_exclusive(pj_smem(n, 3), B);
  int rc = set_smem(kl_bwd_prep_kernel, smem);
  if (rc) return rc;
  const size_t nn = (size_t)B * n * n;
  double *U = save + nn, *Li = U + nn, *sc = save + 4 * nn + (size_t)B * n, *K = sc + (size_t)B * KL_SC;
  kl_bwd_prep_kernel<<<(unsigned)B, KL_THREADS, smem, (cudaStream_t)stream>>>(U, Li, sc, K, n);
  TCE_CHECK_LAUNCH("kl_bwd_prep_kernel");
  return TCE_OK;
}

extern "C" int tce_proj_kl_bwd_sigma_k(const float *L, const double *grad_sigma, const double *save, int fused_entropy,
                                       double tr_coeff, float *grad_L, int64_t B, int n, void *stream) {
  return kl_bwd_sigma_launch(L, grad_sigma, save, fused_entropy, tr_coeff, grad_L, B, n, stream, 1);
}

/* ..._k with the adjoint of the policy head fused in: the result is the gradient w.r.t. the covariance vector(s)
 * [B, n + n(n-1)/2] (overwritten), L = the factor tce_proj_kl_entropy_fwd_sigma_vec built from `vec`.           */
extern "C" int tce_proj_kl_bwd_sigma_k_vec(const float *L, const float *vec, int64_t ldb_vec, const double *grad_sigma,
                                           const double *save, int fused_entropy, double tr_coeff, float *grad_vec,
                                           int64_t B, int n, void *stream) {
  return kl_bwd_sigma_launch(L, grad_sigma, save, fused_entropy, tr_coeff, nullptr, B, n, stream, 1, vec, ldb_vec, grad_vec);
}

extern "C" int tce_proj_kl_entropy_bwd_inv(const float *L, const float *proj_L, const float *grad_out,
                                           const double *save, const double *out_inv, float *grad_L, int64_t B, int n,
                                           void *stream) {
  if (B != 0 && !out_inv) return TCE_ERR_INVALID_ARGUMENT;
  return kl_bwd_launch(L, proj_L, grad_out, save, grad_L, B, n, 1, stream, out_inv);
}

extern "C" int tce_proj_frob_cov_fwd(const float *L, const float *L_o, int64_t ldb_Lo, double eps_cov, float *proj_L,
                                     double *save_sc, int32_t *info, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!L || !L_o || !proj_L || !save_sc || B < 0 || !(eps_cov > 0)) return TCE_ERR_INVALID_ARGUMENT;
  PJ_CHECK_N(n);
  const size_t smem = pj_smem_exclusive(pj_smem(n, 3), B);
  int rc = set_smem(proj_frob_cov_fwd_kernel, smem);
  if (rc) return rc;
  proj_frob_cov_fwd_kernel<<<(unsigned)B, PJ_THREADS, smem, (cudaStream_t)stream>>>(L, L_o, ldb_Lo, eps_cov, proj_L, save_sc, info, n);
  TCE_CHECK_LAUNCH("proj_frob_cov_fwd_kernel");
  return TCE_OK;
}

extern "C" int tce_proj_frob_cov_bwd(const float *L, const float *L_o, int64_t ldb_Lo, double eps_cov,
                                     const float *proj_L, const float *grad_out, const double *save_sc, float *grad_L,
                                     int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!L || !L_o || !proj_L || !grad_out || !save_sc || !grad_L || B < 0) return TCE_ERR_INVALID_ARGUMENT;
  PJ_CHECK_N(n);
  const size_t smem = pj_smem_exclusive(pj_smem(n, 4), B);
  int rc = set_smem(proj_frob_cov_bwd_kernel, smem);
  if (rc) return rc;
  proj_frob_cov_bwd_kernel<<<(unsigned)B, PJ_THREADS, smem, (cudaStream_t)stream>>>(L, L_o, ldb_Lo, eps_cov, proj_L, grad_out, save_sc, grad_L, n);
  TCE_CHECK_LAUNCH("proj_frob_cov_bwd_kernel");
  return TCE_OK;
}

extern "C" int tce_proj_w2_cov_fwd(const float *L, const float *L_o, int64_t ldb_Lo, double eps_cov, int scale_prec,
                                   float *proj_L, double *save_sc, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!L || !L_o || !proj_L || !save_sc || B < 0 || !(eps_cov > 0)) return TCE_ERR_INVALID_ARGUMENT;
  PJ_CHECK_N(n);
  const size_t smem = pj_smem_exclusive(pj_smem(n, 5), B);
  int rc = set_smem(proj_w2_cov_kernel, smem);
  if (rc) return rc;
  proj_w2_cov_kernel<<<(unsigned)B, PJ_THREADS, smem, (cudaStream_t)stream>>>(L, L_o, ldb_Lo, eps_cov, scale_prec, nullptr, proj_L, save_sc, n);
  TCE_CHECK_LAUNCH("proj_w2_cov_kernel");
  return TCE_OK;
}

extern "C" int tce_proj_w2_cov_bwd(const float *L, const float *L_o, int64_t ldb_Lo, double eps_cov, int scale_prec,
                                   const float *grad_out, float *grad_L, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!L || !L_o || !grad_out || !grad_L || B < 0) return TCE_ERR_INVALID_ARGUMENT;
  PJ_CHECK_N(n);
  const size_t smem = pj_smem_exclusive(pj_smem(n, 5), B);
  int rc = set_smem(proj_w2_cov_kernel, smem);
  if (rc) return rc;
  proj_w2_cov_kernel<<<(unsigned)B, PJ_THREADS, smem, (cudaStream_t)stream>>>(L, L_o, ldb_Lo, eps_cov, scale_prec, grad_out, grad_L, nullptr, n);
  TCE_CHECK_LAUNCH("proj_w2_cov_kernel(bwd)");
  return TCE_OK;
}

extern "C" int tce_cov_distance(int kind, const float *L, const float *L_o, int64_t ldb_Lo, int scale_prec,
                                const double *grad_val, double *val, float *grad_L, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (kind < 0 || kind > 1 || !L || !L_o || B < 0 || (grad_val && !grad_L) || (!grad_val && !val))
    return TCE_ERR_INVALID_ARGUMENT;
  PJ_CHECK_N(n);
  const size_t smem = pj_smem_exclusive(pj_smem(n, 5), B);
  int rc = set_smem(cov_distance_kernel, smem);
  if (rc) return rc;
  cov_distance_kernel<<<(unsigned)B, PJ_THREADS, smem, (cudaStream_t)stream>>>(kind, L, L_o, ldb_Lo, scale_prec, grad_val, val, grad_L, n);
  TCE_CHECK_LAUNCH("cov_distance_kernel");
  return TCE_OK;
}

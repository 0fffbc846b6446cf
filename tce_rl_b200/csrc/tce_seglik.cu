// (3) TCE segment-wise trajectory likelihood, forward and backward.
// Replaces TemporalCorrelatedPolicy.log_prob (mprl/rl/policy/temporal_correlated_policy.py:104-203):
//   mp.update_inputs(times=[B,P,2], params=[B,P,Dp], params_L=[B,P,Dp,Dp]) ; get_traj_pos(flat) ;
//   get_traj_pos_cov() ; MultivariateNormal(covariance_matrix).log_prob
// without ever expanding L over the P segments (the reference recomputes L L^T per segment, :158).
//
// Math (SURVEY App. A.5 / App. F), per episode b and pair p = (t0, t1), n = 2D, rows (d, k):
//   h_pk   = scaled position basis of the ProDMP with initial conditions at time t_k      [K1]
//   Sigma  = L L^T                                                                        [Dp, Dp]
//   C[(d,k),(d',k')] = h_pk^T Sigma_{dd'} h_pk'   (+ reg on the diagonal),  Sigma_{dd'} = K1 x K1 block
//   mu[(d,k)] = xi1 y0_d + xi2 tau v0_d + h_pk . theta_d ;  r = x - mu
//   lp = -1/2 (n ln 2pi + r^T C^-1 r) - 1/2 logdet C
//   dlp/dmu = alpha = C^-1 r ; G = dlp/dC = 1/2 (alpha alpha^T - C^-1)
//   dlp/dSigma_{dd'} = sum_{p,k,k'} G[(d,k),(d',k')] h_pk h_pk'^T ;  dlp/dL = 2 (dlp/dSigma) L
//
// Precision: the quadratic forms, the residual and the per-segment Cholesky are ill conditioned
// (cond(C) ~ 1e4 because neighbouring time points are almost perfectly correlated); fp32
// accumulation there costs ~3e-4 absolute on the log-prob, above the 1e-4 parity bound.  They run in
// fp64 (B200 DFMA = 1/2 FFMA rate); the two O(Dp^3) products Sigma = L L^T and (dSigma) L run in fp32.
#include "tce_seglik.cuh"

// profiling scaffolding (-DTCE_PROFILE only): SM-clock stamps of block 0 of the last gram [0..15] / bwd [16..31] kernel
#ifdef TCE_PROFILE
__device__ long long g_sl_prof[32];
#define SL_STAMP(i) do { if (blockIdx.x == 0 && threadIdx.x == 0) g_sl_prof[i] = clock64(); } while (0)
#else
#define SL_STAMP(i) do { } while (0)
#endif

namespace {

constexpr int SL_THREADS = 256;

// ---- basis rows of the 2P time points of one episode (fp64) -----------------------------------------
// hs [2P][K1]  : scaled H_pos row of time point q = 2p + k
// xi [2P][2]   : xi1, xi2
// init_row [5 + 2 K1] as for init_row_entry.  The three regions are disjoint (__restrict__): the loop then reads the
// first five entries of init_row once per thread instead of once per basis entry.
template <int K1>
__device__ void basis_points(const TabDev &tb, double t_init, const float *__restrict__ times_b,
                             const int64_t *__restrict__ pairs, int P, double *__restrict__ hs,
                             double *__restrict__ xi, double *__restrict__ init_row) {
  if (threadIdx.x <= K1) init_row_entry<K1>(tb, t_init, threadIdx.x, init_row);
  __syncthreads();
  for (int it = threadIdx.x; it < 2 * P * (K1 + 1); it += blockDim.x) {
    const int q = it / (K1 + 1), j = it - q * (K1 + 1);       // pairs is [P][2] row-major -> q = 2p + k
    basis_entry<K1>(tb, init_row, (double)times_b[pairs[q]], j, hs + q * K1, xi + 2 * q);
  }
  __syncthreads();
}

// load the lower triangle of a dense [n, n] matrix into padded shared memory (row stride LD), upper = 0,
// rows n..NR-1 = 0
__device__ void load_lower(const float *__restrict__ L, float *Ls, int n, int NR, int LD) {
  for (int e = threadIdx.x; e < NR * LD; e += blockDim.x) {
    const int i = e / LD, c = e % LD;
    Ls[e] = (i < n && c <= i) ? L[(size_t)i * n + c] : 0.0f;
  }
}

// =====================================================================================================
// Stage 1: gram.  One CTA per episode.
// DC > 0: the number of DoF is the compile-time DC (the shapes of TCE_FOR_SHAPES); DC = 0: it is read from the tables
// (every other supported shape, K1 still a template parameter).  Only the DC = 0 instantiations take the covariance
// itself (Sigma = *sigma_scale * Sigma0, [Dp, Dp] fp64, ONE matrix for the batch) instead of its factor.
// =====================================================================================================
template <int DC, int K1>
__global__ void __launch_bounds__(SL_THREADS, DC ? 4 : 2)
seglik_gram_kernel(TabDev tb, const float *__restrict__ smp_traj, const float *__restrict__ mean,
                   const float *__restrict__ L, long long ldb_L, const float *__restrict__ times,
                   const float *__restrict__ init_time, const float *__restrict__ init_pos,
                   const float *__restrict__ init_vel, const int64_t *__restrict__ pairs, double *__restrict__ Cmat,
                   double *__restrict__ Rres, double *__restrict__ diag_max, int T, int P,
                   const double *__restrict__ Sigma0, const double *__restrict__ sigma_scale) {
  const int D = DC ? DC : tb.D;
  const int Dp = D * K1, N = 2 * D, NT = tri(N);
  const int NR = (Dp + 1) & ~1;              // Sg rows / cols (even)
  const int NR4 = (Dp + 3) & ~3;             // Ls rows padded to a multiple of 4 for the 4x4 tiles
  const int LD = NR4 + 1;                    // padded row stride of Ls (floats)
  const int SD = NR + 1;                     // row stride of Sg (doubles), odd, >= NR (tile padding)
  const bool sigma_in = DC == 0 && Sigma0 != nullptr;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double *Sg = reinterpret_cast<double *>(smem_raw);              // [NR][SD]
  double *hs = Sg + NR * SD;                                      // [2P][K1]
  double *xi = hs + 2 * P * K1;                                   // [2P][2]
  double *init_row = xi + 4 * P;                                  // [5 + 2 K1]
  float *Ls = reinterpret_cast<float *>(init_row + 5 + 2 * K1 + 1);  // [NR4][LD]
  __shared__ double s_max[SL_THREADS / 32];

  const long long b = blockIdx.x;
  const float *times_b = times + b * T;

  SL_STAMP(0);
  if (sigma_in) {
    const double sc = sigma_scale ? *sigma_scale : 1.0;
    for (int e = threadIdx.x; e < NR * NR; e += blockDim.x) {
      const int i = e / NR, c = e - i * NR;
      Sg[i * SD + c] = (i < Dp && c < Dp) ? sc * Sigma0[i * Dp + c] : 0.0;
    }
  } else {
    load_lower(L + b * ldb_L, Ls, Dp, NR4, LD);
  }
  __syncthreads();
  SL_STAMP(1);
  basis_points<K1>(tb, (double)init_time[b], times_b, pairs, P, hs, xi, init_row);   // ends with a barrier
  SL_STAMP(2);

  // ---- Sigma = L L^T (fp32 FFMA, 4x4 register tiles over the lower triangle: 8 LDS per 16 FFMA) -> Sg (fp64,
  //      mirrored).  Rows/cols are padded to NR4 (multiple of 4) with zeros.
  if (!sigma_in) {
    const int NT4 = NR4 / 4;
    for (int t = threadIdx.x; t < tri(NT4); t += blockDim.x) {
      int I, J;
      tri_decode(t, I, J);
      const float *a = Ls + (4 * I) * LD, *bq = Ls + (4 * J) * LD;
      float c[4][4];
#pragma unroll
      for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) c[x][y] = 0.f;
      const int kmax = 4 * J + 3;                                 // L[j][k] = 0 for k > j
      for (int k = 0; k <= kmax; ++k) {
        float av[4], bv[4];
#pragma unroll
        for (int x = 0; x < 4; ++x) { av[x] = a[x * LD + k]; bv[x] = bq[x * LD + k]; }
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
          for (int y = 0; y < 4; ++y) c[x][y] = fmaf(av[x], bv[y], c[x][y]);
      }
#pragma unroll
      for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) {
          const int i = 4 * I + x, j = 4 * J + y;
          if (i < NR && j < NR) { Sg[i * SD + j] = c[x][y]; Sg[j * SD + i] = c[x][y]; }
        }
    }
  }
  __syncthreads();

  SL_STAMP(3);
  // ---- C blocks (fp64).  When the pairs form a chain (second time of pair p == first time of pair p+1: the
  //      fixed-interval selection of every TCE config) the P+1 distinct time points are processed once:
  //      task (blk, u): v = Sigma_dd' h_u, then K[u,u], K[u+1,u], K[u-1,u] -> 108 instead of 198 DFMA per pair.
  double my_max = 0.0;
  double *Cb = Cmat + (size_t)b * NT * P;
  int chain_ok = 1;
  for (int pp = threadIdx.x; pp + 1 < P; pp += blockDim.x) chain_ok &= (pairs[2 * pp + 1] == pairs[2 * pp + 2]);
  const bool chained = __syncthreads_and(chain_ok) != 0;
  if (chained) {
    const int U = P + 1;
    for (int task = threadIdx.x; task < tri(D) * U; task += blockDim.x) {
      const int blk = task / U, u = task - blk * U;
      int d, dd;
      tri_decode(blk, d, dd);
      const double *hu = hs + (u < P ? 2 * u : 2 * P - 1) * K1;
      const double *hn = hs + (u + 1 < P ? 2 * (u + 1) : 2 * P - 1) * K1;      // time u + 1 (valid when u < P)
      const double *hm = hs + (u >= 1 ? 2 * (u - 1) : 0) * K1;                  // time u - 1 (valid when u >= 1)
      double h[K1];
#pragma unroll
      for (int j = 0; j < K1; ++j) h[j] = hu[j];
      double kuu = 0.0, kup = 0.0, kum = 0.0;
      const double *S = Sg + (d * K1) * SD + dd * K1;
#pragma unroll
      for (int i = 0; i < K1; ++i) {
        double v = 0.0;
#pragma unroll
        for (int j = 0; j < K1; ++j) v = fma(S[i * SD + j], h[j], v);
        kuu = fma(hu[i], v, kuu);
        kup = fma(hn[i], v, kup);
        kum = fma(hm[i], v, kum);
      }
      const int r0 = 2 * d, q0 = 2 * dd;
      if (u < P) {                      // pair p = u: time u is its first point
        Cb[(size_t)tri_idx(r0, q0) * P + u] = kuu;
        Cb[(size_t)tri_idx(r0 + 1, q0) * P + u] = kup;          // (d, t_{u+1}) x (d', t_u)
      }
      if (u >= 1) {                     // pair p = u - 1: time u is its second point
        Cb[(size_t)tri_idx(r0 + 1, q0 + 1) * P + (u - 1)] = kuu;
        if (d != dd) Cb[(size_t)tri_idx(r0, q0 + 1) * P + (u - 1)] = kum;   // (d, t_{u-1}) x (d', t_u)
      }
      if (d == dd) my_max = fmax(my_max, kuu);
    }
  } else
  for (int task = threadIdx.x; task < tri(D) * P; task += blockDim.x) {
    const int blk = task / P, p = task % P;
    int d, dd;
    tri_decode(blk, d, dd);
    double h0[K1], h1[K1];
#pragma unroll
    for (int j = 0; j < K1; ++j) { h0[j] = hs[(2 * p) * K1 + j]; h1[j] = hs[(2 * p + 1) * K1 + j]; }
    double c00 = 0.0, c01 = 0.0, c10 = 0.0, c11 = 0.0;
    const double *S = Sg + (d * K1) * SD + dd * K1;
#pragma unroll
    for (int i = 0; i < K1; ++i) {
      double t0 = 0.0, t1 = 0.0;
#pragma unroll
      for (int j = 0; j < K1; ++j) {
        const double s = S[i * SD + j];
        t0 = fma(s, h0[j], t0);
        t1 = fma(s, h1[j], t1);
      }
      c00 = fma(h0[i], t0, c00); c01 = fma(h0[i], t1, c01);
      c10 = fma(h1[i], t0, c10); c11 = fma(h1[i], t1, c11);
    }
    const int r0 = 2 * d, q0 = 2 * dd;
    Cb[(size_t)tri_idx(r0, q0) * P + p] = c00;
    Cb[(size_t)tri_idx(r0 + 1, q0) * P + p] = c10;
    Cb[(size_t)tri_idx(r0 + 1, q0 + 1) * P + p] = c11;
    if (d != dd) {
      Cb[(size_t)tri_idx(r0, q0 + 1) * P + p] = c01;
    } else {
      my_max = fmax(my_max, fmax(c00, c11));
    }
  }

  SL_STAMP(4);
  // ---- residual r = x - mu (fp64): task (p, k, d)
  double *Rb = Rres + (size_t)b * N * P;
  const double tau = tb.tau;
  for (int task = threadIdx.x; task < 2 * P * D; task += blockDim.x) {
    const int d = task / (2 * P), q = task % (2 * P);          // q = 2p + k
    const int p = q >> 1, k = q & 1;
    const double y0 = (double)init_pos[b * D + d], v0 = (double)init_vel[b * D + d] * tau;
    double mu = xi[2 * q] * y0 + xi[2 * q + 1] * v0;
    const float *th = mean + b * Dp + d * K1;
#pragma unroll
    for (int j = 0; j < K1; ++j) mu = fma(hs[q * K1 + j], (double)th[j], mu);
    if (tb.relative_goal) {
      const double shift = tb.relative_goal_scaled ? y0 : y0 / tb.scale[K1 - 1];
      mu = fma(hs[q * K1 + K1 - 1], shift, mu);
    }
    const double x = (double)smp_traj[(b * T + pairs[q]) * (2 * D) + d];
    Rb[(size_t)(2 * d + k) * P + p] = x - mu;
  }

  SL_STAMP(5);
  // ---- batch-global max of the un-regularised diagonal
  my_max = warp_max(my_max);
  if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = my_max;
  __syncthreads();
  if (threadIdx.x == 0) {
    double m = 0.0;
    for (int w = 0; w < SL_THREADS / 32; ++w) m = fmax(m, s_max[w]);
    atomic_max_pos_double(diag_max, m);
  }
  SL_STAMP(6);
}

// =====================================================================================================
// Stage 2: per-segment Cholesky / log-prob / adjoints (seg_* of tce_seglik.cuh).  One thread per (b, p).
// N <= 14: the packed triangle and z live in registers, every loop fully unrolled.  N = 16 (D = 8): its 136-entry
// triangle does not fit the 255-register budget (N = 14 spills 44 bytes already); the triangle and z live in shared
// memory as [entry][thread] (conflict free, 39 KB), the loops stay rolled (unrolled, the compiler caches the shared
// values in registers and spills ~2 KB per thread).
// =====================================================================================================
constexpr int CH_THREADS = 32;

template <int N>
__global__ void __launch_bounds__(CH_THREADS)
seglik_chol_kernel(const double *Cmat, const double *Rres, double *Gout, double *Aout, const double *__restrict__ diag_max,
                   double reg_rel, const float *__restrict__ grad_logp, const float *__restrict__ logp_old,
                   const float *__restrict__ advantage, double grad_scale, double *__restrict__ loss_acc,
                   float *__restrict__ logp, int32_t *__restrict__ info, long long BP, int P, int want_grad) {
  constexpr int NT = tri(N);
  constexpr bool IN_REGS = N <= 14;
  const long long gid = (long long)blockIdx.x * CH_THREADS + threadIdx.x;
  double loss_part = 0.0, ratio_part = 0.0;
  auto segment = [&](auto &c, auto &z) {
    const long long b = gid / P;
    const int p = (int)(gid % P);
    const double *Cb = Cmat + (size_t)b * NT * P + p;
    const double *Rb = Rres + (size_t)b * N * P + p;
    double *Gb = Gout + (size_t)b * NT * P + p;
    double *Ab = Aout + (size_t)b * N * P + p;
    const double reg = reg_rel * (*diag_max);
    seg_for<IN_REGS>(0, NT, [&](int e) { c[e] = Cb[(size_t)e * P]; });
    seg_for<IN_REGS>(0, N, [&](int i) { z[i] = Rb[(size_t)i * P]; });
    int bad;
    const double lp = seg_factor<N, IN_REGS>(c, z, reg, bad);
    if (logp) logp[gid] = (float)lp;
    if (info) info[gid] = bad;
    if (!want_grad) return;
    const SegIO io{grad_logp, logp_old, advantage, logp, info, grad_scale, reg, logp_old ? 2 : 1};
    const double g = seg_upstream(io, lp, gid, loss_part, ratio_part);
    seg_adjoint<N, IN_REGS>(c, z, g, c);
    seg_for<IN_REGS>(0, NT, [&](int e) { Gb[(size_t)e * P] = c[e]; });
    seg_for<IN_REGS>(0, N, [&](int i) { Ab[(size_t)i * P] = g * z[i]; });
  };
  if (gid < BP) {
    if constexpr (IN_REGS) {
      double c[NT], z[N];
      segment(c, z);
    } else {
      __shared__ double sm[(NT + N) * CH_THREADS];
      Strided c{sm + threadIdx.x, CH_THREADS}, z{sm + NT * CH_THREADS + threadIdx.x, CH_THREADS};
      segment(c, z);
    }
  }
  if (loss_acc) {
    loss_part = warp_sum(loss_part);
    ratio_part = warp_sum(ratio_part);
    if ((threadIdx.x & 31) == 0 && ratio_part != 0.0) {
      atomicAdd(loss_acc, loss_part);
      atomicAdd(loss_acc + 1, ratio_part);
    }
  }
}

// =====================================================================================================
// Stage 2 for N = 2 D in 18..32 (D = 9..16): one warp per segment, lane r owns row r of the packed triangle in
// registers (every loop fully unrolled over N, rows padded with zeros past the diagonal; lanes >= N idle).  The same
// arithmetic as seg_factor / seg_adjoint, in the same order where a lane owns the sum (Cholesky, forward substitution,
// X = S^-1, the rows of C^-1); |z|^2, log det and alpha = X^T z are summed across lanes (xor butterflies, so every lane
// and every call gets the same bits).  A pivot row or an X row is broadcast with __shfl_sync when the lanes below it
// need it; X is then stored in a per-warp shared triangle so that lane i can read its column X[k][i].
// G / A may overwrite C / R (the surrogate passes adj == work): a warp reads its segment before it writes it.
// =====================================================================================================
constexpr int CW_WARPS = 8;

template <int N>
__global__ void __launch_bounds__(CW_WARPS * 32)
seglik_chol_warp_kernel(const double *Cmat, const double *Rres, double *Gout, double *Aout,
                        const double *__restrict__ diag_max, double reg_rel, const float *__restrict__ grad_logp,
                        const float *__restrict__ logp_old, const float *__restrict__ advantage, double grad_scale,
                        double *__restrict__ loss_acc, float *__restrict__ logp, int32_t *__restrict__ info,
                        long long BP, int P, int want_grad) {
  constexpr int NT = tri(N);
  __shared__ double s_x[CW_WARPS][NT];
  __shared__ double s_loss[CW_WARPS][2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long gid = (long long)blockIdx.x * CW_WARPS + warp;
  double loss_part = 0.0, ratio_part = 0.0;
  if (gid < BP) {                                     // warp-uniform
    const long long b = gid / P;
    const int p = (int)(gid % P);
    const double *Cb = Cmat + (size_t)b * NT * P + p;
    const double *Rb = Rres + (size_t)b * N * P + p;
    const bool own = lane < N;
    const int row0 = own ? tri_idx(lane, 0) : 0;
    double a[N];
#pragma unroll
    for (int k = 0; k < N; ++k) a[k] = (own && k <= lane) ? Cb[(size_t)(row0 + k) * P] : 0.0;
    double z = own ? Rb[(size_t)lane * P] : 0.0;
    const double reg = reg_rel * (*diag_max);

    // ---- left-looking Cholesky C + reg I = S S^T (diagonal <- 1/S_jj), z <- S^-1 z column by column
    int bad = 0;
    double my_d = 1.0;                                // lane j: its pivot
#pragma unroll
    for (int j = 0; j < N; ++j) {
      double v = a[j];
      if (lane == j) v += reg;
#pragma unroll
      for (int k = 0; k < j; ++k) v = fma(-a[k], __shfl_sync(0xffffffffu, a[k], j), v);   // row j is final left of j
      const double dj = __shfl_sync(0xffffffffu, v, j);
      if (!(dj > 0.0) && bad == 0) bad = j + 1;
      double inv = (double)rsqrtf((float)dj);
      inv = inv * fma(-0.5 * dj, inv * inv, 1.5);
      inv = inv * fma(-0.5 * dj, inv * inv, 1.5);
      if (lane == j) { a[j] = inv; my_d = dj; z *= inv; }
      else if (own && lane > j) a[j] = v * inv;
      const double zj = __shfl_sync(0xffffffffu, z, j);
      if (own && lane > j) z = fma(-a[j], zj, z);
    }
    const double half_logdet = warp_sum(own ? 0.5 * log(my_d) : 0.0);
    const double maha = warp_sum(z * z);
    const double lp = -0.5 * ((double)N * LN_2PI + maha) - half_logdet;
    if (lane == 0) {
      if (logp) logp[gid] = (float)lp;
      if (info) info[gid] = bad;
    }
    if (want_grad) {
      const SegIO io{grad_logp, logp_old, advantage, logp, info, grad_scale, reg, logp_old ? 2 : 1};
      double lpart = 0.0, rpart = 0.0;
      const double g = seg_upstream(io, lp, gid, lpart, rpart);
      if (lane == 0) { loss_part = lpart; ratio_part = rpart; }
      // ---- X = S^-1 (right-looking: row k is final once rows < k have been folded in; a[] holds the partial sums)
#pragma unroll
      for (int k = 0; k < N; ++k) {
        if (lane == k) {
#pragma unroll
          for (int j = 0; j < k; ++j) a[j] = -a[j] * a[k];
        }
        const double s = a[k];
#pragma unroll
        for (int j = 0; j <= k; ++j) {
          const double xkj = __shfl_sync(0xffffffffu, a[j], k);
          if (own && lane > k) a[j] = j < k ? fma(s, xkj, a[j]) : s * xkj;
        }
      }
      double *xs = s_x[warp];
#pragma unroll
      for (int j = 0; j < N; ++j)
        if (own && j <= lane) xs[row0 + j] = a[j];
      __syncwarp();
      // ---- alpha = X^T z and row i of C^-1 = X^T X (sum over k >= i, ascending), G = g/2 (alpha alpha^T - C^-1)
      double alpha = 0.0, acc[N];
#pragma unroll
      for (int j = 0; j < N; ++j) acc[j] = 0.0;
#pragma unroll
      for (int k = 0; k < N; ++k) {
        const bool on = own && k >= lane;
        const double xki = on ? xs[tri_idx(k, 0) + lane] : 0.0;
        const double zk = __shfl_sync(0xffffffffu, z, k);
        if (on) alpha = fma(xki, zk, alpha);
#pragma unroll
        for (int j = 0; j <= k; ++j)
          if (on) acc[j] = fma(xki, xs[tri_idx(k, 0) + j], acc[j]);
      }
      double *Gb = Gout + (size_t)b * NT * P + p;
      double *Ab = Aout + (size_t)b * N * P + p;
      const double hg = 0.5 * g;
#pragma unroll
      for (int j = 0; j < N; ++j) {
        const double aj = __shfl_sync(0xffffffffu, alpha, j);
        if (own && j <= lane) Gb[(size_t)(row0 + j) * P] = hg * (alpha * aj - acc[j]);
      }
      if (own) Ab[(size_t)lane * P] = g * alpha;
    }
  }
  if (loss_acc) {                                     // lane 0 of each warp holds its segment's parts
    if (lane == 0) { s_loss[warp][0] = loss_part; s_loss[warp][1] = ratio_part; }
    __syncthreads();
    if (threadIdx.x == 0) {
      double l = 0.0, r = 0.0;
      for (int w = 0; w < CW_WARPS; ++w) { l += s_loss[w][0]; r += s_loss[w][1]; }
      if (r != 0.0) {
        atomicAdd(loss_acc, l);
        atomicAdd(loss_acc + 1, r);
      }
    }
  }
}

// =====================================================================================================
// Stage 3: backward accumulation.  One CTA per episode.
// =====================================================================================================
// The adjoints are staged in shared memory as fp32 [tri(2D)][P].  Above D = 8 the staging is dropped where it would
// take the CTA past BWD_SMEM_LIMIT (e.g. (16, 4) at P = 128: 270 KB alone); the kernel then reads the fp64 adjoints
// from the workspace, as the shared-covariance branch always does.  D <= 8 always stages (and refuses a P whose staging
// does not fit), as it always has.
constexpr size_t BWD_SMEM_LIMIT = 200 * 1024;
constexpr int BWD_ALWAYS_STAGED_DOF = 8;

__host__ __device__ inline size_t bwd_smem_bytes(int D, int K1, int P, bool multi, bool stage) {
  const int Dp = D * K1, N = 2 * D, NT = tri(N), NR = (Dp + 3) & ~3, LD = NR + 1;
  const int gs_need = (stage && NT * P > Dp * Dp) ? NT * P : Dp * Dp + 1;
  const size_t g = sizeof(float) * (size_t)((gs_need + 1) & ~1);
  return g + sizeof(double) * (2 * (size_t)P * K1 + 4 * (size_t)P + 5 + 2 * K1 + 1) + sizeof(float) * 2 * NR * LD +
         (multi ? sizeof(double) * tri(D) * K1 * K1 : 0) + 16;
}

// fp32 staging of the adjoints (else: fp64 reads from the workspace); a function of the shape and P only
__host__ __device__ inline bool bwd_stage(int D, int K1, int P, bool multi) {
  return D <= BWD_ALWAYS_STAGED_DOF || (!multi && bwd_smem_bytes(D, K1, P, false, true) <= BWD_SMEM_LIMIT);
}

// DC as for the gram kernel.  With dsig_part != NULL (DC = 0 only) the covariance is ONE matrix for the batch: CTA c
// owns episodes c, c + gridDim.x, ... (< B), sums upstream * d lp / d Sigma over them in that order and writes the sum
// in block layout to dsig_part[c][tri(D) K1 K1] (fp64, entry (blk, i, j) = M_{d d'}[i][j], (d, d') = tri_decode(blk));
// seglik_dsigma_sum_kernel then adds the partials in a fixed order.  No L is read and grad_L is not written.
template <int DC, int K1>
__global__ void __launch_bounds__(SL_THREADS, DC ? 4 : 2)
seglik_bwd_kernel(TabDev tb, const double *__restrict__ Gmat, const double *__restrict__ Alpha,
                  const float *__restrict__ L, long long ldb_L, const float *__restrict__ times,
                  const float *__restrict__ init_time, const int64_t *__restrict__ pairs,
                  const float *__restrict__ upstream, float *__restrict__ grad_mean, float *__restrict__ grad_L,
                  int T, int P, double *__restrict__ dsig_part, long long B) {
  const int D = DC ? DC : tb.D;
  const int Dp = D * K1, N = 2 * D, NT = tri(N);
  const int NR = (Dp + 3) & ~3;              // rows padded to a multiple of 4 for the 4x4 tiles
  const int LD = NR + 1;
  const bool multi = DC == 0 && dsig_part != nullptr;
  const bool stage = bwd_stage(D, K1, P, multi);
  const bool from_ws = multi || !stage;            // adjoints read in fp64 from the workspace
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float *Gs = reinterpret_cast<float *>(smem_raw);                // [NT][P] staged adjoints, fp32 (later: out tile)
  // Gs holds NT * P staged adjoints (and later the Dp x Dp output tile); its size is rounded UP to an even number of
  // floats so that hs is 8-byte aligned and starts after the last adjoint, as bwd_smem_bytes() sizes it.
  const int gs_need = (stage && NT * P > Dp * Dp) ? NT * P : Dp * Dp + 1;
  const int gs_floats = (gs_need + 1) & ~1;
  double *hs = reinterpret_cast<double *>(Gs + gs_floats);       // [2P][K1]
  double *xi = hs + 2 * P * K1;                                   // [2P][2]
  double *init_row = xi + 4 * P;                                  // [5 + 2 K1]
  float *Ls = reinterpret_cast<float *>(init_row + 5 + 2 * K1 + 1);  // [NR][LD]
  float *Ms = Ls + NR * LD;                                       // [NR][LD]  dlp/dSigma (symmetric)
  double *Pacc = reinterpret_cast<double *>(Ms + NR * LD);        // multi: [tri(D) K1][K1] running sum

  const float up = upstream ? *upstream : 1.0f;       // scalar gradient of the fused surrogate loss
  if (multi)
    for (int e = threadIdx.x; e < tri(D) * K1 * K1; e += blockDim.x) Pacc[e] = 0.0;
  for (long long b = blockIdx.x;; b += gridDim.x) {
  const double *Gb = Gmat + (size_t)b * NT * P;
  const double *Ab = Alpha + (size_t)b * N * P;

  SL_STAMP(16);
  if (!multi) load_lower(L + b * ldb_L, Ls, Dp, NR, LD);
  if (!from_ws)
    for (int e = threadIdx.x; e < NT * P; e += blockDim.x) Gs[e] = (float)Gb[e];
  if (!multi)
    for (int e = threadIdx.x; e < NR * LD; e += blockDim.x) Ms[e] = 0.f;
  basis_points<K1>(tb, (double)init_time[b], times + b * T, pairs, P, hs, xi, init_row);

  SL_STAMP(17);
  // ---- grad_mean[d*K1 + j] = sum_{p,k} h_pk[j] * (g alpha)[(d,k)]
  if (grad_mean) {
    for (int o = threadIdx.x; o < Dp; o += blockDim.x) {
      const int d = o / K1, j = o % K1;
      double acc = 0.0;
      for (int q = 0; q < 2 * P; ++q) acc = fma(hs[q * K1 + j], Ab[(size_t)(2 * d + (q & 1)) * P + (q >> 1)], acc);
      grad_mean[b * Dp + o] = up * (float)acc;
    }
  }
  if (!grad_L && !multi) return;

  SL_STAMP(18);
  // ---- M_{dd'}[i][:] = sum_p sum_{k,k'} G[(d,k),(d',k')] h_pk[i] h_pk'[:]   (fp64), task (blk, i)
  for (int task = threadIdx.x; task < tri(D) * K1; task += blockDim.x) {
    const int blk = task / K1, i = task % K1;
    int d, dd;
    tri_decode(blk, d, dd);
    double acc[K1];
#pragma unroll
    for (int j = 0; j < K1; ++j) acc[j] = 0.0;
    const int r0 = 2 * d, q0 = 2 * dd;
    const float *g00 = Gs + (size_t)tri_idx(r0, q0) * P;
    const float *g10 = Gs + (size_t)tri_idx(r0 + 1, q0) * P;
    const float *g11 = Gs + (size_t)tri_idx(r0 + 1, q0 + 1) * P;
    const float *g01 = (d != dd) ? Gs + (size_t)tri_idx(r0, q0 + 1) * P : g10;    // symmetric inside a diagonal block
    // multi: the adjoints are read in fp64 from the workspace.  The batch sum of a shared covariance's gradient
    // cancels (advantages of both signs) far below the size of its terms; fp32-staged adjoints then cost ~1e-3 of it.
    // (!stage: read from the workspace as well, their staging does not fit.)
    const double *G00 = Gb + (size_t)tri_idx(r0, q0) * P, *G10 = Gb + (size_t)tri_idx(r0 + 1, q0) * P;
    const double *G11 = Gb + (size_t)tri_idx(r0 + 1, q0 + 1) * P;
    const double *G01 = (d != dd) ? Gb + (size_t)tri_idx(r0, q0 + 1) * P : G10;
    for (int p = 0; p < P; ++p) {
      const double a0 = hs[(2 * p) * K1 + i], a1 = hs[(2 * p + 1) * K1 + i];
      const double w0 = from_ws ? a0 * G00[p] + a1 * G10[p] : a0 * (double)g00[p] + a1 * (double)g10[p];   // coefficient of h_p0[:]
      const double w1 = from_ws ? a0 * G01[p] + a1 * G11[p] : a0 * (double)g01[p] + a1 * (double)g11[p];   // coefficient of h_p1[:]
#pragma unroll
      for (int j = 0; j < K1; ++j)
        acc[j] = fma(w0, hs[(2 * p) * K1 + j], fma(w1, hs[(2 * p + 1) * K1 + j], acc[j]));
    }
    if (multi) {                                  // this thread owns these entries for every episode: fixed order
#pragma unroll
      for (int j = 0; j < K1; ++j) Pacc[task * K1 + j] += (double)up * acc[j];
      continue;
    }
#pragma unroll
    for (int j = 0; j < K1; ++j) {
      const float v = (float)acc[j];
      Ms[(d * K1 + i) * LD + dd * K1 + j] = v;
      if (d != dd) Ms[(dd * K1 + j) * LD + d * K1 + i] = v;
    }
  }
  __syncthreads();
  if (multi) {                                    // (the barrier above: Gs / hs are free for the next episode)
    if (b + gridDim.x < B) continue;
    for (int e = threadIdx.x; e < tri(D) * K1 * K1; e += blockDim.x)
      dsig_part[(size_t)blockIdx.x * tri(D) * K1 * K1 + e] = Pacc[e];
    return;
  }

  SL_STAMP(19);
  // ---- grad_L = 2 * tril(M L)  (fp32 FFMA, 4x4 tiles over the lower triangle), staged in the Gs buffer
  float *out = Gs;                                // [Dp][Dp] dense (the Gs region is sized for it)
  for (int e = threadIdx.x; e < Dp * Dp; e += blockDim.x) out[e] = 0.f;
  __syncthreads();
  {
    const int NT4 = NR / 4;
    for (int t = threadIdx.x; t < tri(NT4); t += blockDim.x) {
      int I, J;
      tri_decode(t, I, J);
      const float *mrow = Ms + (4 * I) * LD;
      float c[4][4];
#pragma unroll
      for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) c[x][y] = 0.f;
      for (int k = NR - 1; k >= 4 * J; --k) {            // L[k][c] = 0 for k < c; descending: lanes share k
        float mv[4], lv[4];
#pragma unroll
        for (int x = 0; x < 4; ++x) { mv[x] = mrow[x * LD + k]; lv[x] = Ls[k * LD + 4 * J + x]; }
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
          for (int y = 0; y < 4; ++y) c[x][y] = fmaf(mv[x], lv[y], c[x][y]);
      }
#pragma unroll
      for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) {
          const int i = 4 * I + x, j = 4 * J + y;
          if (i < Dp && j <= i) out[i * Dp + j] = 2.f * up * c[x][y];
        }
    }
  }
  __syncthreads();
  SL_STAMP(20);
  float *gL = grad_L + (size_t)b * Dp * Dp;
  for (int e = threadIdx.x; e < Dp * Dp; e += blockDim.x) gL[e] = out[e];
  SL_STAMP(21);
  return;
  }
}

// dS [Dp][Dp] fp64 = sum over the nparts partials of seglik_bwd_kernel (fixed order), mirrored: thread per entry.
__global__ void __launch_bounds__(256)
seglik_dsigma_sum_kernel(const double *__restrict__ part, int nparts, int D, int K1, double *__restrict__ dS) {
  const int NE = tri(D) * K1 * K1, Dp = D * K1;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= NE) return;
  double s = 0.0;
  for (int c = 0; c < nparts; ++c) s += part[(size_t)c * NE + e];
  const int blk = e / (K1 * K1), r = e - blk * K1 * K1, i = r / K1, j = r - i * K1;
  int d, dd;
  tri_decode(blk, d, dd);
  dS[(d * K1 + i) * Dp + dd * K1 + j] = s;
  if (d != dd) dS[(dd * K1 + j) * Dp + d * K1 + i] = s;
}

// grad_L [n][n] = 2 tril(dS L) for ONE shared factor L (dS symmetric, fp64): CTA per row, thread per column.
__global__ void __launch_bounds__(64)
seglik_dsigma_to_dl_kernel(const double *__restrict__ dS, const float *__restrict__ L, int n, float *__restrict__ grad_L) {
  const int i = blockIdx.x;
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    double acc = 0.0;
    if (j <= i)
      for (int k = j; k < n; ++k) acc = fma(dS[(size_t)i * n + k], (double)L[(size_t)k * n + j], acc);
    grad_L[(size_t)i * n + j] = (float)(2.0 * acc);
  }
}

// =====================================================================================================
// Diagonal covariance (std_only policies), per-episode standard deviations s [B, Dp] (strided: s[b ldb + i inc]).
// H is block diagonal per DoF, so C is block diagonal with one 2 x 2 block per (pair, DoF):
//   C_d[k,k'] = sum_j h_kj h_k'j s_{d,j}^2 + reg delta_kk',   lp = sum_d log N(r_d; 0, C_d)
// backward: d/d theta_{d,j} = sum_{p,k} h_pk[j] (g alpha)_{d,k},
//           d/d s_{d,j} = 2 s_{d,j} sum_{p,k,k'} G_d[k,k'] h_pk[j] h_pk'[j],  G = g/2 (alpha alpha^T - C^-1).
// One CTA per episode.  MODE 0: batch-global max of diag C (the regulariser seed; its own launch so that an
// all-reduce(MAX) can run in between at >1 GPU), 1: log-probs, 2: gradients.  fp64 throughout (as the dense path);
// the sums over segments run in a fixed order.
// =====================================================================================================
constexpr int SD_THREADS = 128;

template <int DC, int K1, int MODE>           // DC as for the gram kernel
__global__ void __launch_bounds__(SD_THREADS)
seglik_diag_kernel(TabDev tb, const float *__restrict__ smp_traj, const float *__restrict__ mean,
                   const float *__restrict__ s, long long ldb_s, long long inc_s, const float *__restrict__ times,
                   const float *__restrict__ init_time, const float *__restrict__ init_pos,
                   const float *__restrict__ init_vel, const int64_t *__restrict__ pairs, double *__restrict__ diag_max,
                   double reg_rel, const float *__restrict__ grad_logp, float *__restrict__ logp,
                   int32_t *__restrict__ info, float *__restrict__ grad_mean, float *__restrict__ grad_s,
                   long long ldb_gs, long long inc_gs, int T, int P) {
  const int D = DC ? DC : tb.D;
  const int Dp = D * K1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double *hs = reinterpret_cast<double *>(smem_raw);             // [2P][K1]
  double *xi = hs + 2 * P * K1;                                   // [2P][2]
  double *init_row = xi + 4 * P;                                  // [5 + 2 K1]
  double *s2 = init_row + 5 + 2 * K1;                             // [Dp] variances
  double *part = s2 + Dp;                                         // MODE 1: [D][P] log-prob parts; MODE 2: [D][5][P]
  int *bad_s = reinterpret_cast<int *>(part + (MODE == 2 ? 5 : 1) * D * P);   // MODE 1: [D][P]
  __shared__ double s_max[SD_THREADS / 32];

  const long long b = blockIdx.x;
  const float *sb = s + b * ldb_s;
  for (int i = threadIdx.x; i < Dp; i += blockDim.x) {
    const double v = sb[i * inc_s];
    s2[i] = v * v;
  }
  basis_points<K1>(tb, (double)init_time[b], times + b * T, pairs, P, hs, xi, init_row);   // ends with a barrier

  if (MODE == 0) {
    double my_max = 0.0;
    for (int task = threadIdx.x; task < 2 * P * D; task += blockDim.x) {
      const int d = task / (2 * P), q = task - d * 2 * P;
      double c = 0.0;
#pragma unroll
      for (int j = 0; j < K1; ++j) c = fma(hs[q * K1 + j] * hs[q * K1 + j], s2[d * K1 + j], c);
      my_max = fmax(my_max, c);
    }
    my_max = warp_max(my_max);
    if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = my_max;
    __syncthreads();
    if (threadIdx.x == 0) {
      double m = 0.0;
      for (int w = 0; w < SD_THREADS / 32; ++w) m = fmax(m, s_max[w]);
      atomic_max_pos_double(diag_max, m);
    }
    return;
  }

  const double reg = reg_rel * (*diag_max), tau = tb.tau;
  for (int task = threadIdx.x; task < P * D; task += blockDim.x) {
    const int d = task / P, p = task - d * P;
    const double *h0 = hs + (2 * p) * K1, *h1 = h0 + K1;
    double c00 = 0.0, c01 = 0.0, c11 = 0.0;
#pragma unroll
    for (int j = 0; j < K1; ++j) {
      const double v = s2[d * K1 + j];
      c00 = fma(h0[j] * h0[j], v, c00);
      c01 = fma(h0[j] * h1[j], v, c01);
      c11 = fma(h1[j] * h1[j], v, c11);
    }
    c00 += reg;
    c11 += reg;
    // residual r_k = x - mu (as the dense path)
    const double y0 = (double)init_pos[b * D + d], v0 = (double)init_vel[b * D + d] * tau;
    const float *th = mean + b * Dp + d * K1;
    double r[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int q = 2 * p + k;
      double mu = xi[2 * q] * y0 + xi[2 * q + 1] * v0;
#pragma unroll
      for (int j = 0; j < K1; ++j) mu = fma(hs[q * K1 + j], (double)th[j], mu);
      if (tb.relative_goal) {
        const double shift = tb.relative_goal_scaled ? y0 : y0 / tb.scale[K1 - 1];
        mu = fma(hs[q * K1 + K1 - 1], shift, mu);
      }
      r[k] = (double)smp_traj[(b * T + pairs[q]) * (2 * D) + d] - mu;
    }
    // 2 x 2 Cholesky; bad = first non-positive pivot as row (2 d + k) + 1 of the full matrix
    int bad = 0;
    if (!(c00 > 0.0)) bad = 2 * d + 1;
    const double l00 = sqrt(c00), l10 = c01 / l00, d11 = c11 - l10 * l10;
    if (!(d11 > 0.0) && bad == 0) bad = 2 * d + 2;
    const double l11 = sqrt(d11);
    const double z0 = r[0] / l00, z1 = (r[1] - l10 * z0) / l11;
    if (MODE == 1) {
      part[d * P + p] = -0.5 * (2.0 * LN_2PI + z0 * z0 + z1 * z1) - 0.5 * (log(c00) + log(d11));
      bad_s[d * P + p] = bad;
    } else {
      const double g = (double)grad_logp[b * P + p];
      const double idet = 1.0 / (c00 * c11 - c01 * c01);
      const double i00 = c11 * idet, i01 = -c01 * idet, i11 = c00 * idet;          // C^-1
      const double a0 = i00 * r[0] + i01 * r[1], a1 = i01 * r[0] + i11 * r[1];      // alpha = C^-1 r
      double *pd = part + (size_t)d * 5 * P + p;
      pd[0] = g * a0;
      pd[P] = g * a1;
      pd[2 * P] = 0.5 * g * (a0 * a0 - i00);
      pd[3 * P] = 0.5 * g * (a0 * a1 - i01);
      pd[4 * P] = 0.5 * g * (a1 * a1 - i11);
    }
  }
  __syncthreads();
  if (MODE == 1) {
    for (int p = threadIdx.x; p < P; p += blockDim.x) {
      double lp = 0.0;
      int bad = 0;
      for (int d = 0; d < D; ++d) {
        lp += part[d * P + p];
        if (bad == 0) bad = bad_s[d * P + p];
      }
      logp[b * P + p] = (float)lp;
      if (info) info[b * P + p] = bad;
    }
    return;
  }
  for (int o = threadIdx.x; o < Dp; o += blockDim.x) {
    const int d = o / K1, j = o - d * K1;
    const double *pd = part + (size_t)d * 5 * P;
    double gm = 0.0, gv = 0.0;
    for (int p = 0; p < P; ++p) {
      const double h0 = hs[(2 * p) * K1 + j], h1 = hs[(2 * p + 1) * K1 + j];
      gm = fma(h0, pd[p], fma(h1, pd[P + p], gm));
      gv = fma(h0 * h0, pd[2 * P + p], fma(2.0 * h0 * h1, pd[3 * P + p], fma(h1 * h1, pd[4 * P + p], gv)));
    }
    if (grad_mean) grad_mean[b * Dp + o] = (float)gm;
    if (grad_s) grad_s[b * ldb_gs + o * inc_gs] = (float)(2.0 * (double)sb[o * inc_s] * gv);
  }
}

// ---- host side ---------------------------------------------------------------------------------------
size_t diag_smem(int D, int K1, int P, int mode) {
  return sizeof(double) * (2 * P * K1 + 4 * P + 5 + 2 * K1 + D * K1 + (mode == 2 ? 5 : 1) * D * P) +
         (mode == 1 ? sizeof(int) * D * P : 0) + 16;
}

size_t gram_smem(int D, int K1, int P) {
  const int Dp = D * K1, NR = (Dp + 1) & ~1, NR4 = (Dp + 3) & ~3, LD = NR4 + 1, SD = NR + 1;
  return sizeof(double) * ((size_t)NR * SD + 2 * P * K1 + 4 * P + 5 + 2 * K1 + 1) + sizeof(float) * NR4 * LD + 16;
}
size_t bwd_smem(int D, int K1, int P, bool multi) {
  return bwd_smem_bytes(D, K1, P, multi, bwd_stage(D, K1, P, multi));
}

int g_sms = 0;
int sm_count() {
  if (!g_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_sms <= 0) g_sms = 148;
  }
  return g_sms;
}

// CTAs (= partials) of the shared-covariance backward: a function of B and the device only, so that the summation
// order -- and the result -- is the same on every call
int64_t shared_parts(int64_t B) {
  const int64_t cap = 2LL * sm_count();
  return B < cap ? B : cap;
}

template <int DC, int K1>
int gram_launch(const tce_tables_t *t, const float *smp_traj, const float *mean, const float *L, int64_t ldb_L,
                const double *Sigma0, const double *sigma_scale, const float *times, const float *init_time,
                const float *init_pos, const float *init_vel, const int64_t *pred_pairs, double *Cmat, double *R,
                double *diag_max, int64_t B, int64_t T, int64_t P, cudaStream_t st) {
  const size_t smem = gram_smem(t->D, K1, (int)P);
  if (smem > 200 * 1024) return TCE_ERR_UNSUPPORTED_SHAPE;
  TCE_CUDA(cudaFuncSetAttribute(seglik_gram_kernel<DC, K1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
           "gram smem attr");
  cudaFuncSetAttribute(seglik_gram_kernel<DC, K1>, cudaFuncAttributePreferredSharedMemoryCarveout,
                       cudaSharedmemCarveoutMaxShared);
  seglik_gram_kernel<DC, K1><<<(unsigned)B, SL_THREADS, smem, st>>>(
      tab_dev(t), smp_traj, mean, L, ldb_L, times, init_time, init_pos, init_vel, pred_pairs, Cmat, R, diag_max, (int)T,
      (int)P, Sigma0, sigma_scale);
  TCE_CHECK_LAUNCH("seglik_gram_kernel");
  return TCE_OK;
}

template <int DC, int K1>
int bwd_launch(const tce_tables_t *t, const double *G, const double *A, const float *L, int64_t ldb_L,
               const float *times, const float *init_time, const int64_t *pred_pairs, const float *upstream,
               float *grad_mean, float *grad_L, double *dsig_part, int64_t B, int64_t T, int64_t P, cudaStream_t st) {
  const size_t smem = bwd_smem(t->D, K1, (int)P, dsig_part != nullptr);
  if (smem > BWD_SMEM_LIMIT) return TCE_ERR_UNSUPPORTED_SHAPE;
  TCE_CUDA(cudaFuncSetAttribute(seglik_bwd_kernel<DC, K1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
           "bwd smem attr");
  cudaFuncSetAttribute(seglik_bwd_kernel<DC, K1>, cudaFuncAttributePreferredSharedMemoryCarveout,
                       cudaSharedmemCarveoutMaxShared);
  const int64_t grid = dsig_part ? shared_parts(B) : B;
  seglik_bwd_kernel<DC, K1><<<(unsigned)grid, SL_THREADS, smem, st>>>(
      tab_dev(t), G, A, L, ldb_L, times, init_time, pred_pairs, upstream, grad_mean, grad_L, (int)T, (int)P, dsig_part,
      (long long)B);
  TCE_CHECK_LAUNCH("seglik_bwd_kernel");
  return TCE_OK;
}

template <int DC, int K1, int MODE>
int diag_launch(const tce_tables_t *t, const float *smp_traj, const float *mean, const float *s, int64_t ldb_s,
                int64_t inc_s, const float *times, const float *init_time, const float *init_pos,
                const float *init_vel, const int64_t *pred_pairs, double *diag_max, double reg_rel,
                const float *grad_logp, float *logp, int32_t *info, float *grad_mean, float *grad_s, int64_t ldb_gs,
                int64_t inc_gs, int64_t B, int64_t T, int64_t P, cudaStream_t st) {
  const size_t smem = diag_smem(t->D, K1, (int)P, MODE);
  if (smem > 200 * 1024) return TCE_ERR_UNSUPPORTED_SHAPE;
  if (smem > 48 * 1024)
    TCE_CUDA(cudaFuncSetAttribute(seglik_diag_kernel<DC, K1, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)smem), "diag smem attr");
  seglik_diag_kernel<DC, K1, MODE><<<(unsigned)B, SD_THREADS, smem, st>>>(
      tab_dev(t), smp_traj, mean, s, ldb_s, inc_s, times, init_time, init_pos, init_vel, pred_pairs, diag_max, reg_rel,
      grad_logp, logp, info, grad_mean, grad_s, ldb_gs, inc_gs, (int)T, (int)P);
  TCE_CHECK_LAUNCH("seglik_diag_kernel");
  return TCE_OK;
}

}  // namespace

// (D, K1) combinations with instantiations specialised on D (and the fused / uniform-grid kernels of
// tce_seglik_fused.cu); every other shape with 1 <= D <= 16, 2 <= K1 <= 16, D K1 <= 64 runs the DC = 0 instantiations
#define TCE_FOR_SHAPES(X) X(7, 9) X(4, 9) X(7, 4) X(3, 4) X(2, 3)

static bool shape_supported(const tce_tables_t *t) {
  return t->D >= 1 && t->D <= TCE_MAX_DOF && t->K1 >= 2 && t->K1 <= TCE_MAX_K1 && t->D * t->K1 <= TCE_MAX_DP;
}

// The diagonal likelihood keeps no Dp x Dp matrix: its work per (pair, DoF) depends on K1 only, so it takes every
// shape the tables accept
static bool diag_shape_supported(const tce_tables_t *t) {
  return t->D >= 1 && t->D <= TCE_MAX_DOF && t->K1 >= 2 && t->K1 <= TCE_MAX_K1 && t->D * t->K1 <= TCE_MAX_TABLE_DP;
}

extern "C" int tce_seglik_compiled(const tce_tables_t *t) {
  if (!t) return TCE_ERR_INVALID_ARGUMENT;
#define X(Dv, Kv) if (t->D == Dv && t->K1 == Kv) return 1;
  TCE_FOR_SHAPES(X)
#undef X
  return shape_supported(t) ? 0 : TCE_ERR_UNSUPPORTED_SHAPE;
}

// debugging aid: SM-clock stamps of block 0 of the last gram ([0..6]) and bwd ([16..21]) launches (synchronises)
extern "C" int tce_debug_seglik_phase_cycles(long long *out32) {
  if (!out32) return TCE_ERR_INVALID_ARGUMENT;
#ifdef TCE_PROFILE
  TCE_CUDA(cudaDeviceSynchronize(), "seglik prof sync");
  TCE_CUDA(cudaMemcpyFromSymbol(out32, g_sl_prof, 32 * sizeof(long long)), "seglik prof copy");
  return TCE_OK;
#else
  return TCE_ERR_UNSUPPORTED_SHAPE;          /* library built without -DTCE_PROFILE */
#endif
}

extern "C" size_t tce_seglik_work_bytes(const tce_tables_t *t, int64_t B, int64_t P) {
  if (!t || B < 0 || P < 0) return 0;
  const size_t N = 2 * (size_t)t->D;
  return sizeof(double) * (size_t)B * (size_t)P * (N * (N + 1) / 2 + N);
}

static inline double *work_R(const tce_tables_t *t, void *work, int64_t B, int64_t P) {
  const size_t N = 2 * (size_t)t->D;
  return (double *)work + (size_t)B * (size_t)P * (N * (N + 1) / 2);
}

static int seglik_gram_any(const tce_tables_t *t, const float *smp_traj, const float *mean, const float *L,
                           int64_t ldb_L, const double *Sigma0, const double *sigma_scale, const float *times,
                           const float *init_time, const float *init_pos, const float *init_vel,
                           const int64_t *pred_pairs, void *work, double *diag_max, int64_t B, int64_t T, int64_t P,
                           void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!t || !smp_traj || !mean || (Sigma0 ? false : !L) || !times || !init_time || !init_pos || !init_vel ||
      !pred_pairs || !work || !diag_max || B < 0 || T < 1 || P < 1 || P > 4096)
    return TCE_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
  double *Cmat = (double *)work, *R = work_R(t, work, B, P);
  if (!Sigma0) {
#define X(Dv, Kv)                                                                                                  \
    if (t->D == Dv && t->K1 == Kv)                                                                                 \
      return gram_launch<Dv, Kv>(t, smp_traj, mean, L, ldb_L, nullptr, nullptr, times, init_time, init_pos,       \
                                 init_vel, pred_pairs, Cmat, R, diag_max, B, T, P, st);
    TCE_FOR_SHAPES(X)
#undef X
  }
  if (!shape_supported(t)) return TCE_ERR_UNSUPPORTED_SHAPE;
  TCE_DISPATCH_K1(t->K1, return (gram_launch<0, K1>(t, smp_traj, mean, L, ldb_L, Sigma0, sigma_scale, times, init_time,
                                                    init_pos, init_vel, pred_pairs, Cmat, R, diag_max, B, T, P, st)));
  return TCE_ERR_UNSUPPORTED_SHAPE;
}

extern "C" int tce_seglik_gram(const tce_tables_t *t, const float *smp_traj, const float *mean, const float *L,
                               int64_t ldb_L, const float *times, const float *init_time, const float *init_pos,
                               const float *init_vel, const int64_t *pred_pairs, void *work, double *diag_max,
                               int64_t B, int64_t T, int64_t P, void *stream) {
  if (B != 0 && !L) return TCE_ERR_INVALID_ARGUMENT;
  return seglik_gram_any(t, smp_traj, mean, L, ldb_L, nullptr, nullptr, times, init_time, init_pos, init_vel,
                         pred_pairs, work, diag_max, B, T, P, stream);
}

extern "C" int tce_seglik_gram_sigma(const tce_tables_t *t, const float *smp_traj, const float *mean,
                                     const double *Sigma0, const double *sigma_scale, const float *times,
                                     const float *init_time, const float *init_pos, const float *init_vel,
                                     const int64_t *pred_pairs, void *work, double *diag_max, int64_t B, int64_t T,
                                     int64_t P, void *stream) {
  if (B != 0 && !Sigma0) return TCE_ERR_INVALID_ARGUMENT;
  return seglik_gram_any(t, smp_traj, mean, nullptr, 0, Sigma0, sigma_scale, times, init_time, init_pos, init_vel,
                         pred_pairs, work, diag_max, B, T, P, stream);
}

extern "C" int tce_seglik_chol(const tce_tables_t *t, const void *work, void *adj, const double *diag_max, double reg_rel,
                               const float *grad_logp, const float *logp_old, const float *advantage,
                               double grad_scale, double *loss_acc, float *logp, int32_t *info, int64_t B,
                               int64_t P, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!t || !work || !diag_max || B < 0 || P < 1) return TCE_ERR_INVALID_ARGUMENT;
  if (logp_old && !advantage) return TCE_ERR_INVALID_ARGUMENT;
  if (!shape_supported(t)) return TCE_ERR_UNSUPPORTED_SHAPE;
  cudaStream_t st = (cudaStream_t)stream;
  const double *Cmat = (const double *)work, *R = work_R(t, const_cast<void *>(work), B, P);
  double *G = (double *)adj, *A = adj ? work_R(t, adj, B, P) : nullptr;
  const long long BP = (long long)B * P;
  const unsigned grid = (unsigned)((BP + CH_THREADS - 1) / CH_THREADS);
  const int want_grad = (grad_logp != nullptr) || (logp_old != nullptr);
  if (want_grad && !adj) return TCE_ERR_INVALID_ARGUMENT;
  const unsigned wgrid = (unsigned)((BP + CW_WARPS - 1) / CW_WARPS);
  switch (t->D) {
#define Y(Dv)                                                                                                  \
  case Dv:                                                                                                     \
    seglik_chol_kernel<2 * Dv><<<grid, CH_THREADS, 0, st>>>(Cmat, R, G, A, diag_max, reg_rel, grad_logp, logp_old, \
                                                            advantage, grad_scale, loss_acc, logp, info, BP,   \
                                                            (int)P, want_grad);                                \
    break;
    Y(1) Y(2) Y(3) Y(4) Y(5) Y(6) Y(7) Y(8)
#undef Y
#define W(Dv)                                                                                                  \
  case Dv:                                                                                                     \
    seglik_chol_warp_kernel<2 * Dv><<<wgrid, CW_WARPS * 32, 0, st>>>(Cmat, R, G, A, diag_max, reg_rel, grad_logp, \
                                                                     logp_old, advantage, grad_scale, loss_acc,   \
                                                                     logp, info, BP, (int)P, want_grad);          \
    break;
    W(9) W(10) W(11) W(12) W(13) W(14) W(15) W(16)
#undef W
    default: return TCE_ERR_UNSUPPORTED_SHAPE;
  }
  TCE_CHECK_LAUNCH("seglik_chol_kernel");
  return TCE_OK;
}

extern "C" int tce_seglik_bwd(const tce_tables_t *t, const void *work, const float *L, int64_t ldb_L,
                              const float *times, const float *init_time, const int64_t *pred_pairs,
                              const float *upstream, float *grad_mean, float *grad_L, int64_t B, int64_t T,
                              int64_t P, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!t || !work || !L || !times || !init_time || !pred_pairs || B < 0 || T < 1 || P < 1)
    return TCE_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
  const double *G = (const double *)work, *A = work_R(t, const_cast<void *>(work), B, P);
#define X(Dv, Kv)                                                                                                \
  if (t->D == Dv && t->K1 == Kv)                                                                                 \
    return bwd_launch<Dv, Kv>(t, G, A, L, ldb_L, times, init_time, pred_pairs, upstream, grad_mean, grad_L,       \
                              nullptr, B, T, P, st);
  TCE_FOR_SHAPES(X)
#undef X
  if (!shape_supported(t)) return TCE_ERR_UNSUPPORTED_SHAPE;
  TCE_DISPATCH_K1(t->K1, return (bwd_launch<0, K1>(t, G, A, L, ldb_L, times, init_time, pred_pairs, upstream, grad_mean,
                                                   grad_L, nullptr, B, T, P, st)));
  return TCE_ERR_UNSUPPORTED_SHAPE;
}

extern "C" size_t tce_seglik_shared_part_doubles(const tce_tables_t *t, int64_t B) {
  if (!t || B < 1 || !shape_supported(t)) return 0;
  const int64_t Dp = (int64_t)t->D * t->K1;
  return (size_t)(shared_parts(B) * (int64_t)(t->D * (t->D + 1) / 2) * t->K1 * t->K1 + Dp * Dp);
}

extern "C" int tce_seglik_bwd_shared(const tce_tables_t *t, const void *work, const float *L, const float *times,
                                     const float *init_time, const int64_t *pred_pairs, const float *upstream,
                                     float *grad_mean, double *part, float *grad_L, double *grad_sigma, int64_t B,
                                     int64_t T, int64_t P, void *stream) {
  if (!t || !part || (!grad_L && !grad_sigma) || (grad_L && !L) || B < 1 || T < 1 || P < 1 || !work || !times ||
      !init_time || !pred_pairs)
    return TCE_ERR_INVALID_ARGUMENT;
  if (!shape_supported(t)) return TCE_ERR_UNSUPPORTED_SHAPE;
  cudaStream_t st = (cudaStream_t)stream;
  const double *G = (const double *)work, *A = work_R(t, const_cast<void *>(work), B, P);
  const int D = t->D, K1 = t->K1, Dp = D * K1, NE = tri(D) * K1 * K1;
  const int64_t nparts = shared_parts(B);
  double *dS = grad_sigma ? grad_sigma : part + (size_t)nparts * NE;
  int rc = TCE_ERR_UNSUPPORTED_SHAPE;
  TCE_DISPATCH_K1(K1, rc = (bwd_launch<0, K1>(t, G, A, nullptr, 0, times, init_time, pred_pairs, upstream, grad_mean,
                                              nullptr, part, B, T, P, st)));
  if (rc != TCE_OK) return rc;
  seglik_dsigma_sum_kernel<<<(NE + 255) / 256, 256, 0, st>>>(part, (int)nparts, D, K1, dS);
  TCE_CHECK_LAUNCH("seglik_dsigma_sum_kernel");
  if (grad_L) {
    seglik_dsigma_to_dl_kernel<<<Dp, 64, 0, st>>>(dS, L, Dp, grad_L);
    TCE_CHECK_LAUNCH("seglik_dsigma_to_dl_kernel");
  }
  return TCE_OK;
}

template <int MODE>
static int seglik_diag_launch(const tce_tables_t *t, const float *smp_traj, const float *mean, const float *s,
                              int64_t ldb_s, int64_t inc_s, const float *times, const float *init_time,
                              const float *init_pos, const float *init_vel, const int64_t *pred_pairs, double *diag_max,
                              double reg_rel, const float *grad_logp, float *logp, int32_t *info, float *grad_mean,
                              float *grad_s, int64_t ldb_gs, int64_t inc_gs, int64_t B, int64_t T, int64_t P,
                              void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!t || !s || !times || !init_time || !pred_pairs || !diag_max || B < 0 || T < 1 || P < 1 || P > 4096 ||
      ldb_s < 0)
    return TCE_ERR_INVALID_ARGUMENT;
  if (MODE >= 1 && (!smp_traj || !mean || !init_pos || !init_vel)) return TCE_ERR_INVALID_ARGUMENT;
  if (MODE == 1 && !logp) return TCE_ERR_INVALID_ARGUMENT;
  if (MODE == 2 && (!grad_logp || (!grad_mean && !grad_s) || (grad_s && (ldb_gs < 0 || (ldb_gs == 0 && B > 1)))))
    return TCE_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
#define X(Dv, Kv)                                                                                                  \
  if (t->D == Dv && t->K1 == Kv)                                                                                   \
    return diag_launch<Dv, Kv, MODE>(t, smp_traj, mean, s, ldb_s, inc_s, times, init_time, init_pos, init_vel,     \
                                     pred_pairs, diag_max, reg_rel, grad_logp, logp, info, grad_mean, grad_s,      \
                                     ldb_gs, inc_gs, B, T, P, st);
  TCE_FOR_SHAPES(X)
#undef X
  if (!diag_shape_supported(t)) return TCE_ERR_UNSUPPORTED_SHAPE;
  TCE_DISPATCH_K1(t->K1, return (diag_launch<0, K1, MODE>(t, smp_traj, mean, s, ldb_s, inc_s, times, init_time,
                                                          init_pos, init_vel, pred_pairs, diag_max, reg_rel, grad_logp,
                                                          logp, info, grad_mean, grad_s, ldb_gs, inc_gs, B, T, P, st)));
  return TCE_ERR_UNSUPPORTED_SHAPE;
}

extern "C" int tce_seglik_diag_max(const tce_tables_t *t, const float *s, int64_t ldb_s, int64_t inc_s,
                                   const float *times, const float *init_time, const int64_t *pred_pairs,
                                   double *diag_max, int64_t B, int64_t T, int64_t P, void *stream) {
  return seglik_diag_launch<0>(t, nullptr, nullptr, s, ldb_s, inc_s, times, init_time, nullptr, nullptr, pred_pairs,
                               diag_max, 0.0, nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0, B, T, P, stream);
}

extern "C" int tce_seglik_diag_fwd(const tce_tables_t *t, const float *smp_traj, const float *mean, const float *s,
                                   int64_t ldb_s, int64_t inc_s, const float *times, const float *init_time,
                                   const float *init_pos, const float *init_vel, const int64_t *pred_pairs,
                                   const double *diag_max, double reg_rel, float *logp, int32_t *info, int64_t B,
                                   int64_t T, int64_t P, void *stream) {
  return seglik_diag_launch<1>(t, smp_traj, mean, s, ldb_s, inc_s, times, init_time, init_pos, init_vel, pred_pairs,
                               const_cast<double *>(diag_max), reg_rel, nullptr, logp, info, nullptr, nullptr, 0, 0, B,
                               T, P, stream);
}

extern "C" int tce_seglik_diag_bwd(const tce_tables_t *t, const float *smp_traj, const float *mean, const float *s,
                                   int64_t ldb_s, int64_t inc_s, const float *times, const float *init_time,
                                   const float *init_pos, const float *init_vel, const int64_t *pred_pairs,
                                   const double *diag_max, double reg_rel, const float *grad_logp, float *grad_mean,
                                   float *grad_s, int64_t ldb_gs, int64_t inc_gs, int64_t B, int64_t T, int64_t P,
                                   void *stream) {
  return seglik_diag_launch<2>(t, smp_traj, mean, s, ldb_s, inc_s, times, init_time, init_pos, init_vel, pred_pairs,
                               const_cast<double *>(diag_max), reg_rel, grad_logp, nullptr, nullptr, grad_mean, grad_s,
                               ldb_gs, inc_gs, B, T, P, stream);
}

// (3) TCE segment-wise trajectory likelihood, fused: ONE persistent kernel per call does
//     basis rows -> gram C = H Sigma H^T -> per-segment Cholesky / log-prob (+ fused surrogate) -> adjoints ->
//     grad_mean and d logp / d Sigma (accumulated in the CTA over its episodes) [-> grad_L per episode],
// with no HBM workspace.  Replaces the staged kernels of tce_seglik.cu (gram / chol / bwd / dsigma_to_dl, ~80 MB of
// fp64 round trips at B = 1024) on the product path; the staged entry points stay for cross-checks.
// Reference semantics: TemporalCorrelatedPolicy.log_prob, mprl/rl/policy/temporal_correlated_policy.py:104-203
// (mp.update_inputs + get_traj_pos(flat) + get_traj_pos_cov + MultivariateNormal(covariance_matrix).log_prob) and
// TemporalCorrelatedAgent.surrogate_loss, mprl/rl/agent/temporal_correlated_agent.py:718-739.
//
// The batch-global regulariser reg = reg_rel * max_{b,p,i} C_bp[i,i] (mp_pytorch get_traj_pos_cov) is produced by a
// diagonal-only pre-pass (tce_seglik_diagmax, ~20 % of the gram work) BEFORE the fused kernel, so the
// all-reduce(MAX) of a multi-GPU run sits between two launches and nothing else splits the computation.
//
// Work decomposition of the fused kernel (one CTA of 256 threads per SM, E episodes per iteration, S = E * P):
//   phase 0  basis rows of the distinct time points (fp64 table lerps) and residuals r = x - mu  -> smem
//   phase 1  gram: warp task = (DoF block (d, d'), 32 (episode, time point) items): v = Sigma_dd' h (Sigma block rows
//            are warp-uniform -> broadcast 128-bit shared loads), then h.v, h_next.v, h_prev.v  -> C [entry][slot] smem
//   phase 2  thread per segment: packed 14 x 14 triangle in REGISTERS (compile-time indices), Cholesky with
//            reciprocal pivots, forward substitution, log-prob, upstream gradient (given or fused surrogate),
//            C^-1 via the explicit inverse of the factor, G = g/2 (alpha alpha^T - C^-1) in place
//   phase 3  thread per (episode, DoF block): 81 register accumulators,
//            dSigma_dd' = sum_q w_q h_q^T, w_q = (G-weighted) combination of h_q, h_next, h_prev  (chained pairs: the
//            P + 1 distinct time points are visited once); grad_mean by thread per (episode, parameter)
//   shared covariance : dSigma summed over the CTA's episodes in smem (fp32), ONE partial per CTA -> global;
//                       tce_seglik_dsigma_reduce sums the <= 148 partials and applies grad_L = 2 tril(dSigma L) once
//   per-episode factor: Sigma_b = L_b L_b^T (fp32 4x4 register tiles) before phase 1 of each episode and
//                       grad_L_b = 2 tril(dSigma_b L_b) after phase 3, both in shared memory.
//
// Uniform time grid (all episodes share init_time and hence the basis rows) + shared covariance -- the situation of
// every shipped TCE config -- makes C_p, its factor and its inverse identical for all episodes:
// tce_seglik_uniform_* evaluate them once and reduce the per-episode work to a residual, two 14 x 14 triangular
// products and a rank-1 update (~50x fewer FLOPs).
#include "tce_seglik.cuh"

namespace {

constexpr int FT = 256;                      // threads of the fused kernel

// ---- links between time points and pairs -------------------------------------------------------------
// chained pairs (second time of pair p == first time of pair p + 1: the fixed-interval selection of every TCE
// config): nq = P + 1 distinct points, point q is the first point of pair q (q < P) and the second of pair q - 1.
// otherwise: nq = 2 P points, q = 2 p + k.
struct Links { int pf, ps, nxt, prv; };    // pair where q is first / second (-1: none), the partner points
__device__ __forceinline__ Links links(int chained, int q, int P) {
  Links l;
  if (chained) { l.pf = q < P ? q : -1; l.ps = q >= 1 ? q - 1 : -1; l.nxt = q + 1; l.prv = q - 1; }
  else if (q & 1) { l.pf = -1; l.ps = q >> 1; l.nxt = q; l.prv = q - 1; }
  else { l.pf = q >> 1; l.ps = -1; l.nxt = q + 1; l.prv = q; }
  return l;
}
__device__ __forceinline__ long long point_time_index(const int64_t *__restrict__ pairs, int chained, int q, int P) {
  if (!chained) return pairs[q];
  return q < P ? pairs[2 * q] : pairs[2 * P - 1];
}
__device__ __forceinline__ int point_of(int chained, int p, int k) { return chained ? p + k : 2 * p + k; }

__device__ int block_chained(const int64_t *__restrict__ pairs, int P) {
  int ok = 1;
  for (int pp = threadIdx.x; pp + 1 < P; pp += blockDim.x) ok &= (pairs[2 * pp + 1] == pairs[2 * pp + 2]);
  return __syncthreads_and(ok) != 0;
}

// phase 2 of the fused kernel for one segment: column `slot` of C [NT][S] / r [N][S] in shared memory -> log-prob,
// upstream gradient, adjoints written back in place.  Deliberately NOT inlined: the packed triangle needs ~240
// registers; as a separate function it gets the whole register file instead of competing with the kernel's
// loop state (inlined: 4-6 KB of spill traffic per thread).
template <int N>
__device__ __noinline__ void segment_thread(double *Ccol, double *Rcol, int S, long long gid, const SegIO &io,
                                            double &loss_part, double &ratio_part) {
  // The packed triangle (N (N + 1) / 2 doubles = 210 registers at N = 14) lives in registers with compile-time
  // indices; the residual / z / alpha vector stays in the thread's shared-memory column (Rcol, stride S): with it in
  // registers too the function spills ~1.4 KB per thread, and with ~215 KB of the SM's L1 configured as shared
  // memory those spills go to L2.  G goes straight to the column of C.
  constexpr int NT = tri(N);
  double c[NT];
  Strided z{Rcol, S}, G{Ccol, S};
#pragma unroll
  for (int t = 0; t < NT; ++t) c[t] = Ccol[(size_t)t * S];
  int bad;
  const double lp = seg_factor<N, true>(c, z, io.reg, bad);
  if (io.logp) io.logp[gid] = (float)lp;
  if (io.info) io.info[gid] = bad;
  if (io.grad_mode == 0) return;
  const double g = seg_upstream(io, lp, gid, loss_part, ratio_part);
  seg_adjoint<N, true>(c, z, g, G);
#pragma unroll
  for (int i = 0; i < N; ++i) z[i] = g * z[i];
}

// phase 3b of the fused kernel: dSigma_dd'[i][j] = sum_q w_q[i] h_q[j] for one (episode, DoF block), 81 register
// accumulators; G = the episode's adjoints (rows of C [NT][S], first pair at G).  Called by ALL threads (it contains
// the barrier after which the C region -- which `dst` aliases -- may be overwritten); not inlined for the same
// reason as segment_thread.  ld == 0: dst[K1*K1] contiguous; else row stride ld and, if dst_t, the transposed block.
template <int K1>
__device__ __noinline__ void dsigma_block_store(bool own, const double *G, int S, const double *hm_e, int bd, int bdd,
                                                int chained, int nq, int P, float *dst, int ld, float *dst_t) {
  double acc[K1 * K1];
  if (own) {
#pragma unroll
    for (int t = 0; t < K1 * K1; ++t) acc[t] = 0.0;
    const int r0 = 2 * bd, q0 = 2 * bdd;
    const double *g00 = G + (size_t)tri_idx(r0, q0) * S, *g10 = G + (size_t)tri_idx(r0 + 1, q0) * S;
    const double *g11 = G + (size_t)tri_idx(r0 + 1, q0 + 1) * S;
    const double *g01 = (bd != bdd) ? G + (size_t)tri_idx(r0, q0 + 1) * S : g10;    // symmetric in a diagonal block
    for (int q = 0; q < nq; ++q) {
      const Links lk = links(chained, q, P);
      const double *hq = hm_e + q * K1;
      double cs = 0.0, cn = 0.0, cp = 0.0;               // coefficients of h_q, h_next, h_prev on the row side
      if (lk.pf >= 0) { cs += g00[lk.pf]; cn = g10[lk.pf]; }
      if (lk.ps >= 0) { cs += g11[lk.ps]; cp = g01[lk.ps]; }
      const double *hn = hm_e + (lk.pf >= 0 ? lk.nxt : q) * K1, *hp = hm_e + (lk.ps >= 0 ? lk.prv : q) * K1;
      double h[K1], w[K1];
#pragma unroll
      for (int j = 0; j < K1; ++j) h[j] = hq[j];
#pragma unroll
      for (int i = 0; i < K1; ++i) w[i] = fma(cs, h[i], fma(cn, hn[i], cp * hp[i]));
#pragma unroll
      for (int i = 0; i < K1; ++i)
#pragma unroll
        for (int j = 0; j < K1; ++j) acc[i * K1 + j] = fma(w[i], h[j], acc[i * K1 + j]);
    }
  }
  __syncthreads();
  if (own) {
    if (ld == 0) {
#pragma unroll
      for (int t = 0; t < K1 * K1; ++t) dst[t] = (float)acc[t];
    } else {
#pragma unroll
      for (int i = 0; i < K1; ++i)
#pragma unroll
        for (int j = 0; j < K1; ++j) {
          const float v = (float)acc[i * K1 + j];
          dst[i * ld + j] = v;
          if (dst_t) dst_t[j * ld + i] = v;
        }
    }
  }
}

// ---- pre-pass workspace: per episode  hm [nq][K1] | r [N][P]  (doubles) -------------------------------------------
__host__ __device__ inline size_t pre_doubles(int nq, int K1, int N, int P) { return (size_t)nq * K1 + (size_t)N * P; }

// ---- shared-memory layout of the fused kernel (host + device) ------------------------------------------------
template <int D, int K1>
struct FusedLayout {
  static constexpr int Dp = D * K1, N = 2 * D, NT = tri(N), NB = tri(D);
  static constexpr int KP = (K1 + 1) & ~1;                  // padded row of a Sigma block (16-byte aligned rows)
  static constexpr int NR4 = (Dp + 3) & ~3, LD = NR4 + 1;   // fp32 staging of a factor: [NR4][LD]
  static constexpr int IR = (5 + 2 * K1 + 1) & ~1;          // init row doubles (even)
  static constexpr int LCNT = (NR4 * NR4 + FT - 1) / FT;    // factor elements per thread (register prefetch)
  size_t sblk, dsacc, cs, rs, hm, total;
  int E, S, SP, nq;        // SP: row stride (doubles) of the [entry][slot] arrays, odd -> rows fall into distinct banks
  __host__ __device__ FusedLayout(int E_, int P, int chained) {
    E = E_; S = E * P; SP = S | 1; nq = chained ? P + 1 : 2 * P;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += (bytes + 15) & ~(size_t)15; return at; };
    const size_t sb = sizeof(double) * NB * K1 * KP, ls = sizeof(float) * NR4 * LD;
    sblk = take(sb > ls ? sb : ls);
    dsacc = take(sizeof(float) * NB * K1 * K1);
    // C [NT][SP]; after phase 3 the region is scratch: dSigma_b [E][NR4][LD] or block partials [E][NB][K1 K1] (fp32)
    const size_t c1 = sizeof(double) * NT * SP, c2 = sizeof(float) * (size_t)E * NR4 * LD;
    const size_t c3 = sizeof(float) * (size_t)E * NB * K1 * K1, c12 = c1 > c2 ? c1 : c2;
    cs = take(c12 > c3 ? c12 : c3);
    rs = take(sizeof(double) * N * SP);
    hm = take(sizeof(double) * (size_t)E * nq * K1);
    total = o;
  }
};

// Sigma block (d, dd), d >= dd, entry (i, j): Sblk[tri_idx(d, dd)][i][j] with row stride KP
template <int K1, int KP>
__device__ __forceinline__ double *sblk_at(double *Sblk, int blk) { return Sblk + (size_t)blk * K1 * KP; }

// store an element (i >= j) of the symmetric Sigma into the block layout (diagonal blocks are stored full)
template <int K1, int KP>
__device__ __forceinline__ void sblk_store(double *Sblk, int i, int j, double v) {
  const int d = i / K1, dd = j / K1, ii = i - d * K1, jj = j - dd * K1;
  double *blk = sblk_at<K1, KP>(Sblk, tri_idx(d, dd));
  blk[ii * KP + jj] = v;
  if (d == dd) blk[jj * KP + ii] = v;
}

// load the lower triangle of a dense [n, n] fp32 matrix into padded shared memory, zero elsewhere
__device__ __forceinline__ void stage_lower(const float *__restrict__ L, float *Ls, int n, int NR, int LD) {
  for (int e0 = threadIdx.x; e0 < NR * NR; e0 += 4 * FT) {
    float v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int e = e0 + u * FT, i = e / NR, c = e - i * NR;
      v[u] = (e < NR * NR && i < n && c <= i) ? L[(size_t)i * n + c] : 0.0f;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int e = e0 + u * FT, i = e / NR, c = e - i * NR;
      if (e < NR * NR) Ls[i * LD + c] = v[u];
    }
  }
}

// Sigma = L L^T: one 4x4 register tile of the lower triangle per thread (tri(NR4 / 4) <= 256 tiles), then -> Sblk fp64
template <int D, int K1>
__device__ __forceinline__ void sigma_from_factor(const float *Ls, double *Sblk) {
  using FL = FusedLayout<D, K1>;
  constexpr int NT4 = FL::NR4 / 4, LD = FL::LD, Dp = FL::Dp;
  static_assert(tri(NT4) <= FT, "one tile per thread");
  float c[4][4];
  int I = 0, J = 0;
  const bool act = threadIdx.x < tri(NT4);
  if (act) {
    tri_decode(threadIdx.x, I, J);
    const float *a = Ls + (4 * I) * LD, *bq = Ls + (4 * J) * LD;
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
      for (int y = 0; y < 4; ++y) c[x][y] = 0.f;
    const int kmax = 4 * J + 3;
    for (int k = 0; k <= kmax; ++k) {
      float av[4], bv[4];
#pragma unroll
      for (int x = 0; x < 4; ++x) { av[x] = a[x * LD + k]; bv[x] = bq[x * LD + k]; }
#pragma unroll
      for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) c[x][y] = fmaf(av[x], bv[y], c[x][y]);
    }
  }
  __syncthreads();                                         // everybody has read Ls: the region becomes Sblk
  if (act) {
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
      for (int y = 0; y < 4; ++y) {
        const int i = 4 * I + x, j = 4 * J + y;
        if (i < Dp && j <= i) sblk_store<K1, FL::KP>(Sblk, i, j, (double)c[x][y]);
      }
  }
  __syncthreads();
}

// one gram item: DoF block (d, dd), point q of episode slot e -> up to four entries of C (chained: of two pairs)
template <int D, int K1>
__device__ __forceinline__ double gram_item(const double *__restrict__ Sb, const double *__restrict__ hm_e, int q,
                                            const Links &lk, int d, int dd, double *CS, int S, int slot0) {
  constexpr int KP = FusedLayout<D, K1>::KP;
  double h[K1], v[K1];
  const double *hq = hm_e + q * K1;
#pragma unroll
  for (int j = 0; j < K1; ++j) h[j] = hq[j];
#pragma unroll
  for (int i = 0; i < K1; ++i) {
    const double *row = Sb + i * KP;
    double a0 = 0.0, a1 = 0.0;
#pragma unroll
    for (int j = 0; j + 1 < K1; j += 2) {
      const double2 s = *reinterpret_cast<const double2 *>(row + j);
      a0 = fma(s.x, h[j], a0);
      a1 = fma(s.y, h[j + 1], a1);
    }
    if (K1 & 1) a0 = fma(row[K1 - 1], h[K1 - 1], a0);
    v[i] = a0 + a1;
  }
  double kuu = 0.0;
#pragma unroll
  for (int i = 0; i < K1; ++i) kuu = fma(h[i], v[i], kuu);
  const int r0 = 2 * d, q0 = 2 * dd;
  if (lk.pf >= 0) {                          // q is the first point of pair pf; partner = its second point
    const double *hn = hm_e + lk.nxt * K1;
    double kup = 0.0;
#pragma unroll
    for (int i = 0; i < K1; ++i) kup = fma(hn[i], v[i], kup);
    CS[(size_t)tri_idx(r0, q0) * S + slot0 + lk.pf] = kuu;
    CS[(size_t)tri_idx(r0 + 1, q0) * S + slot0 + lk.pf] = kup;          // (d, second) x (dd, first)
  }
  if (lk.ps >= 0) {                          // q is the second point of pair ps; partner = its first point
    CS[(size_t)tri_idx(r0 + 1, q0 + 1) * S + slot0 + lk.ps] = kuu;
    if (d != dd) {
      const double *hp = hm_e + lk.prv * K1;
      double kum = 0.0;
#pragma unroll
      for (int i = 0; i < K1; ++i) kum = fma(hp[i], v[i], kum);
      CS[(size_t)tri_idx(r0, q0 + 1) * S + slot0 + lk.ps] = kum;        // (d, first) x (dd, second)
    }
  }
  return kuu;
}

// a factor's elements of this thread, in registers (global loads all in flight at once)
template <int NR4, int CNT>
__device__ __forceinline__ void prefetch_lower(const float *__restrict__ L, int n, float (&v)[CNT]) {
#pragma unroll
  for (int u = 0; u < CNT; ++u) {
    const int e = threadIdx.x + u * FT, i = e / NR4, c = e - i * NR4;
    v[u] = (e < NR4 * NR4 && i < n && c <= i) ? L[(size_t)i * n + c] : 0.0f;
  }
}
template <int NR4, int CNT>
__device__ __forceinline__ void commit_lower(const float (&v)[CNT], float *Ls, int LD) {
#pragma unroll
  for (int u = 0; u < CNT; ++u) {
    const int e = threadIdx.x + u * FT, i = e / NR4, c = e - i * NR4;
    if (e < NR4 * NR4) Ls[i * LD + c] = v[u];
  }
}

// =====================================================================================================
// pre-pass: basis rows, residuals, max_{b, p, i} C_bp[i, i] -> *diag_max (atomic max on a positive double)
// =====================================================================================================
constexpr int PT = 128;
template <int D, int K1, bool SIGMA_IN>
__global__ void __launch_bounds__(PT)
seglik_prepass_kernel(TabDev tb, const float *__restrict__ smp_traj, const float *__restrict__ mean,
                      const float *__restrict__ L, long long ldb_L, const double *__restrict__ Sigma0,
                      const double *__restrict__ sigma_scale, const float *__restrict__ times,
                      const float *__restrict__ init_time, const float *__restrict__ init_pos,
                      const float *__restrict__ init_vel, const int64_t *__restrict__ pairs,
                      double *__restrict__ pre, double *__restrict__ diag_max, long long B, int T, int P,
                      int chained) {
  using FL = FusedLayout<D, K1>;
  constexpr int Dp = FL::Dp, N = FL::N, IR = FL::IR;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double *Sd = reinterpret_cast<double *>(smem_raw);                   // [D][K1][K1] diagonal blocks of Sigma
  double *hm = Sd + D * K1 * K1;                                       // [nq][K1]
  double *xi = hm + (size_t)2 * P * K1;                                // [nq][2]
  double *init_row = xi + (size_t)4 * P;                               // [IR]
  float *Lsm = reinterpret_cast<float *>(init_row + IR);               // [Dp][Dp + 1] (factor input only)
  __shared__ double s_max[PT / 32];
  if (chained && !block_chained(pairs, P)) return;                     // wrong claim: the fused kernel reports it
  const int nq = chained ? P + 1 : 2 * P;
  const size_t pstride = pre_doubles(nq, K1, N, P);
  const bool shared_cov = SIGMA_IN || ldb_L == 0;
  const double tau = tb.tau;
  double my_max = 0.0;
  auto load_diag_blocks = [&](long long b) {
    if (SIGMA_IN) {
      const double sc = sigma_scale ? *sigma_scale : 1.0;
      for (int e = threadIdx.x; e < D * K1 * K1; e += PT) {
        const int d = e / (K1 * K1), r = e - d * K1 * K1, i = r / K1, j = r - i * K1;
        Sd[e] = sc * Sigma0[(size_t)(d * K1 + i) * Dp + d * K1 + j];
      }
    } else {
      // (L L^T)_dd: rows d*K1+i and d*K1+j over the first d*K1 + min(i,j) + 1 columns, factor staged in smem
      const float *Lb = L + b * ldb_L;
      for (int e0 = threadIdx.x; e0 < Dp * Dp; e0 += 8 * PT) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = (e0 + u * PT < Dp * Dp) ? Lb[e0 + u * PT] : 0.f;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int e = e0 + u * PT;
          if (e < Dp * Dp) Lsm[(e / Dp) * (Dp + 1) + (e % Dp)] = v[u];
        }
      }
      __syncthreads();
      for (int e = threadIdx.x; e < D * K1 * K1; e += PT) {
        const int d = e / (K1 * K1), r = e - d * K1 * K1, i = r / K1, j = r - i * K1;
        const float *a = Lsm + (d * K1 + i) * (Dp + 1), *bq = Lsm + (d * K1 + j) * (Dp + 1);
        const int kmax = d * K1 + (i < j ? i : j);
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        int k = 0;
        for (; k + 3 <= kmax; k += 4) {
          a0 = fmaf(a[k], bq[k], a0); a1 = fmaf(a[k + 1], bq[k + 1], a1);
          a2 = fmaf(a[k + 2], bq[k + 2], a2); a3 = fmaf(a[k + 3], bq[k + 3], a3);
        }
        for (; k <= kmax; ++k) a0 = fmaf(a[k], bq[k], a0);
        Sd[e] = (double)((a0 + a1) + (a2 + a3));
      }
    }
  };
  if (shared_cov) load_diag_blocks(0);
  for (long long b = blockIdx.x; b < B; b += gridDim.x) {
    __syncthreads();
    if (!shared_cov) load_diag_blocks(b);
    if (threadIdx.x <= K1) init_row_entry<K1>(tb, (double)init_time[b], threadIdx.x, init_row);
    __syncthreads();
    for (int it = threadIdx.x; it < nq * (K1 + 1); it += PT) {
      const int q = it / (K1 + 1), j = it - q * (K1 + 1);
      basis_entry<K1>(tb, init_row, (double)times[b * T + point_time_index(pairs, chained, q, P)], j, hm + q * K1,
                      xi + 2 * q);
    }
    __syncthreads();
    double *pb = pre + (size_t)b * pstride;
    for (int it = threadIdx.x; it < nq * K1; it += PT) pb[it] = hm[it];
    double *rb = pb + (size_t)nq * K1;
    for (int it = threadIdx.x; it < P * N; it += PT) {                 // residual r = x - mu, task (d, p, k)
      const int d = it / (2 * P), pk = it - d * 2 * P, p = pk >> 1, k = pk & 1;
      const int q = point_of(chained, p, k);
      const double *hq = hm + q * K1;
      const double y0 = (double)init_pos[b * D + d], v0 = (double)init_vel[b * D + d] * tau;
      double mu = xi[2 * q] * y0 + xi[2 * q + 1] * v0;
      const float *th = mean + b * Dp + d * K1;
#pragma unroll
      for (int j = 0; j < K1; ++j) mu = fma(hq[j], (double)th[j], mu);
      if (tb.relative_goal) {
        const double shift = tb.relative_goal_scaled ? y0 : y0 / tb.scale[K1 - 1];
        mu = fma(hq[K1 - 1], shift, mu);
      }
      const double x = (double)smp_traj[(b * T + pairs[2 * p + k]) * (2 * D) + d];
      rb[(size_t)(2 * d + k) * P + p] = x - mu;
    }
    for (int it = threadIdx.x; it < D * nq; it += PT) {                // diagonal of C
      const int d = it / nq, q = it - d * nq;
      const double *S = Sd + d * K1 * K1, *h = hm + q * K1;
      double acc = 0.0;
#pragma unroll
      for (int i = 0; i < K1; ++i) {
        double v = 0.0;
#pragma unroll
        for (int j = 0; j < K1; ++j) v = fma(S[i * K1 + j], h[j], v);
        acc = fma(h[i], v, acc);
      }
      my_max = fmax(my_max, acc);
    }
  }
  my_max = warp_max(my_max);
  if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = my_max;
  __syncthreads();
  if (threadIdx.x == 0) {
    double m = 0.0;
    for (int w = 0; w < PT / 32; ++w) m = fmax(m, s_max[w]);
    atomic_max_pos_double(diag_max, m);
  }
}

// =====================================================================================================
// fused kernel
// =====================================================================================================
// grad_mode: 0 = log-probs only, 1 = upstream gradient grad_logp [B, P], 2 = fused surrogate
//            (g = -exp(lp - lp_old) * adv * grad_scale, loss_acc[0] += sum g, loss_acc[1] += sum ratio * grad_scale)
template <int D, int K1, bool SIGMA_IN>
__global__ void __launch_bounds__(FT, 1)
seglik_fused_kernel(const double *__restrict__ pre, const float *__restrict__ L, long long ldb_L,
                    const double *__restrict__ Sigma0, const double *__restrict__ sigma_scale,
                    const int64_t *__restrict__ pairs, const double *__restrict__ diag_max, double reg_rel,
                    int grad_mode, const float *__restrict__ grad_logp, const float *__restrict__ logp_old,
                    const float *__restrict__ advantage, double grad_scale, double *__restrict__ loss_acc,
                    float *__restrict__ logp, int32_t *__restrict__ info, float *__restrict__ grad_mean,
                    float *__restrict__ grad_L, float *__restrict__ dsigma_part, long long B, int P, int E,
                    int chained) {
  using FL = FusedLayout<D, K1>;
  constexpr int Dp = FL::Dp, N = FL::N, NT = FL::NT, NB = FL::NB, KP = FL::KP, NR4 = FL::NR4, LD = FL::LD;
  constexpr int LCNT = FL::LCNT;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // `chained` is the caller's claim (the shared-memory layout was sized with it): refuse a wrong one
  if (chained && !block_chained(pairs, P)) {
    if (blockIdx.x == 0 && threadIdx.x == 0 && info) info[0] = -7;
    return;
  }
  const FL lay(E, P, chained);
  const int S = lay.SP, nq = lay.nq;     // S: row stride of CS / RS
  double *Sblk = reinterpret_cast<double *>(smem_raw + lay.sblk);
  float *Ls = reinterpret_cast<float *>(smem_raw + lay.sblk);          // aliases Sblk (per-episode factor staging)
  float *dsacc = reinterpret_cast<float *>(smem_raw + lay.dsacc);      // [NB][K1][K1] running dSigma of this CTA
  double *CS = reinterpret_cast<double *>(smem_raw + lay.cs);          // [NT][S]
  float *dSb = reinterpret_cast<float *>(smem_raw + lay.cs);           // aliases CS after phase 3
  double *RS = reinterpret_cast<double *>(smem_raw + lay.rs);          // [N][S]
  double *hm = reinterpret_cast<double *>(smem_raw + lay.hm);          // [E][nq][K1]
  __shared__ double s_red[2 * (FT / 32)];

  const bool shared_cov = SIGMA_IN || ldb_L == 0;
  const bool want_grad = grad_mode != 0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const double reg = reg_rel * (*diag_max);
  const size_t pstride = pre_doubles(nq, K1, N, P);
  double loss_part = 0.0, ratio_part = 0.0;
  if (blockIdx.x == 0 && threadIdx.x == 0 && dsigma_part && want_grad)   // ticket of the reduce kernel (see there)
    *reinterpret_cast<unsigned int *>(dsigma_part + ((size_t)gridDim.x + 1) * NB * K1 * K1) = 0u;

  // ---- the shared covariance is staged once per CTA ----------------------------------------------------
  if (shared_cov) {
    if (SIGMA_IN) {
      const double sc = sigma_scale ? *sigma_scale : 1.0;
      for (int e0 = threadIdx.x; e0 < Dp * Dp; e0 += 4 * FT) {
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = (e0 + u * FT < Dp * Dp) ? Sigma0[e0 + u * FT] : 0.0;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int e = e0 + u * FT, i = e / Dp, j = e - i * Dp;
          if (e < Dp * Dp && j <= i) sblk_store<K1, KP>(Sblk, i, j, sc * v[u]);
        }
      }
      __syncthreads();
    } else {
      float lr[LCNT];
      prefetch_lower<NR4, LCNT>(L, Dp, lr);
      commit_lower<NR4, LCNT>(lr, Ls, LD);
      __syncthreads();
      sigma_from_factor<D, K1>(Ls, Sblk);
    }
    if (want_grad && dsigma_part)
      for (int e = threadIdx.x; e < NB * K1 * K1; e += FT) dsacc[e] = 0.f;
  }

  const long long n_groups = (B + E - 1) / E;
  for (long long grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
    const long long b0 = grp * E;
    const int Ec = (int)((B - b0) < E ? (B - b0) : E);
    __syncthreads();
    // ---- phase 0: basis rows and residuals of this group from the pre-pass workspace ---------------------------
    {
      const double *pg = pre + (size_t)b0 * pstride;        // the group's episodes are contiguous in `pre`
      const int total = Ec * (int)pstride, hme = nq * K1;
      for (int it0 = threadIdx.x; it0 < total; it0 += 6 * FT) {
        double v[6];
#pragma unroll
        for (int u = 0; u < 6; ++u) v[u] = (it0 + u * FT < total) ? pg[it0 + u * FT] : 0.0;
#pragma unroll
        for (int u = 0; u < 6; ++u) {
          const int it = it0 + u * FT;
          if (it < total) {
            const int e = it / (int)pstride, r = it - e * (int)pstride;
            if (r < hme) hm[(size_t)e * hme + r] = v[u];
            else { const int rr = r - hme, i = rr / P, p = rr - i * P; RS[(size_t)i * S + e * P + p] = v[u]; }
          }
        }
      }
    }
    __syncthreads();
    // ---- phase 1: gram ------------------------------------------------------------------------------------
    if (shared_cov) {
      const int items = Ec * nq, chunks = (items + 31) >> 5;
      for (int wt = warp; wt < NB * chunks; wt += FT / 32) {
        const int blk = wt / chunks, item = (wt - blk * chunks) * 32 + lane;
        if (item < items) {
          int d, dd;
          tri_decode(blk, d, dd);
          const int e = item / nq, q = item - e * nq;
          gram_item<D, K1>(sblk_at<K1, KP>(Sblk, blk), hm + (size_t)e * nq * K1, q, links(chained, q, P), d, dd, CS, S,
                           e * P);
        }
      }
    } else {
      float lr[LCNT];
      prefetch_lower<NR4, LCNT>(L + b0 * ldb_L, Dp, lr);
      for (int e = 0; e < Ec; ++e) {
        __syncthreads();                                     // the previous episode's gram has read Sblk
        commit_lower<NR4, LCNT>(lr, Ls, LD);
        if (e + 1 < Ec) prefetch_lower<NR4, LCNT>(L + (b0 + e + 1) * ldb_L, Dp, lr);   // in flight during the gram
        __syncthreads();
        sigma_from_factor<D, K1>(Ls, Sblk);
        const int chunks = (nq + 31) >> 5;
        for (int wt = warp; wt < NB * chunks; wt += FT / 32) {
          const int blk = wt / chunks, q = (wt - blk * chunks) * 32 + lane;
          if (q < nq) {
            int d, dd;
            tri_decode(blk, d, dd);
            gram_item<D, K1>(sblk_at<K1, KP>(Sblk, blk), hm + (size_t)e * nq * K1, q, links(chained, q, P), d, dd, CS,
                             S, e * P);
          }
        }
      }
    }
    __syncthreads();
    // ---- phase 2: thread per segment ---------------------------------------------------------------------
    if ((int)threadIdx.x < Ec * P) {
      const int slot = threadIdx.x, e = slot / P, p = slot - e * P;
      SegIO io{grad_logp, logp_old, advantage, logp, info, grad_scale, reg, grad_mode};
      segment_thread<N>(CS + slot, RS + slot, S, (b0 + e) * P + p, io, loss_part, ratio_part);
    }
    if (!want_grad) continue;
    __syncthreads();
    // ---- phase 3a: grad_mean[d K1 + j] = sum_{p, k} h_{p,k}[j] (g alpha)[(d, k)] ---------------------------------
    if (grad_mean) {
      for (int it = threadIdx.x; it < Ec * Dp; it += FT) {
        const int e = it / Dp, o = it - e * Dp, d = o / K1, j = o - d * K1;
        const double *hm_e = hm + (size_t)e * nq * K1;
        const double *a0 = RS + (size_t)(2 * d) * S + e * P, *a1 = RS + (size_t)(2 * d + 1) * S + e * P;
        double acc0 = 0.0, acc1 = 0.0;
        for (int p = 0; p < P; ++p) {
          acc0 = fma(hm_e[point_of(chained, p, 0) * K1 + j], a0[p], acc0);
          acc1 = fma(hm_e[point_of(chained, p, 1) * K1 + j], a1[p], acc1);
        }
        grad_mean[(b0 + e) * Dp + o] = (float)(acc0 + acc1);
      }
    }
    if (!grad_L && !dsigma_part) continue;
    // ---- phase 3b: thread per (episode, DoF block) -> fp32 blocks in the (now free) C region ------------------------
    const bool own = (int)threadIdx.x < Ec * NB;
    int be = 0, bblk = 0, bd = 0, bdd = 0;
    if (own) {
      be = threadIdx.x / NB; bblk = threadIdx.x - be * NB;
      tri_decode(bblk, bd, bdd);
    }
    if (shared_cov) {
      // block partials [E][NB][K1 K1], then dsacc += their sum over the episodes of this group
      dsigma_block_store<K1>(own, CS + be * P, S, hm + (size_t)be * nq * K1, bd, bdd, chained, nq, P,
                             dSb + ((size_t)be * NB + bblk) * (K1 * K1), 0, nullptr);
      __syncthreads();
      for (int e2 = threadIdx.x; e2 < NB * K1 * K1; e2 += FT) {
        float s = dsacc[e2];
        for (int e = 0; e < Ec; ++e) s += dSb[(size_t)e * NB * K1 * K1 + e2];
        dsacc[e2] = s;
      }
    } else {
      // dSigma_b dense symmetric fp32 [E][NR4][LD], then grad_L_b = 2 tril(dSigma_b L_b) per episode
      float *M0 = dSb + (size_t)be * NR4 * LD;
      dsigma_block_store<K1>(own, CS + be * P, S, hm + (size_t)be * nq * K1, bd, bdd, chained, nq, P,
                             M0 + (bd * K1) * LD + bdd * K1, LD, bd != bdd ? M0 + (bdd * K1) * LD + bd * K1 : nullptr);
      if (NR4 > Dp) {                                        // zero padding rows / columns
        for (int it = threadIdx.x; it < Ec * (NR4 - Dp) * NR4; it += FT) {
          const int e = it / ((NR4 - Dp) * NR4), r = it - e * (NR4 - Dp) * NR4, a = Dp + r / NR4, c = r - (r / NR4) * NR4;
          float *M = dSb + (size_t)e * NR4 * LD;
          M[a * LD + c] = 0.f;
          M[c * LD + a] = 0.f;
        }
      }
      float lr[LCNT];
      prefetch_lower<NR4, LCNT>(L + b0 * ldb_L, Dp, lr);
      for (int e = 0; e < Ec; ++e) {
        __syncthreads();                                     // dSigma blocks written / previous product done with Ls
        commit_lower<NR4, LCNT>(lr, Ls, LD);
        if (e + 1 < Ec) prefetch_lower<NR4, LCNT>(L + (b0 + e + 1) * ldb_L, Dp, lr);
        __syncthreads();
        const float *M = dSb + (size_t)e * NR4 * LD;
        float *gL = grad_L + (size_t)(b0 + e) * Dp * Dp;
        constexpr int NT4 = NR4 / 4;
        if (threadIdx.x < tri(NT4)) {
          int I, J;
          tri_decode(threadIdx.x, I, J);
          const float *mrow = M + (4 * I) * LD;
          float c4[4][4];
#pragma unroll
          for (int x = 0; x < 4; ++x)
#pragma unroll
            for (int y = 0; y < 4; ++y) c4[x][y] = 0.f;
          for (int k = NR4 - 1; k >= 4 * J; --k) {           // L[k][c] = 0 for k < c
            float mv[4], lv[4];
#pragma unroll
            for (int x = 0; x < 4; ++x) { mv[x] = mrow[x * LD + k]; lv[x] = Ls[k * LD + 4 * J + x]; }
#pragma unroll
            for (int x = 0; x < 4; ++x)
#pragma unroll
              for (int y = 0; y < 4; ++y) c4[x][y] = fmaf(mv[x], lv[y], c4[x][y]);
          }
#pragma unroll
          for (int x = 0; x < 4; ++x)
#pragma unroll
            for (int y = 0; y < 4; ++y) {
              const int i = 4 * I + x, j = 4 * J + y;
              if (i < Dp && j < Dp) gL[(size_t)i * Dp + j] = j <= i ? 2.f * c4[x][y] : 0.f;
            }
        } else {
          // threads without a tile zero the strictly-upper tiles (grad_L is dense [Dp, Dp], upper = 0)
          for (int t = threadIdx.x - tri(NT4); t < NT4 * NT4; t += FT - tri(NT4)) {
            const int I = t / NT4, J = t - I * NT4;
            if (J > I)
              for (int x = 0; x < 4; ++x)
                for (int y = 0; y < 4; ++y) {
                  const int i = 4 * I + x, j = 4 * J + y;
                  if (i < Dp && j < Dp) gL[(size_t)i * Dp + j] = 0.f;
                }
          }
        }
      }
    }
  }
  // ---- epilogue --------------------------------------------------------------------------------------------
  __syncthreads();
  if (shared_cov && want_grad && dsigma_part) {
    float *out = dsigma_part + (size_t)blockIdx.x * NB * K1 * K1;
    for (int e = threadIdx.x; e < NB * K1 * K1; e += FT) out[e] = dsacc[e];
  }
  if (grad_mode == 2 && loss_acc) {
    loss_part = warp_sum(loss_part);
    ratio_part = warp_sum(ratio_part);
    if (lane == 0) { s_red[2 * warp] = loss_part; s_red[2 * warp + 1] = ratio_part; }
    __syncthreads();
    if (threadIdx.x == 0) {
      double a = 0.0, r = 0.0;
      for (int w = 0; w < FT / 32; ++w) { a += s_red[2 * w]; r += s_red[2 * w + 1]; }
      if (r != 0.0) { atomicAdd(loss_acc, a); atomicAdd(loss_acc + 1, r); }
    }
  }
}

// dense symmetric dSigma (fp32, smem M [NR4][LD], zero padded) and a shared factor (smem Ls) -> grad_L = 2 tril(M L)
// (lower, upper = 0) with 2x2 register tiles; any block size.
template <int D, int K1>
__device__ __forceinline__ void dl_from_dsigma(const float *M, const float *Ls, float *__restrict__ grad_L) {
  using FL = FusedLayout<D, K1>;
  constexpr int Dp = FL::Dp, NR4 = FL::NR4, LD = FL::LD, NT2 = NR4 / 2;
  for (int t = threadIdx.x; t < tri(NT2); t += blockDim.x) {
    int I, J;
    tri_decode(t, I, J);
    const float *m0 = M + (2 * I) * LD, *m1 = m0 + LD;
    float c00 = 0.f, c01 = 0.f, c10 = 0.f, c11 = 0.f;
    for (int k = 2 * J; k < NR4; ++k) {
      const float a0 = m0[k], a1 = m1[k], l0 = Ls[k * LD + 2 * J], l1 = Ls[k * LD + 2 * J + 1];
      c00 = fmaf(a0, l0, c00); c01 = fmaf(a0, l1, c01);
      c10 = fmaf(a1, l0, c10); c11 = fmaf(a1, l1, c11);
    }
    const int i0 = 2 * I, j0 = 2 * J;
    if (i0 < Dp && j0 < Dp) grad_L[(size_t)i0 * Dp + j0] = 2.f * c00;
    if (i0 < Dp && j0 + 1 < Dp) grad_L[(size_t)i0 * Dp + j0 + 1] = j0 + 1 <= i0 ? 2.f * c01 : 0.f;
    if (i0 + 1 < Dp && j0 < Dp) grad_L[(size_t)(i0 + 1) * Dp + j0] = 2.f * c10;
    if (i0 + 1 < Dp && j0 + 1 < Dp) grad_L[(size_t)(i0 + 1) * Dp + j0 + 1] = 2.f * c11;
  }
  for (int e = threadIdx.x; e < Dp * Dp; e += blockDim.x) {  // the part above the diagonal tiles
    const int i = e / Dp, j = e - i * Dp;
    if (j / 2 > i / 2) grad_L[e] = 0.f;
  }
}

// unpack block-layout dSigma values [NB][K1][K1] (global, written by other CTAs: read through L2) into M
template <int D, int K1>
__device__ __forceinline__ void unpack_blocks(const float *blocks, float scale, float *M) {
  using FL = FusedLayout<D, K1>;
  constexpr int NB = FL::NB, LD = FL::LD, NE = NB * K1 * K1;
  for (int e = threadIdx.x; e < NE; e += blockDim.x) {
    const float v = scale * __ldcg(blocks + e);
    const int blk = e / (K1 * K1), r = e - blk * K1 * K1, i = r / K1, j = r - i * K1;
    int d, dd;
    tri_decode(blk, d, dd);
    M[(d * K1 + i) * LD + dd * K1 + j] = v;
    if (d != dd) M[(dd * K1 + j) * LD + d * K1 + i] = v;
  }
}

// =====================================================================================================
// reduce of the per-CTA dSigma partials (block layout) + grad_L = 2 tril(dSigma L) for ONE shared factor
// =====================================================================================================
// part: [nparts][NE] partials | [NE] sum (written here) | ticket (uint32, zeroed by the fused kernel), NE = NB K1 K1.
// CTA c sums entries [32 c, 32 c + 32) with 8 threads per entry (fixed order: deterministic); the last CTA to finish
// (ticket) forms grad_L / grad_sigma from the full sum.
constexpr int RT = 256;
template <int D, int K1>
__global__ void __launch_bounds__(RT)
dsigma_reduce_kernel(float *part, int nparts, const float *__restrict__ L, const float *__restrict__ upstream,
                     float *__restrict__ grad_L, double *__restrict__ grad_sigma) {
  using FL = FusedLayout<D, K1>;
  constexpr int Dp = FL::Dp, NB = FL::NB, NR4 = FL::NR4, LD = FL::LD, NE = NB * K1 * K1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float *M = reinterpret_cast<float *>(smem_raw);          // [NR4][LD]
  float *Ls = M + NR4 * LD;                                // [NR4][LD]
  __shared__ float s_part[8][33];
  __shared__ int s_last;
  float *dsum = part + (size_t)nparts * NE;
  unsigned int *ticket = reinterpret_cast<unsigned int *>(dsum + NE);
  const int el = threadIdx.x & 31, sl = threadIdx.x >> 5, e = blockIdx.x * 32 + el;
  float a[4] = {0.f, 0.f, 0.f, 0.f};
  if (e < NE) {
    int k = sl;
    for (; k + 24 < nparts; k += 32) {
#pragma unroll
      for (int u = 0; u < 4; ++u) a[u] += part[(size_t)(k + 8 * u) * NE + e];
    }
    for (; k < nparts; k += 8) a[0] += part[(size_t)k * NE + e];
  }
  s_part[sl][el] = (a[0] + a[1]) + (a[2] + a[3]);
  __syncthreads();
  if (threadIdx.x < 32 && e < NE) {
    float t = 0.f;
#pragma unroll
    for (int u = 0; u < 8; ++u) t += s_part[u][el];
    dsum[e] = t;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const float up = upstream ? *upstream : 1.0f;
  for (int t = threadIdx.x; t < NR4 * LD; t += RT) M[t] = 0.f;
  for (int e0 = threadIdx.x; e0 < NR4 * NR4; e0 += RT) {
    const int i = e0 / NR4, c = e0 - i * NR4;
    Ls[i * LD + c] = (L && i < Dp && c <= i) ? L[(size_t)i * Dp + c] : 0.f;
  }
  __syncthreads();
  unpack_blocks<D, K1>(dsum, up, M);
  __syncthreads();
  if (grad_sigma)
    for (int t = threadIdx.x; t < Dp * Dp; t += RT) grad_sigma[t] = (double)M[(t / Dp) * LD + (t % Dp)];
  if (grad_L) dl_from_dsigma<D, K1>(M, Ls, grad_L);
}

// =====================================================================================================
// uniform time grid + shared covariance
// =====================================================================================================
// ws (doubles): hm [2P][K1] | xi [2P][2] | X = S^-1 (lower, packed) [P][NT] | Cinv [P][NT] | hld [P] | flags {chained, nq}
template <int D, int K1>
struct UniLayout {
  static constexpr int N = 2 * D, NT = tri(N);
  size_t hm, xi, xinv, cinv, gbuf, hld, flags, total;    // flags: chained, nq, ticket (uint32, zeroed by the prep kernel)
  __host__ __device__ UniLayout(int P) {
    size_t o = 0;
    auto take = [&](size_t n) { size_t at = o; o += (n + 1) & ~(size_t)1; return at; };
    hm = take((size_t)2 * P * K1); xi = take((size_t)4 * P); xinv = take((size_t)P * NT);
    cinv = take((size_t)P * NT); gbuf = take((size_t)P * NT); hld = take(P); flags = take(4); total = o;
  }
};

// phase 1 (what & 1): basis rows of the common grid, C_p (no regulariser) -> ws.xinv region, max diag -> *diag_max
// phase 2 (what & 2): per segment (one thread each, packed triangle in registers): X = S^-1, C^-1, half logdet
constexpr int UT = 1024;
template <int D, int K1, bool SIGMA_IN>
__global__ void __launch_bounds__(UT)
uniform_prep_kernel(TabDev tb, const float *__restrict__ L, const double *__restrict__ Sigma0,
                    const double *__restrict__ sigma_scale, const float *__restrict__ times,
                    const float *__restrict__ init_time, const int64_t *__restrict__ pairs, double *ws,
                    double *diag_max, double reg_rel, int P, int what) {
  using FL = FusedLayout<D, K1>;
  using UL = UniLayout<D, K1>;
  constexpr int Dp = FL::Dp, N = FL::N, NT = FL::NT, NB = FL::NB, KP = FL::KP, NR4 = FL::NR4, LD = FL::LD, IR = FL::IR;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const UL ul(P);
  double *Sblk = reinterpret_cast<double *>(smem_raw);
  float *Ls = reinterpret_cast<float *>(smem_raw);
  const size_t sb = sizeof(double) * NB * K1 * KP, ls = sizeof(float) * NR4 * LD;
  double *irow = reinterpret_cast<double *>(smem_raw + (((sb > ls ? sb : ls) + 15) & ~(size_t)15));   // [IR]
  double *hm = irow + IR;                                  // [2P][K1]
  __shared__ double s_max[UT / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int chained = block_chained(pairs, P);
  const int nq = chained ? P + 1 : 2 * P;
  double *g_c = ws + ul.xinv;                              // C_p lives in the X region between the two phases
  if (what & 1) {
    // tables first (their latency overlaps the covariance staging)
    if (threadIdx.x <= K1) init_row_entry<K1>(tb, (double)init_time[0], threadIdx.x, irow);
    if (SIGMA_IN) {
      const double sc = sigma_scale ? *sigma_scale : 1.0;
      for (int e0 = threadIdx.x; e0 < Dp * Dp; e0 += 4 * UT) {
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = (e0 + u * UT < Dp * Dp) ? Sigma0[e0 + u * UT] : 0.0;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int e = e0 + u * UT, i = e / Dp, j = e - i * Dp;
          if (e < Dp * Dp && j <= i) sblk_store<K1, KP>(Sblk, i, j, sc * v[u]);
        }
      }
      __syncthreads();
    } else {
      for (int e0 = threadIdx.x; e0 < NR4 * NR4; e0 += 4 * UT) {
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int e = e0 + u * UT, i = e / NR4, c = e - i * NR4;
          v[u] = (e < NR4 * NR4 && i < Dp && c <= i) ? L[(size_t)i * Dp + c] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int e = e0 + u * UT, i = e / NR4, c = e - i * NR4;
          if (e < NR4 * NR4) Ls[i * LD + c] = v[u];
        }
      }
      __syncthreads();
      // Sigma = L L^T, entry per thread (fp32 accumulation as in the per-episode path), lower triangle
      float vals[(Dp * (Dp + 1) / 2 + UT - 1) / UT];
      int cnt = 0;
      for (int t = threadIdx.x; t < tri(Dp); t += UT, ++cnt) {
        int i, j;
        tri_decode(t, i, j);
        const float *a = Ls + i * LD, *bq = Ls + j * LD;
        float a0 = 0.f, a1 = 0.f;
        int k = 0;
        for (; k + 1 <= j; k += 2) { a0 = fmaf(a[k], bq[k], a0); a1 = fmaf(a[k + 1], bq[k + 1], a1); }
        if (k <= j) a0 = fmaf(a[k], bq[k], a0);
        vals[cnt] = a0 + a1;
      }
      __syncthreads();
      cnt = 0;
      for (int t = threadIdx.x; t < tri(Dp); t += UT, ++cnt) {
        int i, j;
        tri_decode(t, i, j);
        sblk_store<K1, KP>(Sblk, i, j, (double)vals[cnt]);
      }
      __syncthreads();
    }
    // ---- basis rows of the common grid (episode 0) ----
    for (int it = threadIdx.x; it < nq * (K1 + 1); it += UT) {
      const int q = it / (K1 + 1), j = it - q * (K1 + 1);
      double xr[2];
      basis_entry<K1>(tb, irow, (double)times[point_time_index(pairs, chained, q, P)], j, hm + (size_t)q * K1, xr);
      if (j < K1) ws[ul.hm + (size_t)q * K1 + j] = hm[(size_t)q * K1 + j];
      else { ws[ul.xi + 2 * q] = xr[0]; ws[ul.xi + 2 * q + 1] = xr[1]; }
    }
    __syncthreads();
    // ---- gram: C [P][NT] ----
    double my_max = 0.0;
    for (int it = threadIdx.x; it < NB * nq; it += UT) {
      const int blk = it / nq, q = it - blk * nq;
      int d, dd;
      tri_decode(blk, d, dd);
      const Links lk = links(chained, q, P);
      double h[K1], v[K1];
      const double *Sb = sblk_at<K1, KP>(Sblk, blk), *hq = hm + (size_t)q * K1;
#pragma unroll
      for (int j = 0; j < K1; ++j) h[j] = hq[j];
#pragma unroll
      for (int i = 0; i < K1; ++i) {
        double a0 = 0.0, a1 = 0.0;
#pragma unroll
        for (int j = 0; j + 1 < K1; j += 2) { a0 = fma(Sb[i * KP + j], h[j], a0); a1 = fma(Sb[i * KP + j + 1], h[j + 1], a1); }
        if (K1 & 1) a0 = fma(Sb[i * KP + K1 - 1], h[K1 - 1], a0);
        v[i] = a0 + a1;
      }
      double kuu = 0.0;
#pragma unroll
      for (int i = 0; i < K1; ++i) kuu = fma(h[i], v[i], kuu);
      const int r0 = 2 * d, q0 = 2 * dd;
      if (lk.pf >= 0) {
        const double *hn = hm + (size_t)lk.nxt * K1;
        double kup = 0.0;
#pragma unroll
        for (int i = 0; i < K1; ++i) kup = fma(hn[i], v[i], kup);
        g_c[(size_t)lk.pf * NT + tri_idx(r0, q0)] = kuu;
        g_c[(size_t)lk.pf * NT + tri_idx(r0 + 1, q0)] = kup;
      }
      if (lk.ps >= 0) {
        g_c[(size_t)lk.ps * NT + tri_idx(r0 + 1, q0 + 1)] = kuu;
        if (d != dd) {
          const double *hp = hm + (size_t)lk.prv * K1;
          double kum = 0.0;
#pragma unroll
          for (int i = 0; i < K1; ++i) kum = fma(hp[i], v[i], kum);
          g_c[(size_t)lk.ps * NT + tri_idx(r0, q0 + 1)] = kum;
        }
      }
      if (d == dd) my_max = fmax(my_max, kuu);
    }
    my_max = warp_max(my_max);
    if (lane == 0) s_max[warp] = my_max;
    __syncthreads();
    if (threadIdx.x == 0) {
      double m = 0.0;
      for (int w = 0; w < UT / 32; ++w) m = fmax(m, s_max[w]);
      atomic_max_pos_double(diag_max, m);
      ws[ul.flags] = (double)chained;
      ws[ul.flags + 1] = (double)nq;
      *reinterpret_cast<unsigned int *>(ws + ul.flags + 2) = 0u;       // ticket of uniform_finish_kernel
    }
  }
}

// phase 2: per segment, ONE warp each (the P segments run on P different SMs): Cholesky with lane = row, X = S^-1 with
// lane = column, C^-1 = X^T X with lane = entry, the matrix in shared memory.  This is a latency chain on the critical
// path of the epoch (a single thread with the triangle in registers needs ~19 k cycles, this ~4 k).
// C_p is read from / X written to the same workspace region.
template <int D, int K1>
__global__ void __launch_bounds__(32)
uniform_factor_kernel(double *ws, const double *__restrict__ diag_max, double reg_rel, int P) {
  using UL = UniLayout<D, K1>;
  constexpr int N = 2 * D, NT = tri(N);
  static_assert(N <= 32, "lane = row");
  const UL ul(P);
  __shared__ double A[NT], X[NT], dinv[N];
  const int p = blockIdx.x, lane = threadIdx.x;
  const double reg = reg_rel * (*diag_max);
  double *g_x = ws + ul.xinv + (size_t)p * NT;
  for (int t = lane; t < NT; t += 32) A[t] = g_x[t];
  __syncwarp();
  double hld = 0.0;
  const int i = lane;
  for (int j = 0; j < N; ++j) {
    double s = 0.0;
    if (i >= j && i < N) {
      s = A[tri_idx(i, j)] + (i == j ? reg : 0.0);
      const double *ri = A + tri_idx(i, 0), *rj = A + tri_idx(j, 0);
      double s1 = 0.0;
      int k = 0;
      for (; k + 1 < j; k += 2) { s = fma(-ri[k], rj[k], s); s1 = fma(-ri[k + 1], rj[k + 1], s1); }
      if (k < j) s = fma(-ri[k], rj[k], s);
      s += s1;
    }
    const double d = __shfl_sync(0xffffffffu, s, j);
    double inv = (double)rsqrtf((float)d);
    inv = inv * fma(-0.5 * d, inv * inv, 1.5);
    inv = inv * fma(-0.5 * d, inv * inv, 1.5);
    hld += 0.5 * log(d);
    __syncwarp();
    if (i == j) { A[tri_idx(j, j)] = d * inv; dinv[j] = inv; }
    else if (i > j && i < N) A[tri_idx(i, j)] = s * inv;
    __syncwarp();
  }
  // X = S^-1: lane j solves column j by forward substitution; its column lives in registers (compile-time indices)
  if (lane < N) {
    const int j = lane;
    double x[N];
#pragma unroll
    for (int r = 0; r < N; ++r) {
      double v = (r == j) ? 1.0 : 0.0;
#pragma unroll
      for (int k = 0; k < r; ++k) v = fma(-A[r * (r + 1) / 2 + k], (k >= j) ? x[k] : 0.0, v);
      x[r] = (r >= j) ? v * dinv[r] : 0.0;
    }
#pragma unroll
    for (int r = 0; r < N; ++r)
      if (r >= j) X[tri_idx(r, j)] = x[r];
  }
  __syncwarp();
  for (int t = lane; t < NT; t += 32) {
    int r, c;
    tri_decode(t, r, c);
    double v = 0.0;
    for (int k = r; k < N; ++k) v = fma(X[tri_idx(k, r)], X[tri_idx(k, c)], v);
    ws[ul.cinv + (size_t)p * NT + t] = v;
    g_x[t] = X[t];
  }
  if (lane == 0) ws[ul.hld + p] = hld;
}

// main: a CTA works on chunks of 32 episodes.  Per chunk: (A) coalesced staging of the chunk's means, initial
// conditions and the sampled positions at the nq distinct time points; (B) residuals r = x - mu at those points, in
// place; (C) thread per (episode = lane, pair = warp-uniform): z = X_p r (X_p read by broadcast), log-prob, upstream
// gradient, alpha = X_p^T z -> shared memory; (D) grad_mean; (E) the CTA's running sums
// A_p += sum_b g alpha alpha^T, gs_p += sum_b g.  apart [gridDim.x][P][NT + 1] fp64 receives the sums of this CTA.
constexpr int UM_THREADS = 256;            // 255 registers per thread: no spills (the L1 is mostly shared memory)
// EP = episodes per chunk: 32 (lane = episode) for large batches, 8 (lane = (pair slot, episode): four pairs per warp)
// when the batch would otherwise fill only a fraction of the SMs.
template <int D, int K1, int EP>
struct UniMainSmem {
  static constexpr int UM_EP = EP;
  static constexpr int Dp = D * K1, N = 2 * D, NT = tri(N), AL = UM_EP + 1, MS = Dp | 1;
  size_t X, h, xi, hld, al, g, mean, r, y0, pidx, total;
  int RS;                                   // row stride (doubles) of r [episode][point * D + d], odd
  __host__ __device__ UniMainSmem(int P) {
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += (bytes + 15) & ~(size_t)15; return at; };
    RS = (2 * P * D) | 1;
    X = take(sizeof(double) * P * NT); h = take(sizeof(double) * 2 * P * K1); xi = take(sizeof(double) * 4 * P);
    hld = take(sizeof(double) * P); al = take(sizeof(double) * (size_t)P * N * AL);
    g = take(sizeof(double) * (size_t)P * AL); r = take(sizeof(double) * (size_t)UM_EP * RS);
    mean = take(sizeof(float) * UM_EP * MS); y0 = take(sizeof(float) * 2 * UM_EP * D);
    pidx = take(sizeof(int) * 2 * P);
    total = o;
  }
};
template <int D, int K1, int UM_EP>
__global__ void __launch_bounds__(UM_THREADS, 1)
uniform_main_kernel(TabDev tb, const double *__restrict__ ws, const float *__restrict__ smp_traj,
                    const float *__restrict__ mean, const float *__restrict__ init_pos,
                    const float *__restrict__ init_vel, const int64_t *__restrict__ pairs, int grad_mode,
                    const float *__restrict__ grad_logp, const float *__restrict__ logp_old,
                    const float *__restrict__ advantage, double grad_scale, double *__restrict__ loss_acc,
                    float *__restrict__ logp, int32_t *__restrict__ info, float *__restrict__ grad_mean,
                    double *__restrict__ apart, long long B, int T, int P) {
  using UL = UniLayout<D, K1>;
  using SM = UniMainSmem<D, K1, UM_EP>;
  constexpr int Dp = D * K1, N = 2 * D, NT = tri(N), AL = SM::AL, MS = SM::MS;
  const UL ul(P);
  const SM sm(P);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double *sX = reinterpret_cast<double *>(smem_raw + sm.X);          // [P][NT]
  double *sh = reinterpret_cast<double *>(smem_raw + sm.h);          // hm [nq][K1]
  double *sxi = reinterpret_cast<double *>(smem_raw + sm.xi);        // [nq][2]
  double *shld = reinterpret_cast<double *>(smem_raw + sm.hld);      // [P]
  double *sal = reinterpret_cast<double *>(smem_raw + sm.al);        // alpha [P][N][AL]
  double *sg = reinterpret_cast<double *>(smem_raw + sm.g);          // g [P][AL]
  double *sr = reinterpret_cast<double *>(smem_raw + sm.r);          // r [UM_EP][RS]: x then residual at (point, d)
  float *smean = reinterpret_cast<float *>(smem_raw + sm.mean);      // [UM_EP][MS]
  float *sy0 = reinterpret_cast<float *>(smem_raw + sm.y0);          // y0 [UM_EP][D] | v0 [UM_EP][D]
  int *spidx = reinterpret_cast<int *>(smem_raw + sm.pidx);          // time index of each distinct point
  __shared__ double s_red[2 * (UM_THREADS / 32)];
  const int chained = (int)ws[ul.flags], nq = (int)ws[ul.flags + 1];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = UM_THREADS / 32;
  const int RS = sm.RS;
  const bool want_grad = grad_mode != 0;
  const double tau = tb.tau;
  for (int t = threadIdx.x; t < P * NT; t += UM_THREADS) sX[t] = ws[ul.xinv + t];
  for (int t = threadIdx.x; t < nq * K1; t += UM_THREADS) sh[t] = ws[ul.hm + t];
  for (int t = threadIdx.x; t < 2 * nq; t += UM_THREADS) sxi[t] = ws[ul.xi + t];
  for (int t = threadIdx.x; t < P; t += UM_THREADS) shld[t] = ws[ul.hld + t];
  for (int t = threadIdx.x; t < nq; t += UM_THREADS) spidx[t] = (int)point_time_index(pairs, chained, t, P);
  // running sums of this CTA: entry e = p (NT + 1) + t, NE = P (NT + 1); up to MAXACC per thread
  constexpr int MAXACC = 12;
  const int NE = P * (NT + 1);
  double racc[MAXACC];
#pragma unroll
  for (int u = 0; u < MAXACC; ++u) racc[u] = 0.0;
  double loss_part = 0.0, ratio_part = 0.0;
  const long long n_chunks = (B + UM_EP - 1) / UM_EP;
  for (long long ch = blockIdx.x; ch < n_chunks; ch += gridDim.x) {
    const long long bbase = ch * UM_EP;
    const int nb = (int)((B - bbase) < UM_EP ? (B - bbase) : UM_EP);
    __syncthreads();                                       // staging tables done / previous chunk consumed
    // ---- (A) staging: the chunk's episodes are contiguous in every input ----
    for (int t = threadIdx.x; t < nb * Dp; t += UM_THREADS) smean[(t / Dp) * MS + (t % Dp)] = mean[bbase * Dp + t];
    for (int t = threadIdx.x; t < nb * D; t += UM_THREADS) {
      sy0[t] = init_pos[bbase * D + t];
      sy0[UM_EP * D + t] = init_vel[bbase * D + t];
    }
    for (int t0 = threadIdx.x; t0 < nb * nq * D; t0 += 8 * UM_THREADS) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int t = t0 + u * UM_THREADS;
        if (t < nb * nq * D) {
          const int l = t / (nq * D), r = t - l * nq * D, q = r / D, d = r - q * D;
          v[u] = smp_traj[((bbase + l) * T + spidx[q]) * (2 * D) + d];
        }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int t = t0 + u * UM_THREADS;
        if (t < nb * nq * D) { const int l = t / (nq * D); sr[(size_t)l * RS + (t - l * nq * D)] = (double)v[u]; }
      }
    }
    __syncthreads();
    // ---- (B) residual at the distinct points, in place: r[l][q][d] = x - (xi1 y0 + xi2 tau v0 + h_q . theta_d) ----
    for (int t = threadIdx.x; t < nb * nq * D; t += UM_THREADS) {
      const int l = t / (nq * D), r = t - l * nq * D, q = r / D, d = r - q * D;
      const double y0 = (double)sy0[l * D + d], v0 = (double)sy0[UM_EP * D + l * D + d] * tau;
      const double *hq = sh + (size_t)q * K1;
      const float *th = smean + l * MS + d * K1;
      double mu = sxi[2 * q] * y0 + sxi[2 * q + 1] * v0;
#pragma unroll
      for (int j = 0; j < K1; ++j) mu = fma(hq[j], (double)th[j], mu);
      if (tb.relative_goal) {
        const double shift = tb.relative_goal_scaled ? y0 : y0 / tb.scale[K1 - 1];
        mu = fma(hq[K1 - 1], shift, mu);
      }
      sr[(size_t)l * RS + r] -= mu;
    }
    __syncthreads();
    // ---- (C) thread per (episode, pair) ----
    constexpr int PPW = 32 / UM_EP;                       // pairs per warp pass
    const int el = lane % UM_EP;                           // episode slot of this thread
    const long long b = bbase + el;
    for (int p = warp * PPW + lane / UM_EP; p < P; p += nwarps * PPW) {
      double g = 0.0, al[N];
#pragma unroll
      for (int i = 0; i < N; ++i) al[i] = 0.0;
      if (el < nb) {
        const double *X = sX + (size_t)p * NT;
        const double *r0 = sr + (size_t)el * RS + point_of(chained, p, 0) * D;
        const double *r1 = sr + (size_t)el * RS + point_of(chained, p, 1) * D;
        double r[N], z[N];
#pragma unroll
        for (int d = 0; d < D; ++d) { r[2 * d] = r0[d]; r[2 * d + 1] = r1[d]; }
        double maha = 0.0;
#pragma unroll
        for (int i = 0; i < N; ++i) {                       // z = X r  (X = S^-1, lower)
          double v = 0.0;
#pragma unroll
          for (int j = 0; j <= i; ++j) v = fma(X[i * (i + 1) / 2 + j], r[j], v);
          z[i] = v;
          maha = fma(v, v, maha);
        }
        const double lp = -0.5 * ((double)N * LN_2PI + maha) - shld[p];
        const long long gid = b * P + p;
        if (logp) logp[gid] = (float)lp;
        if (info) info[gid] = 0;
        if (want_grad) {
          if (grad_mode == 2) {
            const double ratio = exp(lp - (double)logp_old[gid]);
            g = -ratio * (double)advantage[gid] * grad_scale;
            loss_part += g;
            ratio_part += ratio * grad_scale;
          } else {
            g = (double)grad_logp[gid];
          }
#pragma unroll
          for (int j = 0; j < N; ++j) {                     // alpha = X^T z
            double v = 0.0;
#pragma unroll
            for (int i = j; i < N; ++i) v = fma(X[i * (i + 1) / 2 + j], z[i], v);
            al[j] = v;
          }
        }
      }
      if (want_grad) {
#pragma unroll
        for (int j = 0; j < N; ++j) sal[((size_t)p * N + j) * AL + el] = al[j];
        sg[(size_t)p * AL + el] = g;
      }
    }
    if (!want_grad) continue;
    __syncthreads();
    if (grad_mean) {
      // ---- (D) grad_mean[b][d K1 + j] = sum_{p, k} h_{p,k}[j] g alpha_bp[(d, k)]
      for (int it = threadIdx.x; it < UM_EP * Dp; it += UM_THREADS) {
        const int o = it / UM_EP, l = it - o * UM_EP, d = o / K1, j = o - d * K1;
        if (l >= nb) continue;
        double acc0 = 0.0, acc1 = 0.0;
        for (int p = 0; p < P; ++p) {
          const double gg = sg[(size_t)p * AL + l];
          acc0 = fma(gg * sh[(size_t)point_of(chained, p, 0) * K1 + j], sal[((size_t)p * N + 2 * d) * AL + l], acc0);
          acc1 = fma(gg * sh[(size_t)point_of(chained, p, 1) * K1 + j], sal[((size_t)p * N + 2 * d + 1) * AL + l], acc1);
        }
        grad_mean[(bbase + l) * Dp + o] = (float)(acc0 + acc1);
      }
    }
    if (apart) {
      // ---- (E) running sums (slots >= nb hold g = 0, alpha = 0)
      constexpr int nb_even = UM_EP;
#pragma unroll
      for (int u = 0; u < MAXACC; ++u) {
        const int e = threadIdx.x + u * UM_THREADS;
        if (e < NE) {
          const int p = e / (NT + 1), t = e - p * (NT + 1);
          const double *gp = sg + (size_t)p * AL;
          double a0 = 0.0, a1 = 0.0;
          if (t < NT) {
            int i, j;
            tri_decode(t, i, j);
            const double *ai = sal + ((size_t)p * N + i) * AL, *aj = sal + ((size_t)p * N + j) * AL;
#pragma unroll 4
            for (int l = 0; l < nb_even; l += 2) {
              a0 = fma(gp[l] * ai[l], aj[l], a0);
              a1 = fma(gp[l + 1] * ai[l + 1], aj[l + 1], a1);
            }
          } else {
            for (int l = 0; l < nb_even; ++l) a0 += gp[l];
          }
          racc[u] += a0 + a1;
        }
      }
    }
  }
  if (want_grad && apart) {
#pragma unroll
    for (int u = 0; u < MAXACC; ++u) {
      const int e = threadIdx.x + u * UM_THREADS;
      if (e < NE) apart[(size_t)blockIdx.x * NE + e] = racc[u];
    }
  }
  if (grad_mode == 2 && loss_acc) {
    loss_part = warp_sum(loss_part);
    ratio_part = warp_sum(ratio_part);
    if (lane == 0) { s_red[2 * warp] = loss_part; s_red[2 * warp + 1] = ratio_part; }
    __syncthreads();
    if (threadIdx.x == 0) {
      double a = 0.0, rr = 0.0;
      for (int w = 0; w < nwarps; ++w) { a += s_red[2 * w]; rr += s_red[2 * w + 1]; }
      if (rr != 0.0) { atomicAdd(loss_acc, a); atomicAdd(loss_acc + 1, rr); }
    }
  }
}

// finish: CTA p sums the per-CTA A_p / gs_p partials (8 threads per entry, fixed order) and forms
// G_p = 1/2 (A_p - gs_p C_p^-1) -> ws.gbuf; the LAST CTA to finish (ticket) turns the P adjoints into dSigma
// (task (DoF block, row)) and grad_L = 2 tril(dSigma L) * upstream and / or grad_sigma.
template <int D, int K1>
__global__ void __launch_bounds__(UT)
uniform_finish_kernel(double *ws, const double *__restrict__ apart, int nparts, const float *__restrict__ L,
                      const float *__restrict__ upstream, float *__restrict__ grad_L, double *__restrict__ grad_sigma,
                      int P) {
  using FL = FusedLayout<D, K1>;
  using UL = UniLayout<D, K1>;
  constexpr int Dp = FL::Dp, NT = FL::NT, NB = FL::NB, NR4 = FL::NR4, LD = FL::LD;
  static_assert(NT + 1 <= 128, "128 entry slots");
  const UL ul(P);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float *M = reinterpret_cast<float *>(smem_raw);          // [NR4][LD]
  float *Ls = M + NR4 * LD;                                // [NR4][LD]
  double *G = reinterpret_cast<double *>(Ls + NR4 * LD + (NR4 * LD & 1));   // [P][NT]
  double *hm = G + (size_t)P * NT;                         // [2P][K1]
  __shared__ double s_part[8][129];
  __shared__ int s_last;
  const int NE = P * (NT + 1);
  const int p = blockIdx.x, t = threadIdx.x & 127, sl = threadIdx.x >> 7;
  unsigned int *ticket = reinterpret_cast<unsigned int *>(ws + ul.flags + 2);
  // the factor (used by the last CTA only): loads in flight during the reduction
  float lreg[(NR4 * NR4 + UT - 1) / UT];
#pragma unroll
  for (int u = 0; u < (NR4 * NR4 + UT - 1) / UT; ++u) {
    const int e = threadIdx.x + u * UT, i = e / NR4, c = e - i * NR4;
    lreg[u] = (L && e < NR4 * NR4 && i < Dp && c <= i) ? L[(size_t)i * Dp + c] : 0.f;
  }
  double a[4] = {0.0, 0.0, 0.0, 0.0};
  if (t <= NT) {
    const double *src = apart + (size_t)p * (NT + 1) + t;
    int k = sl;
    for (; k + 24 < nparts; k += 32) {
#pragma unroll
      for (int u = 0; u < 4; ++u) a[u] += src[(size_t)(k + 8 * u) * NE];
    }
    for (; k < nparts; k += 8) a[0] += src[(size_t)k * NE];
  }
  s_part[sl][t] = (a[0] + a[1]) + (a[2] + a[3]);
  __syncthreads();
  if (threadIdx.x <= NT) {
    double v = 0.0;
#pragma unroll
    for (int u = 0; u < 8; ++u) v += s_part[u][threadIdx.x];
    s_part[0][threadIdx.x] = v;
  }
  __syncthreads();
  if (threadIdx.x < NT)
    ws[ul.gbuf + (size_t)p * NT + threadIdx.x] =
        0.5 * (s_part[0][threadIdx.x] - s_part[0][NT] * ws[ul.cinv + (size_t)p * NT + threadIdx.x]);
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const int chained = (int)ws[ul.flags], nq = (int)ws[ul.flags + 1];
  const float up = upstream ? *upstream : 1.0f;
  for (int e = threadIdx.x; e < P * NT; e += UT) G[e] = __ldcg(ws + ul.gbuf + e);
  for (int e = threadIdx.x; e < nq * K1; e += UT) hm[e] = ws[ul.hm + e];
  for (int e = threadIdx.x; e < NR4 * LD; e += UT) M[e] = 0.f;
#pragma unroll
  for (int u = 0; u < (NR4 * NR4 + UT - 1) / UT; ++u) {
    const int e = threadIdx.x + u * UT, i = e / NR4, c = e - i * NR4;
    if (e < NR4 * NR4) Ls[i * LD + c] = lreg[u];
  }
  __syncthreads();
  // ---- dSigma blocks: task (blk, i) = row i of the K1 x K1 block (d, dd)
  for (int task = threadIdx.x; task < NB * K1; task += UT) {
    const int blk = task / K1, i = task - blk * K1;
    int d, dd;
    tri_decode(blk, d, dd);
    const int r0 = 2 * d, q0 = 2 * dd;
    const int e00 = tri_idx(r0, q0), e10 = tri_idx(r0 + 1, q0), e11 = tri_idx(r0 + 1, q0 + 1);
    const int e01 = (d != dd) ? tri_idx(r0, q0 + 1) : e10;
    double acc[K1];
#pragma unroll
    for (int j = 0; j < K1; ++j) acc[j] = 0.0;
    for (int q = 0; q < nq; ++q) {
      const Links lk = links(chained, q, P);
      double w = 0.0;
      const double hqi = hm[(size_t)q * K1 + i];
      if (lk.pf >= 0) {
        const double *Gp = G + (size_t)lk.pf * NT;
        w += Gp[e00] * hqi + Gp[e10] * hm[(size_t)lk.nxt * K1 + i];
      }
      if (lk.ps >= 0) {
        const double *Gp = G + (size_t)lk.ps * NT;
        w += Gp[e11] * hqi + Gp[e01] * hm[(size_t)lk.prv * K1 + i];
      }
#pragma unroll
      for (int j = 0; j < K1; ++j) acc[j] = fma(w, hm[(size_t)q * K1 + j], acc[j]);
    }
#pragma unroll
    for (int j = 0; j < K1; ++j) {
      const float v = up * (float)acc[j];
      M[(d * K1 + i) * LD + dd * K1 + j] = v;
      if (d != dd) M[(dd * K1 + j) * LD + d * K1 + i] = v;
    }
  }
  __syncthreads();
  if (grad_sigma)
    for (int e = threadIdx.x; e < Dp * Dp; e += UT) grad_sigma[e] = (double)M[(e / Dp) * LD + (e % Dp)];
  if (grad_L) dl_from_dsigma<D, K1>(M, Ls, grad_L);
}

}  // namespace

// ---- host side ---------------------------------------------------------------------------------------
#define TCE_FOR_SHAPES(X) X(7, 9) X(4, 9) X(7, 4) X(3, 4) X(2, 3)

namespace {
constexpr size_t SMEM_LIMIT = 227 * 1024;

template <int D, int K1>
int fused_pick_E(int P, int chained) {
  int E = FT / P;
  if (E > FT / tri(D)) E = FT / tri(D);              // phase 3b: one thread per (episode, DoF block)
  while (E > 1 && FusedLayout<D, K1>(E, P, chained).total > SMEM_LIMIT) --E;
  if (E < 1 || FusedLayout<D, K1>(E, P, chained).total > SMEM_LIMIT) return 0;
  return E;
}

int sm_count() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}
}  // namespace

extern "C" int tce_seglik_fused_config(const tce_tables_t *t, int64_t B, int64_t P, int chained, int32_t *E_out,
                                       int32_t *grid_out, int64_t *part_floats, int64_t *pre_doubles_per_episode) {
  if (!t || B < 0 || P < 1) return TCE_ERR_INVALID_ARGUMENT;
#define X(Dv, Kv)                                                                              \
  if (t->D == Dv && t->K1 == Kv) {                                                             \
    if (P > FT) return TCE_ERR_UNSUPPORTED_SHAPE;                                              \
    const int E = fused_pick_E<Dv, Kv>((int)P, chained);                                       \
    if (!E) return TCE_ERR_UNSUPPORTED_SHAPE;                                                  \
    const int64_t groups = (B + E - 1) / E;                                                    \
    int grid = (int)(groups < sm_count() ? groups : sm_count());                               \
    if (grid < 1) grid = 1;                                                                    \
    if (E_out) *E_out = E;                                                                     \
    if (grid_out) *grid_out = grid;                                                            \
    /* [grid] partials + the sum + the ticket (padded to 4 floats) */                           \
    if (part_floats) *part_floats = ((int64_t)grid + 1) * tri(Dv) * Kv * Kv + 4;               \
    if (pre_doubles_per_episode)                                                               \
      *pre_doubles_per_episode = (int64_t)pre_doubles(chained ? (int)P + 1 : 2 * (int)P, Kv, 2 * Dv, (int)P); \
    return TCE_OK;                                                                             \
  }
  TCE_FOR_SHAPES(X)
#undef X
  return TCE_ERR_UNSUPPORTED_SHAPE;
}

template <bool SIGMA_IN>
static int prepass_launch(const tce_tables_t *t, const float *smp_traj, const float *mean, const float *L,
                          int64_t ldb_L, const double *Sigma0, const double *sigma_scale, const float *times,
                          const float *init_time, const float *init_pos, const float *init_vel,
                          const int64_t *pred_pairs, double *pre, double *diag_max, int chained, int64_t B, int64_t T,
                          int64_t P, void *stream) {
  if (B == 0) return TCE_OK;
  if (!t || !smp_traj || !mean || (SIGMA_IN ? !Sigma0 : !L) || !times || !init_time || !init_pos || !init_vel ||
      !pred_pairs || !pre || !diag_max || B < 0 || T < 1 || P < 1)
    return TCE_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
#define X(Dv, Kv)                                                                                                  \
  if (t->D == Dv && t->K1 == Kv) {                                                                                 \
    using FL = FusedLayout<Dv, Kv>;                                                                                \
    const size_t smem = sizeof(double) * ((size_t)Dv * Kv * Kv + 2 * P * Kv + 4 * P + FL::IR) + 32 +               \
                        (SIGMA_IN ? 0 : sizeof(float) * FL::Dp * (FL::Dp + 1));                                    \
    if (smem > SMEM_LIMIT) return TCE_ERR_UNSUPPORTED_SHAPE;                                                       \
    auto kern = seglik_prepass_kernel<Dv, Kv, SIGMA_IN>;                                                           \
    TCE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "prepass smem");  \
    int64_t grid = B;                                                                                              \
    const int64_t cap = (int64_t)sm_count() * 16;                                                                  \
    if (grid > cap) grid = cap;                                                                                    \
    kern<<<(unsigned)grid, PT, smem, st>>>(tab_dev(t), smp_traj, mean, L, ldb_L, Sigma0, sigma_scale, times,       \
                                           init_time, init_pos, init_vel, pred_pairs, pre, diag_max, (long long)B, \
                                           (int)T, (int)P, chained);                                               \
    TCE_CHECK_LAUNCH("seglik_prepass_kernel");                                                                     \
    return TCE_OK;                                                                                                 \
  }
  TCE_FOR_SHAPES(X)
#undef X
  return TCE_ERR_UNSUPPORTED_SHAPE;
}

extern "C" int tce_seglik_prepass(const tce_tables_t *t, const float *smp_traj, const float *mean, const float *L,
                                  int64_t ldb_L, const double *Sigma0, const double *sigma_scale, const float *times,
                                  const float *init_time, const float *init_pos, const float *init_vel,
                                  const int64_t *pred_pairs, double *pre, double *diag_max, int chained, int64_t B,
                                  int64_t T, int64_t P, void *stream) {
  if (Sigma0)
    return prepass_launch<true>(t, smp_traj, mean, nullptr, 0, Sigma0, sigma_scale, times, init_time, init_pos,
                                init_vel, pred_pairs, pre, diag_max, chained, B, T, P, stream);
  return prepass_launch<false>(t, smp_traj, mean, L, ldb_L, nullptr, nullptr, times, init_time, init_pos, init_vel,
                               pred_pairs, pre, diag_max, chained, B, T, P, stream);
}

template <bool SIGMA_IN>
static int fused_launch(const tce_tables_t *t, const double *pre, const float *L, int64_t ldb_L, const double *Sigma0,
                        const double *sigma_scale, const int64_t *pred_pairs, const double *diag_max, double reg_rel,
                        int grad_mode, const float *grad_logp, const float *logp_old, const float *advantage,
                        double grad_scale, double *loss_acc, float *logp, int32_t *info, float *grad_mean,
                        float *grad_L, float *dsigma_part, int chained, int64_t B, int64_t P, void *stream) {
  if (B == 0) return TCE_OK;
  if (!t || !pre || (SIGMA_IN ? !Sigma0 : !L) || !pred_pairs || !diag_max || B < 0 || P < 1 || grad_mode < 0 ||
      grad_mode > 2)
    return TCE_ERR_INVALID_ARGUMENT;
  if (grad_mode == 1 && !grad_logp) return TCE_ERR_INVALID_ARGUMENT;
  if (grad_mode == 2 && (!logp_old || !advantage)) return TCE_ERR_INVALID_ARGUMENT;
  const bool shared_cov = SIGMA_IN || ldb_L == 0;
  if (grad_mode && !shared_cov && dsigma_part) return TCE_ERR_INVALID_ARGUMENT;
  if (grad_mode && shared_cov && grad_L) return TCE_ERR_INVALID_ARGUMENT;   /* shared: partials + tce_seglik_dsigma_reduce */
  cudaStream_t st = (cudaStream_t)stream;
  int32_t E = 0, grid = 0;
  int rc = tce_seglik_fused_config(t, B, P, chained, &E, &grid, nullptr, nullptr);
  if (rc != TCE_OK) return rc;
#define X(Dv, Kv)                                                                                                  \
  if (t->D == Dv && t->K1 == Kv) {                                                                                 \
    const size_t smem = FusedLayout<Dv, Kv>(E, (int)P, chained).total;                                             \
    auto kern = seglik_fused_kernel<Dv, Kv, SIGMA_IN>;                                                             \
    TCE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "fused smem");    \
    kern<<<(unsigned)grid, FT, smem, st>>>(pre, L, ldb_L, Sigma0, sigma_scale, pred_pairs, diag_max, reg_rel,      \
                                           grad_mode, grad_logp, logp_old, advantage, grad_scale, loss_acc, logp,  \
                                           info, grad_mean, grad_L, dsigma_part, (long long)B, (int)P, (int)E,     \
                                           chained);                                                               \
    TCE_CHECK_LAUNCH("seglik_fused_kernel");                                                                       \
    return TCE_OK;                                                                                                 \
  }
  TCE_FOR_SHAPES(X)
#undef X
  return TCE_ERR_UNSUPPORTED_SHAPE;
}

extern "C" int tce_seglik_fused(const tce_tables_t *t, const double *pre, const float *L, int64_t ldb_L,
                                const double *Sigma0, const double *sigma_scale, const int64_t *pred_pairs,
                                const double *diag_max, double reg_rel, int grad_mode, const float *grad_logp,
                                const float *logp_old, const float *advantage, double grad_scale, double *loss_acc,
                                float *logp, int32_t *info, float *grad_mean, float *grad_L, float *dsigma_part,
                                int chained, int64_t B, int64_t P, void *stream) {
  if (Sigma0)
    return fused_launch<true>(t, pre, nullptr, 0, Sigma0, sigma_scale, pred_pairs, diag_max, reg_rel, grad_mode,
                              grad_logp, logp_old, advantage, grad_scale, loss_acc, logp, info, grad_mean, grad_L,
                              dsigma_part, chained, B, P, stream);
  return fused_launch<false>(t, pre, L, ldb_L, nullptr, nullptr, pred_pairs, diag_max, reg_rel, grad_mode, grad_logp,
                             logp_old, advantage, grad_scale, loss_acc, logp, info, grad_mean, grad_L, dsigma_part,
                             chained, B, P, stream);
}

extern "C" int tce_seglik_dsigma_reduce(const tce_tables_t *t, float *dsigma_part, int nparts, const float *L,
                                        const float *upstream, float *grad_L, double *grad_sigma, void *stream) {
  if (!t || !dsigma_part || nparts < 1 || (!grad_L && !grad_sigma) || (grad_L && !L)) return TCE_ERR_INVALID_ARGUMENT;
#define X(Dv, Kv)                                                                                               \
  if (t->D == Dv && t->K1 == Kv) {                                                                              \
    using FL = FusedLayout<Dv, Kv>;                                                                             \
    const size_t smem = sizeof(float) * 2 * FL::NR4 * FL::LD + 16;                                              \
    auto kern = dsigma_reduce_kernel<Dv, Kv>;                                                                   \
    TCE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "reduce smem"); \
    const int NE = FL::NB * Kv * Kv;                                                                            \
    kern<<<(NE + 31) / 32, RT, smem, (cudaStream_t)stream>>>(dsigma_part, nparts, L, upstream, grad_L, grad_sigma); \
    TCE_CHECK_LAUNCH("dsigma_reduce_kernel");                                                                   \
    return TCE_OK;                                                                                              \
  }
  TCE_FOR_SHAPES(X)
#undef X
  return TCE_ERR_UNSUPPORTED_SHAPE;
}

/* ---- uniform time grid + shared covariance ---------------------------------------------------------------- */
extern "C" size_t tce_seglik_uniform_ws_doubles(const tce_tables_t *t, int64_t P) {
  if (!t || P < 1) return 0;
#define X(Dv, Kv) if (t->D == Dv && t->K1 == Kv) return UniLayout<Dv, Kv>((int)P).total;
  TCE_FOR_SHAPES(X)
#undef X
  return 0;
}

/* episodes per chunk of tce_seglik_uniform_main: 32 once 8 would give every SM more than one chunk, unless the
   32-episode layout does not fit in shared memory at this P (large P: the 8-episode CTAs then loop over chunks) */
static int uniform_ep(const tce_tables_t *t, int64_t B, int64_t P) {
  if (B <= 8 * (int64_t)sm_count()) return 8;
#define X(Dv, Kv) \
  if (t->D == Dv && t->K1 == Kv) return UniMainSmem<Dv, Kv, 32>((int)P).total <= SMEM_LIMIT ? 32 : 8;
  TCE_FOR_SHAPES(X)
#undef X
  return 32;
}
static int uniform_grid(int ep, int64_t B) {
  const int64_t chunks = (B + ep - 1) / ep;
  const int64_t cap = (int64_t)sm_count();
  return (int)(chunks < cap ? (chunks < 1 ? 1 : chunks) : cap);
}

/* number of CTAs of tce_seglik_uniform_main (= partial sums) and the doubles of its `apart` buffer */
extern "C" int tce_seglik_uniform_parts(const tce_tables_t *t, int64_t B, int64_t P, int32_t *nparts,
                                        int64_t *apart_doubles) {
  if (!t || P < 1 || B < 0) return TCE_ERR_INVALID_ARGUMENT;
  const int g = uniform_grid(uniform_ep(t, B, P), B);
  const int64_t N = 2 * (int64_t)t->D, NT = N * (N + 1) / 2;
  if (P * (NT + 1) > 12 * UM_THREADS) return TCE_ERR_UNSUPPORTED_SHAPE;
  if (nparts) *nparts = g;
  if (apart_doubles) *apart_doubles = (int64_t)g * P * (NT + 1);
  return TCE_OK;
}

extern "C" int tce_seglik_uniform_prep(const tce_tables_t *t, const float *L, const double *Sigma0,
                                       const double *sigma_scale, const float *times, const float *init_time,
                                       const int64_t *pred_pairs, double *ws, double *diag_max, double reg_rel,
                                       int what, int64_t P, void *stream) {
  if (!t || (!L && !Sigma0) || !times || !init_time || !pred_pairs || !ws || !diag_max || P < 1 || !(what & 3))
    return TCE_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
#define X(Dv, Kv)                                                                                                   \
  if (t->D == Dv && t->K1 == Kv) {                                                                                  \
    using FL = FusedLayout<Dv, Kv>;                                                                                 \
    const size_t sb = sizeof(double) * FL::NB * Kv * FL::KP, ls = sizeof(float) * FL::NR4 * FL::LD;                 \
    const size_t smem = (((sb > ls ? sb : ls) + 15) & ~(size_t)15) + sizeof(double) * (FL::IR + 2 * P * Kv) + 16;   \
    if (smem > SMEM_LIMIT) return TCE_ERR_UNSUPPORTED_SHAPE;                                                        \
    if ((what & 1) && Sigma0) {                                                                                     \
      auto kern = uniform_prep_kernel<Dv, Kv, true>;                                                                \
      TCE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "uprep smem");   \
      kern<<<1, UT, smem, st>>>(tab_dev(t), nullptr, Sigma0, sigma_scale, times, init_time, pred_pairs, ws,         \
                                diag_max, reg_rel, (int)P, what);                                                   \
    } else if (what & 1) {                                                                                          \
      auto kern = uniform_prep_kernel<Dv, Kv, false>;                                                               \
      TCE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "uprep smem");   \
      kern<<<1, UT, smem, st>>>(tab_dev(t), L, nullptr, nullptr, times, init_time, pred_pairs, ws, diag_max,        \
                                reg_rel, (int)P, what);                                                             \
    }                                                                                                               \
    if (what & 1) TCE_CHECK_LAUNCH("uniform_prep_kernel");                                                          \
    if (what & 2) uniform_factor_kernel<Dv, Kv><<<(unsigned)P, 32, 0, st>>>(ws, diag_max, reg_rel, (int)P);         \
    TCE_CHECK_LAUNCH("uniform_factor_kernel");                                                                      \
    return TCE_OK;                                                                                                  \
  }
  TCE_FOR_SHAPES(X)
#undef X
  return TCE_ERR_UNSUPPORTED_SHAPE;
}

extern "C" int tce_seglik_uniform_main(const tce_tables_t *t, const double *ws, const float *smp_traj,
                                       const float *mean, const float *init_pos, const float *init_vel,
                                       const int64_t *pred_pairs, int grad_mode, const float *grad_logp,
                                       const float *logp_old, const float *advantage, double grad_scale,
                                       double *loss_acc, float *logp, int32_t *info, float *grad_mean, double *apart,
                                       int64_t B, int64_t T, int64_t P, void *stream) {
  if (B == 0) return TCE_OK;
  if (!t || !ws || !smp_traj || !mean || !init_pos || !init_vel || !pred_pairs || B < 0 || T < 1 || P < 1 ||
      grad_mode < 0 || grad_mode > 2)
    return TCE_ERR_INVALID_ARGUMENT;
  if (grad_mode == 1 && !grad_logp) return TCE_ERR_INVALID_ARGUMENT;
  if (grad_mode == 2 && (!logp_old || !advantage)) return TCE_ERR_INVALID_ARGUMENT;
  const int ep = uniform_ep(t, B, P);
  const unsigned grid = (unsigned)uniform_grid(ep, B);
#define X(Dv, Kv)                                                                                                  \
  if (t->D == Dv && t->K1 == Kv) {                                                                                 \
    constexpr int N = 2 * Dv, NT = N * (N + 1) / 2;                                                                \
    if (P * (NT + 1) > 12 * UM_THREADS) return TCE_ERR_UNSUPPORTED_SHAPE;                                          \
    if (ep == 8) {                                                                                                 \
      const size_t smem = UniMainSmem<Dv, Kv, 8>((int)P).total;                                                    \
      if (smem > SMEM_LIMIT) return TCE_ERR_UNSUPPORTED_SHAPE;                                                     \
      auto kern = uniform_main_kernel<Dv, Kv, 8>;                                                                  \
      TCE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "umain smem");  \
      kern<<<grid, UM_THREADS, smem, (cudaStream_t)stream>>>(                                                      \
          tab_dev(t), ws, smp_traj, mean, init_pos, init_vel, pred_pairs, grad_mode, grad_logp, logp_old,          \
          advantage, grad_scale, loss_acc, logp, info, grad_mean, apart, (long long)B, (int)T, (int)P);            \
    } else {                                                                                                       \
      const size_t smem = UniMainSmem<Dv, Kv, 32>((int)P).total;                                                   \
      if (smem > SMEM_LIMIT) return TCE_ERR_UNSUPPORTED_SHAPE;                                                     \
      auto kern = uniform_main_kernel<Dv, Kv, 32>;                                                                 \
      TCE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "umain smem");  \
      kern<<<grid, UM_THREADS, smem, (cudaStream_t)stream>>>(                                                      \
          tab_dev(t), ws, smp_traj, mean, init_pos, init_vel, pred_pairs, grad_mode, grad_logp, logp_old,          \
          advantage, grad_scale, loss_acc, logp, info, grad_mean, apart, (long long)B, (int)T, (int)P);            \
    }                                                                                                              \
    TCE_CHECK_LAUNCH("uniform_main_kernel");                                                                       \
    return TCE_OK;                                                                                                 \
  }
  TCE_FOR_SHAPES(X)
#undef X
  return TCE_ERR_UNSUPPORTED_SHAPE;
}

extern "C" int tce_seglik_uniform_finish(const tce_tables_t *t, double *ws, const double *apart, int nparts,
                                         const float *L, const float *upstream, float *grad_L, double *grad_sigma,
                                         int64_t P, void *stream) {
  if (!t || !ws || !apart || nparts < 1 || (!grad_L && !grad_sigma) || (grad_L && !L) || P < 1)
    return TCE_ERR_INVALID_ARGUMENT;
#define X(Dv, Kv)                                                                                          \
  if (t->D == Dv && t->K1 == Kv) {                                                                         \
    using FL = FusedLayout<Dv, Kv>;                                                                        \
    const size_t smem = sizeof(float) * (2 * FL::NR4 * FL::LD + 2) +                                       \
                        sizeof(double) * ((size_t)P * FL::NT + 2 * P * Kv) + 16;                           \
    if (smem > SMEM_LIMIT) return TCE_ERR_UNSUPPORTED_SHAPE;                                               \
    auto kern = uniform_finish_kernel<Dv, Kv>;                                                             \
    TCE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "ufin smem"); \
    kern<<<(unsigned)P, UT, smem, (cudaStream_t)stream>>>(ws, apart, nparts, L, upstream, grad_L, grad_sigma, \
                                                          (int)P);                                         \
    TCE_CHECK_LAUNCH("uniform_finish_kernel");                                                             \
    return TCE_OK;                                                                                         \
  }
  TCE_FOR_SHAPES(X)
#undef X
  return TCE_ERR_UNSUPPORTED_SHAPE;
}

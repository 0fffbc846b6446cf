// (1b) ProDMP position covariances and standard deviations on any time grid, forward and backward.
// mp_pytorch ProDMP.get_traj_pos_cov / get_traj_pos_std for T time points per episode (T >= 1), rows DoF-major and
// time-minor:
//   Hp [T, K1]   scaled position basis rows with the episode's initial conditions (the rows of the likelihood)
//   F = H L      [D T, Dp], H block diagonal with one Hp block per DoF
//   C = F F^T + r I,   r = reg_rel * max over the whole call of diag(F F^T)
//   std[t, d] = sqrt(C[(d, t), (d, t)])
// C[(d, t), (d', u)] = Hp[t]^T Sigma_dd' Hp[u] with Sigma = L L^T: the inner dimension of the product is K1, not Dp, so
// the covariance forward does O(D^2 T^2 K1) fp64 work per episode for D^2 T^2 fp32 outputs and is bound by writing them.
// Backward (r is a constant, as in the likelihood's regulariser), with respect to L only:
//   cov: dL = tril(M L), M = H^T (G + G^T) H   (Dp x Dp, blocks M_dd' = Hp^T (G_dd' + G_d'd^T) Hp)
//   std: dL = tril(M L), M block diagonal, M_dd = sum_t (g_td / std_td) Hp[t] Hp[t]^T
// One factor shared by the batch (ldb_L = 0) sums M over the episodes in a fixed order (per-episode blocks, then one
// summing launch), so repeated calls give the same bits.  fp64 arithmetic throughout; no host synchronisation.
#include "tce_seglik.cuh"

namespace {

constexpr int TC_THREADS = 256;
constexpr int TC_TILE = 64;       // covariance forward: 64 x 64 output tile inside one (d, d') block, 4 x 4 per thread
constexpr int TB_TILE = 32;       // covariance backward: 32 x 32 tile of G inside one (d, d') block
constexpr size_t WS_HEAD = 2;     // work[0] = max diag(F F^T); the basis rows start 16 bytes in

// (I, J), I >= J, of the lower-triangular index t (64-bit: the tile count of a long horizon passes 2^31 / 8)
__device__ __forceinline__ void tri_decode64(long long t, int &I, int &J) {
  long long i = (long long)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
  while (i * (i + 1) / 2 > t) --i;
  while ((i + 1) * (i + 2) / 2 <= t) ++i;
  I = (int)i;
  J = (int)(t - i * (i + 1) / 2);
}

// the whole scaled basis row at time t: the arithmetic of basis_entry, one table lookup for all K1 entries
template <int K1>
__device__ __forceinline__ void basis_row(const TabDev &tb, const double *init_row, double t, double *h) {
  int i0; double w;
  time_to_index(tb, t, i0, w);
  const double y1 = lerp_t(tb.y1[i0], tb.y1[i0 + 1], w), y2 = lerp_t(tb.y2[i0], tb.y2[i0 + 1], w);
  const double idet = init_row[4];
  const double xi1 = (init_row[3] * y1 - init_row[2] * y2) * idet, xi2 = (init_row[0] * y2 - init_row[1] * y1) * idet;
#pragma unroll
  for (int j = 0; j < K1; ++j) {
    const double pj = lerp_t(tb.pos[(size_t)i0 * K1 + j], tb.pos[(size_t)(i0 + 1) * K1 + j], w);
    h[j] = (pj - xi1 * init_row[5 + j] - xi2 * init_row[5 + K1 + j]) * tb.scale[j];
  }
}

// ---- prep: one CTA per episode ------------------------------------------------------------------------------------
// MODE 0 (cov forward): basis rows -> work H [B][T][K1]; Sigma = L L^T (fp64, both triangles) -> work X [Dp][Dp] per
//        episode (one matrix for a shared factor, written by episode 0); max diag -> work[0].
// MODE 1 (std forward): diag(F F^T) -> work X [B][D][T]; max diag -> work[0].
// MODE 2 (backward): basis rows only.
template <int K1, int MODE>
__global__ void __launch_bounds__(TC_THREADS)
traj_prep_kernel(TabDev tb, const float *__restrict__ L, long long ldb_L, const float *__restrict__ times,
                 const float *__restrict__ init_time, double *__restrict__ work, int T, size_t off_x) {
  const int D = tb.D, Dp = D * K1, LD = Dp + 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double *init_row = reinterpret_cast<double *>(smem_raw);      // [5 + 2 K1] (+1)
  double *Sd = init_row + 6 + 2 * K1;                            // [D][K1][K1] diagonal blocks of Sigma
  float *Ls = reinterpret_cast<float *>(Sd + D * K1 * K1);       // [Dp][Dp + 1] lower triangle of L
  __shared__ double s_max[TC_THREADS / 32];
  const long long b = blockIdx.x;
  double *H = work + WS_HEAD;

  if (threadIdx.x <= K1) init_row_entry<K1>(tb, (double)init_time[b], threadIdx.x, init_row);
  if (MODE != 2) {
    const float *Lb = L + b * ldb_L;
    for (int e = threadIdx.x; e < Dp * Dp; e += blockDim.x) {
      const int i = e / Dp, c = e - i * Dp;
      Ls[i * LD + c] = c <= i ? Lb[e] : 0.0f;
    }
  }
  __syncthreads();
  if (MODE == 0 && (ldb_L != 0 || b == 0)) {
    double *S = work + off_x + (ldb_L ? (size_t)b * Dp * Dp : 0);
    for (int e = threadIdx.x; e < tri(Dp); e += blockDim.x) {
      int i, j;
      tri_decode(e, i, j);
      double v = 0.0;
      for (int k = 0; k <= j; ++k) v = fma((double)Ls[i * LD + k], (double)Ls[j * LD + k], v);
      S[(size_t)i * Dp + j] = v;
      S[(size_t)j * Dp + i] = v;
      const int d = i / K1;
      if (j >= d * K1) {
        const int a = i - d * K1, c = j - d * K1;
        Sd[(d * K1 + a) * K1 + c] = v;
        Sd[(d * K1 + c) * K1 + a] = v;
      }
    }
  } else if (MODE != 2) {
    for (int e = threadIdx.x; e < D * K1 * K1; e += blockDim.x) {
      const int d = e / (K1 * K1), r = e - d * K1 * K1, a = r / K1, c = r - a * K1;
      const int i = d * K1 + (a > c ? a : c), j = d * K1 + (a > c ? c : a);
      double v = 0.0;
      for (int k = 0; k <= j; ++k) v = fma((double)Ls[i * LD + k], (double)Ls[j * LD + k], v);
      Sd[e] = v;
    }
  }
  __syncthreads();

  double my_max = 0.0;
  const int n = MODE == 2 ? T : D * T;
  for (int e = threadIdx.x; e < n; e += blockDim.x) {
    const int d = e / T, t = e - d * T;
    double h[K1];
    basis_row<K1>(tb, init_row, (double)times[b * T + t], h);
    if (MODE != 1 && d == 0) {
      double *Hb = H + ((size_t)b * T + t) * K1;
#pragma unroll
      for (int j = 0; j < K1; ++j) Hb[j] = h[j];
    }
    if (MODE != 2) {
      const double *S = Sd + d * K1 * K1;
      double q = 0.0;
#pragma unroll
      for (int i = 0; i < K1; ++i) {
        double v = 0.0;
#pragma unroll
        for (int j = 0; j < K1; ++j) v = fma(S[i * K1 + j], h[j], v);
        q = fma(h[i], v, q);
      }
      my_max = fmax(my_max, q);
      if (MODE == 1) work[off_x + (size_t)b * D * T + e] = q;
    }
  }
  if (MODE != 2) {
    my_max = warp_max(my_max);
    if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = my_max;
    __syncthreads();
    if (threadIdx.x == 0) {
      double m = 0.0;
      for (int w = 0; w < TC_THREADS / 32; ++w) m = fmax(m, s_max[w]);
      atomic_max_pos_double(work, m);
    }
  }
}

// ---- covariance forward: one CTA per 64 x 64 tile of the lower tile triangle (mirrored on store) -------------------
// Tiles are aligned to the DoF blocks: tile row I = d * nT + ti covers rows (d, ti * 64 ..).  W = Hp_rows Sigma_dd'
// (64 x K1), then C_tile = W Hp_cols^T.  blockIdx.y strides over the episodes.
template <int K1>
__global__ void __launch_bounds__(TC_THREADS)
traj_cov_tile_kernel(const double *__restrict__ work, size_t off_s, long long lds, double reg_rel,
                     float *__restrict__ cov, int D, int T, long long B) {
  constexpr int TT = TC_TILE;
  __shared__ double Hr[TT][K1];
  __shared__ double HcT[K1][TT];
  __shared__ double Sg[K1][K1 + 1];
  __shared__ double W[TT][K1 + 1];
  __shared__ float Cs[TT][TT + 1];
  const int nT = (T + TT - 1) / TT, Dp = D * K1;
  const long long N = (long long)D * T;
  int I, J;
  tri_decode64(blockIdx.x, I, J);
  const int d = I / nT, t0 = (I - d * nT) * TT, dd = J / nT, u0 = (J - dd * nT) * TT;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const double r = reg_rel * work[0];
  const double *H = work + WS_HEAD;

  for (long long b = blockIdx.y; b < B; b += gridDim.y) {
    const double *Hb = H + (size_t)b * T * K1;
    const double *S = work + off_s + (size_t)b * lds;
    for (int e = threadIdx.x; e < TT * K1; e += blockDim.x) {
      const int q = e / K1, k = e - q * K1;
      Hr[q][k] = t0 + q < T ? Hb[(size_t)(t0 + q) * K1 + k] : 0.0;
      HcT[k][q] = u0 + q < T ? Hb[(size_t)(u0 + q) * K1 + k] : 0.0;
    }
    for (int e = threadIdx.x; e < K1 * K1; e += blockDim.x) {
      const int k = e / K1, c = e - k * K1;
      Sg[k][c] = S[(size_t)(d * K1 + k) * Dp + dd * K1 + c];
    }
    __syncthreads();
    for (int e = threadIdx.x; e < TT * K1; e += blockDim.x) {
      const int q = e / K1, c = e - q * K1;
      double v = 0.0;
#pragma unroll
      for (int k = 0; k < K1; ++k) v = fma(Hr[q][k], Sg[k][c], v);
      W[q][c] = v;
    }
    __syncthreads();
    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
#pragma unroll
    for (int k = 0; k < K1; ++k) {
      double hc[4], w[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) hc[j] = HcT[k][tx + 16 * j];
#pragma unroll
      for (int i = 0; i < 4; ++i) w[i] = W[ty + 16 * i][k];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fma(w[i], hc[j], acc[i][j]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int q = ty + 16 * i, c = tx + 16 * j;
        const bool on_diag = I == J && q == c;
        Cs[q][c] = (float)(on_diag ? acc[i][j] + r : acc[i][j]);
      }
    __syncthreads();
    float *Cb = cov + (size_t)b * (size_t)N * (size_t)N;
    const int nr = min(TT, T - t0), nc = min(TT, T - u0);
    for (int e = threadIdx.x; e < TT * TT; e += blockDim.x) {
      const int q = e / TT, c = e - q * TT;
      if (q < nr && c < nc) Cb[(size_t)(d * T + t0 + q) * N + dd * T + u0 + c] = Cs[q][c];
    }
    if (I != J)
      for (int e = threadIdx.x; e < TT * TT; e += blockDim.x) {
        const int c = e / TT, q = e - c * TT;
        if (q < nr && c < nc) Cb[(size_t)(dd * T + u0 + c) * N + d * T + t0 + q] = Cs[q][c];
      }
    __syncthreads();
  }
}

// std[b, t, d] = sqrt(diag + r)
__global__ void __launch_bounds__(TC_THREADS)
traj_std_finish_kernel(const double *__restrict__ work, size_t off_x, double reg_rel, float *__restrict__ out, int D,
                       int T, long long n) {
  const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= n) return;
  const long long bt = o / D, b = bt / T;
  const int d = (int)(o - bt * D), t = (int)(bt - b * T);
  out[o] = (float)sqrt(work[off_x + (size_t)b * D * T + (size_t)d * T + t] + reg_rel * work[0]);
}

// ---- covariance backward: M_dd' = Hp^T (G_dd' + G_d'd^T) Hp for d >= d', one CTA per (d, d') block ----------------
// -> work X [B][tri(D)][K1][K1] (block tri_idx(d, d')).  The T x T block is walked in 32 x 32 tiles in a fixed order.
template <int K1>
__global__ void __launch_bounds__(TC_THREADS)
traj_cov_bwd_kernel(const double *__restrict__ work_h, const float *__restrict__ G, double *__restrict__ X, int D,
                    int T, long long B) {
  constexpr int TT = TB_TILE;
  __shared__ double Ss[TT][TT + 1];
  __shared__ double Hr[TT][K1];
  __shared__ double Hc[TT][K1];
  __shared__ double Y[K1][TT + 1];
  int d, dd;
  tri_decode(blockIdx.x, d, dd);
  const int nT = (T + TT - 1) / TT, NB = tri(D);
  const long long N = (long long)D * T;
  const int k = threadIdx.x / K1, kk = threadIdx.x - k * K1;      // this thread's entry of M_dd' (if < K1^2)

  for (long long b = blockIdx.y; b < B; b += gridDim.y) {
    const double *Hb = work_h + (size_t)b * T * K1;
    const float *Gb = G + (size_t)b * (size_t)N * (size_t)N;
    double m = 0.0;
    for (int ti = 0; ti < nT; ++ti)
      for (int tj = 0; tj < nT; ++tj) {
        const int t0 = ti * TT, u0 = tj * TT, nr = min(TT, T - t0), nc = min(TT, T - u0);
        for (int e = threadIdx.x; e < TT * K1; e += blockDim.x) {
          const int q = e / K1, j = e - q * K1;
          Hr[q][j] = q < nr ? Hb[(size_t)(t0 + q) * K1 + j] : 0.0;
          Hc[q][j] = q < nc ? Hb[(size_t)(u0 + q) * K1 + j] : 0.0;
        }
        for (int e = threadIdx.x; e < TT * TT; e += blockDim.x) {
          const int q = e / TT, c = e - q * TT;
          Ss[q][c] = q < nr && c < nc ? (double)Gb[(size_t)(d * T + t0 + q) * N + dd * T + u0 + c] : 0.0;
        }
        __syncthreads();
        for (int e = threadIdx.x; e < TT * TT; e += blockDim.x) {
          const int c = e / TT, q = e - c * TT;
          if (q < nr && c < nc) Ss[q][c] += (double)Gb[(size_t)(dd * T + u0 + c) * N + d * T + t0 + q];
        }
        __syncthreads();
        for (int e = threadIdx.x; e < K1 * TT; e += blockDim.x) {        // Y = Hr^T S   [K1][TT]
          const int j = e / TT, c = e - j * TT;
          double v = 0.0;
#pragma unroll 8
          for (int q = 0; q < TT; ++q) v = fma(Hr[q][j], Ss[q][c], v);
          Y[j][c] = v;
        }
        __syncthreads();
        if (threadIdx.x < K1 * K1) {
#pragma unroll 8
          for (int c = 0; c < TT; ++c) m = fma(Y[k][c], Hc[c][kk], m);
        }
        __syncthreads();
      }
    if (threadIdx.x < K1 * K1) X[((size_t)b * NB + blockIdx.x) * K1 * K1 + threadIdx.x] = m;
  }
}

// ---- std backward: M_dd = sum_t (g_td / std_td) Hp[t] Hp[t]^T -> work X [B][D][K1][K1]; one CTA per episode ----------
template <int K1>
__global__ void __launch_bounds__(TC_THREADS)
traj_std_bwd_kernel(const double *__restrict__ work_h, const float *__restrict__ sd, const float *__restrict__ g,
                    double *__restrict__ X, int D, int T) {
  const long long b = blockIdx.x;
  const double *Hb = work_h + (size_t)b * T * K1;
  const float *sb = sd + (size_t)b * T * D, *gb = g + (size_t)b * T * D;
  for (int e = threadIdx.x; e < D * K1 * K1; e += blockDim.x) {
    const int d = e / (K1 * K1), r = e - d * K1 * K1, i = r / K1, j = r - i * K1;
    double v = 0.0;
    for (int t = 0; t < T; ++t) {
      const double w = (double)gb[(size_t)t * D + d] / (double)sb[(size_t)t * D + d];
      v = fma(w * Hb[(size_t)t * K1 + i], Hb[(size_t)t * K1 + j], v);
    }
    X[(size_t)b * D * K1 * K1 + e] = v;
  }
}

// sum over the nparts per-episode blocks in a fixed order (shared factor): thread per entry
__global__ void __launch_bounds__(256)
traj_part_sum_kernel(const double *__restrict__ part, long long nparts, int ne, double *__restrict__ out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= ne) return;
  double s = 0.0;
  for (long long c = 0; c < nparts; ++c) s += part[(size_t)c * ne + e];
  out[e] = s;
}

// ---- grad_L = tril(M L) per episode (or once for a shared factor, on the summed M) -----------------------------------
// DIAG: M block diagonal, X [D][K1][K1]; else X [tri(D)][K1][K1] holds M_dd' for d >= d' (M_d'd = M_dd'^T).
template <int K1, bool DIAG>
__global__ void __launch_bounds__(TC_THREADS)
traj_dl_kernel(const double *__restrict__ X, const float *__restrict__ L, long long ldb_L, float *__restrict__ grad_L,
               int D) {
  const int Dp = D * K1, LD = Dp + 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double *Ms = reinterpret_cast<double *>(smem_raw);                       // [Dp][Dp] (DIAG: [D][K1][K1])
  float *Ls = reinterpret_cast<float *>(Ms + (DIAG ? D * K1 * K1 : Dp * Dp)); // [Dp][Dp + 1]
  const long long b = blockIdx.x;
  const double *Xb = X + (size_t)b * (DIAG ? D : tri(D)) * K1 * K1;
  const float *Lb = L + b * ldb_L;
  for (int e = threadIdx.x; e < Dp * Dp; e += blockDim.x) {
    const int i = e / Dp, c = e - i * Dp;
    Ls[i * LD + c] = c <= i ? Lb[e] : 0.0f;
  }
  if (DIAG) {
    for (int e = threadIdx.x; e < D * K1 * K1; e += blockDim.x) Ms[e] = Xb[e];
  } else {
    for (int e = threadIdx.x; e < Dp * Dp; e += blockDim.x) {
      const int i = e / Dp, c = e - i * Dp, d = i / K1, dd = c / K1, a = i - d * K1, q = c - dd * K1;
      Ms[e] = d >= dd ? Xb[(size_t)tri_idx(d, dd) * K1 * K1 + a * K1 + q]
                      : Xb[(size_t)tri_idx(dd, d) * K1 * K1 + q * K1 + a];
    }
  }
  __syncthreads();
  float *gb = grad_L + (size_t)b * Dp * Dp;
  for (int e = threadIdx.x; e < Dp * Dp; e += blockDim.x) {
    const int i = e / Dp, c = e - i * Dp;
    double v = 0.0;
    if (c <= i) {
      if (DIAG) {
        const int d = i / K1, a = i - d * K1, k0 = d * K1 > c ? d * K1 : c;
        for (int k = k0; k < d * K1 + K1; ++k) v = fma(Ms[(d * K1 + a) * K1 + k - d * K1], (double)Ls[k * LD + c], v);
      } else {
        for (int k = c; k < Dp; ++k) v = fma(Ms[(size_t)i * Dp + k], (double)Ls[k * LD + c], v);
      }
    }
    gb[e] = (float)v;
  }
}

// ---- host side ----------------------------------------------------------------------------------------------------
enum { ENTRY_COV_FWD = 0, ENTRY_COV_BWD = 1, ENTRY_STD_FWD = 2, ENTRY_STD_BWD = 3 };

bool shape_ok(const tce_tables_t *t) {
  return t->D >= 1 && t->D <= TCE_MAX_DOF && t->K1 >= 2 && t->K1 <= TCE_MAX_K1 && t->D * t->K1 <= TCE_MAX_TABLE_DP;
}

// doubles of the per-entry region behind the head and the basis rows
size_t x_doubles(const tce_tables_t *t, int64_t B, int64_t T, int64_t ldb_L, int entry) {
  const size_t D = t->D, K1 = t->K1, Dp = D * K1;
  switch (entry) {
    case ENTRY_COV_FWD: return (ldb_L ? (size_t)B : 1) * Dp * Dp;
    case ENTRY_COV_BWD: return ((size_t)B + (ldb_L ? 0 : 1)) * (D * (D + 1) / 2) * K1 * K1;
    case ENTRY_STD_FWD: return (size_t)B * D * (size_t)T;
    default: return ((size_t)B + (ldb_L ? 0 : 1)) * D * K1 * K1;
  }
}

size_t prep_smem(int D, int K1) {
  const int Dp = D * K1;
  return sizeof(double) * (6 + 2 * K1 + D * K1 * K1) + sizeof(float) * Dp * (Dp + 1);
}

template <int K1, int MODE>
int prep_launch(const tce_tables_t *t, const float *L, int64_t ldb_L, const float *times, const float *init_time,
                double *work, int64_t B, int64_t T, size_t off_x, cudaStream_t st) {
  const size_t smem = MODE == 2 ? sizeof(double) * (6 + 2 * K1) : prep_smem(t->D, K1);
  TCE_CUDA(cudaFuncSetAttribute(traj_prep_kernel<K1, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
           "traj prep smem attr");
  traj_prep_kernel<K1, MODE><<<(unsigned)B, TC_THREADS, smem, st>>>(tab_dev(t), L, ldb_L, times, init_time, work,
                                                                    (int)T, off_x);
  TCE_CHECK_LAUNCH("traj_prep_kernel");
  return TCE_OK;
}

// grad_L = tril(M L) from the per-episode blocks at X (or their sum over the batch for a shared factor)
template <int K1, bool DIAG>
int dl_launch(const tce_tables_t *t, double *X, const float *L, int64_t ldb_L, float *grad_L, int64_t B,
              cudaStream_t st) {
  const int D = t->D, Dp = D * K1, ne = (DIAG ? D : tri(D)) * K1 * K1;
  const double *Xs = X;
  if (ldb_L == 0 && B > 1) {
    double *sum = X + (size_t)B * ne;
    traj_part_sum_kernel<<<(ne + 255) / 256, 256, 0, st>>>(X, (long long)B, ne, sum);
    TCE_CHECK_LAUNCH("traj_part_sum_kernel");
    Xs = sum;
  }
  const int64_t grid = ldb_L == 0 ? 1 : B;
  const size_t smem = sizeof(double) * (DIAG ? D * K1 * K1 : Dp * Dp) + sizeof(float) * Dp * (Dp + 1);
  TCE_CUDA(cudaFuncSetAttribute(traj_dl_kernel<K1, DIAG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
           "traj dl smem attr");
  traj_dl_kernel<K1, DIAG><<<(unsigned)grid, TC_THREADS, smem, st>>>(Xs, L, ldb_L, grad_L, D);
  TCE_CHECK_LAUNCH("traj_dl_kernel");
  return TCE_OK;
}

unsigned episode_grid(int64_t B) { return (unsigned)(B < 65535 ? B : 65535); }

int check_args(const tce_tables_t *t, const float *L, int64_t ldb_L, const float *times, const float *init_time,
               const void *work, int64_t B, int64_t T) {
  if (!t || !L || !times || !init_time || !work || B < 0 || T < 1 || ldb_L < 0 || B > INT32_MAX || T > INT32_MAX)
    return TCE_ERR_INVALID_ARGUMENT;
  if (ldb_L != 0 && ldb_L < (int64_t)t->D * t->K1 * t->D * t->K1) return TCE_ERR_INVALID_ARGUMENT;
  return shape_ok(t) ? TCE_OK : TCE_ERR_UNSUPPORTED_SHAPE;
}

}  // namespace

extern "C" size_t tce_prodmp_traj_cov_work_bytes(const tce_tables_t *t, int64_t B, int64_t T, int64_t ldb_L,
                                                 int entry) {
  if (!t || B < 0 || T < 1 || ldb_L < 0 || entry < ENTRY_COV_FWD || entry > ENTRY_STD_BWD || !shape_ok(t)) return 0;
  return sizeof(double) * (WS_HEAD + (size_t)B * (size_t)T * t->K1 + x_doubles(t, B, T, ldb_L, entry));
}

extern "C" int tce_prodmp_traj_cov_fwd(const tce_tables_t *t, const float *L, int64_t ldb_L, const float *times,
                                       const float *init_time, double reg_rel, void *work, float *cov, int64_t B,
                                       int64_t T, void *stream) {
  if (B == 0) return TCE_OK;
  int rc = check_args(t, L, ldb_L, times, init_time, work, B, T);
  if (rc != TCE_OK) return rc;
  if (!cov) return TCE_ERR_INVALID_ARGUMENT;
  const int64_t nT = (T + TC_TILE - 1) / TC_TILE, R = t->D * nT, tiles = R * (R + 1) / 2;
  if (tiles > INT32_MAX) return TCE_ERR_UNSUPPORTED_SHAPE;
  cudaStream_t st = (cudaStream_t)stream;
  double *w = (double *)work;
  const size_t off_x = WS_HEAD + (size_t)B * T * t->K1;
  TCE_CUDA(cudaMemsetAsync(w, 0, sizeof(double), st), "traj cov max reset");
  rc = TCE_ERR_UNSUPPORTED_SHAPE;
  TCE_DISPATCH_K1(t->K1, rc = (prep_launch<K1, 0>(t, L, ldb_L, times, init_time, w, B, T, off_x, st)));
  if (rc != TCE_OK) return rc;
  const long long lds = ldb_L ? (long long)t->D * t->K1 * t->D * t->K1 : 0;
  const dim3 grid((unsigned)tiles, episode_grid(B));
  TCE_DISPATCH_K1(t->K1, (traj_cov_tile_kernel<K1><<<grid, TC_THREADS, 0, st>>>(w, off_x, lds, reg_rel, cov, t->D,
                                                                                 (int)T, (long long)B)));
  TCE_CHECK_LAUNCH("traj_cov_tile_kernel");
  return TCE_OK;
}

extern "C" int tce_prodmp_traj_cov_bwd(const tce_tables_t *t, const float *L, int64_t ldb_L, const float *times,
                                       const float *init_time, const float *grad_cov, void *work, float *grad_L,
                                       int64_t B, int64_t T, void *stream) {
  if (B == 0) return TCE_OK;
  int rc = check_args(t, L, ldb_L, times, init_time, work, B, T);
  if (rc != TCE_OK) return rc;
  if (!grad_cov || !grad_L) return TCE_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
  double *w = (double *)work, *X = w + WS_HEAD + (size_t)B * T * t->K1;
  rc = TCE_ERR_UNSUPPORTED_SHAPE;
  TCE_DISPATCH_K1(t->K1, rc = (prep_launch<K1, 2>(t, L, ldb_L, times, init_time, w, B, T, 0, st)));
  if (rc != TCE_OK) return rc;
  const dim3 grid((unsigned)tri(t->D), episode_grid(B));
  TCE_DISPATCH_K1(t->K1, (traj_cov_bwd_kernel<K1><<<grid, TC_THREADS, 0, st>>>(w + WS_HEAD, grad_cov, X, t->D,
                                                                                (int)T, (long long)B)));
  TCE_CHECK_LAUNCH("traj_cov_bwd_kernel");
  TCE_DISPATCH_K1(t->K1, return (dl_launch<K1, false>(t, X, L, ldb_L, grad_L, B, st)));
  return TCE_ERR_UNSUPPORTED_SHAPE;
}

extern "C" int tce_prodmp_traj_std_fwd(const tce_tables_t *t, const float *L, int64_t ldb_L, const float *times,
                                       const float *init_time, double reg_rel, void *work, float *std_out, int64_t B,
                                       int64_t T, void *stream) {
  if (B == 0) return TCE_OK;
  int rc = check_args(t, L, ldb_L, times, init_time, work, B, T);
  if (rc != TCE_OK) return rc;
  if (!std_out) return TCE_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
  double *w = (double *)work;
  const size_t off_x = WS_HEAD + (size_t)B * T * t->K1;
  TCE_CUDA(cudaMemsetAsync(w, 0, sizeof(double), st), "traj std max reset");
  rc = TCE_ERR_UNSUPPORTED_SHAPE;
  TCE_DISPATCH_K1(t->K1, rc = (prep_launch<K1, 1>(t, L, ldb_L, times, init_time, w, B, T, off_x, st)));
  if (rc != TCE_OK) return rc;
  const long long n = (long long)B * T * t->D;
  traj_std_finish_kernel<<<(unsigned)((n + TC_THREADS - 1) / TC_THREADS), TC_THREADS, 0, st>>>(w, off_x, reg_rel,
                                                                                                std_out, t->D, (int)T, n);
  TCE_CHECK_LAUNCH("traj_std_finish_kernel");
  return TCE_OK;
}

extern "C" int tce_prodmp_traj_std_bwd(const tce_tables_t *t, const float *L, int64_t ldb_L, const float *times,
                                       const float *init_time, const float *std_in, const float *grad_std, void *work,
                                       float *grad_L, int64_t B, int64_t T, void *stream) {
  if (B == 0) return TCE_OK;
  int rc = check_args(t, L, ldb_L, times, init_time, work, B, T);
  if (rc != TCE_OK) return rc;
  if (!std_in || !grad_std || !grad_L) return TCE_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
  double *w = (double *)work, *X = w + WS_HEAD + (size_t)B * T * t->K1;
  rc = TCE_ERR_UNSUPPORTED_SHAPE;
  TCE_DISPATCH_K1(t->K1, rc = (prep_launch<K1, 2>(t, L, ldb_L, times, init_time, w, B, T, 0, st)));
  if (rc != TCE_OK) return rc;
  TCE_DISPATCH_K1(t->K1, (traj_std_bwd_kernel<K1><<<(unsigned)B, TC_THREADS, 0, st>>>(w + WS_HEAD, std_in, grad_std,
                                                                                       X, t->D, (int)T)));
  TCE_CHECK_LAUNCH("traj_std_bwd_kernel");
  TCE_DISPATCH_K1(t->K1, return (dl_launch<K1, true>(t, X, L, ldb_L, grad_L, B, st)));
  return TCE_ERR_UNSUPPORTED_SHAPE;
}

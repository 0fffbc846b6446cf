// (2) Gaussian policy over the MP parameters: rsample, batched small Cholesky (fwd/bwd), the
// vector -> Cholesky policy head and the per-episode Gaussian scalars (maha, trace, logdet, entropy).
// Replaces black_box_policy.py:58-224 (torch MultivariateNormal / cholesky_solve / solve_triangular),
// abstract_policy.py:166-187 + util_matrix.py:12-33 (head) and torch.linalg.cholesky (util_matrix.py:133).
// One CTA per matrix, matrices staged in shared memory, warp shuffles for the reductions.
#include <math.h>

#include "tce_bulk.cuh"
#include "tce_common.cuh"

namespace {

// ---------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al.) -> one standard normal per element (Box-Muller)
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
  const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
  const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
  const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
  c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
}
__device__ __forceinline__ float philox_normal(uint64_t seed, uint64_t offset, uint64_t idx) {
  uint32_t c[4] = {(uint32_t)idx, (uint32_t)(idx >> 32), (uint32_t)offset, (uint32_t)(offset >> 32)};
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    philox_round(c, k0, k1);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  const float u0 = ((float)c[0] + 1.0f) * 2.3283064365386963e-10f;   // (0, 1]
  const float u1 = (float)c[1] * 2.3283064365386963e-10f;            // [0, 1)
  return sqrtf(-2.0f * logf(u0)) * cospif(2.0f * u1);
}

// out[b] = mean[b] + L[b] eps[b];  one CTA (128 threads) per episode, warp per row, lanes over columns
__global__ void __launch_bounds__(128)
rsample_kernel(const float *__restrict__ mean, const float *__restrict__ L, long long ldb_L,
               const float *__restrict__ eps, uint64_t seed, uint64_t offset, float *__restrict__ out, int n,
               long long first) {
  extern __shared__ float s_eps[];
  const long long b = first + blockIdx.x;
  for (int j = threadIdx.x; j < n; j += blockDim.x)
    s_eps[j] = eps ? eps[b * n + j] : philox_normal(seed, offset, (uint64_t)(b * n + j));
  __syncthreads();
  const float *Lb = L + b * ldb_L;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int i = warp; i < n; i += nw) {
    float acc = 0.f;
    for (int j = lane; j <= i; j += 32) acc = fmaf(Lb[(size_t)i * n + j], s_eps[j], acc);
    acc = warp_sum(acc);
    if (lane == 0) out[b * n + i] = mean[b * n + i] + acc;
  }
}

// Per-episode factors, odd n <= 64 (box pushing: 63): the factors of RS_G consecutive episodes are ONE contiguous,
// 16-byte-aligned block of HBM (4 n^2 floats), fetched by one bulk asynchronous copy per CTA iteration into shared
// memory; thread (episode, row) then forms its row of L eps from shared memory (row stride n is odd: the 32 rows of a
// warp hit 32 banks).  One buffer per CTA, three CTAs per SM: while one CTA computes, the copies of the other two are in
// flight (190 KB per SM requested at any time).  The kernel above fetches the lower triangle row by row (252-byte
// rows: partial sectors, 63 dependent-latency rounds per warp); this one moves the dense block at copy-engine speed.
constexpr int RS_G = 4;
__global__ void __launch_bounds__(RS_G * 64)
rsample_bulk_kernel(const float *__restrict__ mean, const float *__restrict__ L, const float *__restrict__ eps,
                    uint64_t seed, uint64_t offset, float *__restrict__ out, int n, long long groups) {
  extern __shared__ __align__(128) unsigned char rs_raw[];
  __shared__ __align__(8) uint64_t bar;
  float *sL = reinterpret_cast<float *>(rs_raw);          // [RS_G][n][n]
  float *sE = sL + (size_t)RS_G * n * n;                   // [RS_G][64]
  const int e = threadIdx.x >> 6, i = threadIdx.x & 63;
  const uint32_t bytes = (uint32_t)(RS_G * n * n * sizeof(float));
  if (threadIdx.x == 0) mbar_init(&bar, 1);
  __syncthreads();
  uint32_t parity = 0;
  for (long long g = blockIdx.x; g < groups; g += gridDim.x) {
    if (threadIdx.x == 0) {
      mbar_arrive_expect_tx(&bar, bytes);
      bulk_copy_g2s(sL, L + (size_t)g * RS_G * n * n, bytes, &bar);
    }
    const long long b = g * RS_G + e;
    float m = 0.f;
    if (i < n) {
      sE[e * 64 + i] = eps ? eps[b * n + i] : philox_normal(seed, offset, (uint64_t)(b * n + i));
      m = mean[b * n + i];
    }
    __syncthreads();
    mbar_wait(&bar, parity);
    parity ^= 1;
    if (i < n) {
      const float *row = sL + (size_t)e * n * n + i * n, *ev = sE + e * 64;
      float a0 = 0.f, a1 = 0.f;
      int j = 0;
      for (; j + 1 <= i; j += 2) {
        a0 = fmaf(row[j], ev[j], a0);
        a1 = fmaf(row[j + 1], ev[j + 1], a1);
      }
      if (j <= i) a0 = fmaf(row[j], ev[j], a0);
      out[b * n + i] = m + (a0 + a1);
    }
    __syncthreads();                    // every read of sL / sE is done before the next copy overwrites them
  }
}

// ---------------------------------------------------------------------------------------------------
// Cholesky forward: left-looking, thread per row, fp64 accumulation, one barrier pair per column
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
chol_fwd_kernel(const float *__restrict__ A, float *__restrict__ Lout, int32_t *__restrict__ info, int n) {
  extern __shared__ float sL[];            // [n][n+1]
  __shared__ int s_bad;
  const int LD = n + 1;
  const long long b = blockIdx.x;
  const float *Ab = A + (size_t)b * n * n;
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) sL[(e / n) * LD + e % n] = Ab[e];
  if (threadIdx.x == 0) s_bad = 0;
  __syncthreads();
  const int i = threadIdx.x;
  for (int j = 0; j < n; ++j) {
    if (i == j) {
      double d = (double)sL[j * LD + j];
      for (int k = 0; k < j; ++k) d -= (double)sL[j * LD + k] * (double)sL[j * LD + k];
      if (!(d > 0.0) && s_bad == 0) s_bad = j + 1;
      sL[j * LD + j] = (float)sqrt(d);
    }
    __syncthreads();
    if (i > j && i < n) {
      double v = (double)sL[i * LD + j];
      for (int k = 0; k < j; ++k) v -= (double)sL[i * LD + k] * (double)sL[j * LD + k];
      sL[i * LD + j] = (float)(v / (double)sL[j * LD + j]);
    }
    __syncthreads();
  }
  float *Lb = Lout + (size_t)b * n * n;
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int r = e / n, c = e % n;
    Lb[e] = c <= r ? sL[r * LD + c] : 0.f;
  }
  if (info && threadIdx.x == 0) info[b] = s_bad;
}

// Cholesky backward: grad_A = sym(S^-T Phi(S^T Gbar) S^-1), Phi = tril with halved diagonal.
// fp64 in shared memory, thread per column / row for the two triangular solves.
__global__ void __launch_bounds__(128)
chol_bwd_kernel(const float *__restrict__ S, const float *__restrict__ gS, float *__restrict__ gA, int n) {
  extern __shared__ double sd[];
  const int LD = n + 1;
  double *sS = sd, *sG = sd + n * LD, *sM = sG + n * LD;
  const long long b = blockIdx.x;
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int r = e / n, c = e % n;
    sS[r * LD + c] = c <= r ? (double)S[(size_t)b * n * n + e] : 0.0;
    sG[r * LD + c] = c <= r ? (double)gS[(size_t)b * n * n + e] : 0.0;
  }
  __syncthreads();
  // M = Phi(S^T G): M[i][j] = sum_{k >= i} S[k][i] G[k][j], i >= j
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, j = e % n;
    double v = 0.0;
    if (j <= i) {
      for (int k = i; k < n; ++k) v = fma(sS[k * LD + i], sG[k * LD + j], v);
      if (i == j) v *= 0.5;
    }
    sM[i * LD + j] = v;
  }
  __syncthreads();
  // Y = S^-T M : column c, back substitution (thread per column) -> sG
  for (int c = threadIdx.x; c < n; c += blockDim.x) {
    for (int i = n - 1; i >= 0; --i) {
      double v = sM[i * LD + c];
      for (int k = i + 1; k < n; ++k) v = fma(-sS[k * LD + i], sG[k * LD + c], v);
      sG[i * LD + c] = v / sS[i * LD + i];
    }
  }
  __syncthreads();
  // X = Y S^-1 : row r, X[r][c] = (Y[r][c] - sum_{k > c} X[r][k] S[k][c]) / S[c][c] (thread per row) -> sM
  for (int r = threadIdx.x; r < n; r += blockDim.x) {
    for (int c = n - 1; c >= 0; --c) {
      double v = sG[r * LD + c];
      for (int k = c + 1; k < n; ++k) v = fma(-sM[r * LD + k], sS[k * LD + c], v);
      sM[r * LD + c] = v / sS[c * LD + c];
    }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int r = e / n, c = e % n;
    gA[(size_t)b * n * n + e] = (float)(0.5 * (sM[r * LD + c] + sM[c * LD + r]));
  }
}

// ---------------------------------------------------------------------------------------------------
// policy head
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ float softplus_f(float x) { return x > 20.f ? x : log1pf(expf(x)); }

__global__ void __launch_bounds__(256)
head_fwd_kernel(const float *__restrict__ vec, long long ldb_vec, float min_std, float *__restrict__ L, int n) {
  const long long b = blockIdx.x;
  const float *v = vec + b * ldb_vec;
  float *Lb = L + (size_t)b * n * n;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int r = warp; r < n; r += nw) {
    const float *off = v + n + r * (r - 1) / 2;
    for (int c = lane; c < n; c += 32) {
      float o = 0.f;
      if (c < r) o = off[c];
      else if (c == r) o = softplus_f(v[r]) + min_std;
      Lb[r * n + c] = o;
    }
  }
}

// Per-episode vectors (contextual covariance), large batches: both sides of the head are contiguous blocks of HBM --
// HD_G vectors in (HD_G nvec floats), HD_G dense factors out (HD_G n^2 floats), each a multiple of 16 bytes.  The
// vectors arrive by one bulk asynchronous copy (mbarrier completion; group k + 1 is requested while group k is written
// out); the CTA scatters the packed rows into a dense shared-memory image of the factors (lower triangle only: the
// zeros above it are written once; the softplus diagonal by one thread per entry, not inside the row loop) and writes
// that image with 128-bit stores, 512 contiguous bytes per warp instruction.  Two CTAs per SM.  The kernel above
// writes 252-byte rows with two partial store instructions each, after a dependent global load per row.
// (A bulk copy OUT of shared memory was measured first: 857 us for 65536 episodes against 606 us for the row kernel.)
constexpr int HD_G = 4;
__global__ void __launch_bounds__(256)
head_fwd_bulk_kernel(const float *__restrict__ vec, float min_std, float *__restrict__ L, int n, long long groups) {
  extern __shared__ __align__(128) unsigned char hd_raw[];
  __shared__ __align__(8) uint64_t bar;
  const int nvec = n + n * (n - 1) / 2, nn = n * n;
  float *sO = reinterpret_cast<float *>(hd_raw);            // [HD_G][n][n]
  float *sV = sO + (size_t)HD_G * nn;                       // [HD_G][nvec]
  const uint32_t in_bytes = (uint32_t)(HD_G * nvec * sizeof(float));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    if ((long long)blockIdx.x < groups) {
      mbar_arrive_expect_tx(&bar, in_bytes);
      bulk_copy_g2s(sV, vec + (size_t)blockIdx.x * HD_G * nvec, in_bytes, &bar);
    }
  }
  // the strict upper triangles of the image are zero for every group: written once
  for (int q = threadIdx.x; q < HD_G * nn; q += blockDim.x) sO[q] = 0.f;
  __syncthreads();
  uint32_t parity = 0;
  const int per_e = nw / HD_G, e = warp / per_e;             // (nw is a multiple of HD_G) warps of one episode
  for (long long g = blockIdx.x; g < groups; g += gridDim.x) {
    mbar_wait(&bar, parity);
    parity ^= 1;
    for (int r = 1 + warp % per_e; r < n; r += per_e) {      // row r of episode e: r packed floats -> r dense ones
      const float *off = sV + e * nvec + n + r * (r - 1) / 2;
      float *o = sO + e * nn + r * n;
      for (int c = lane; c < r; c += 32) o[c] = off[c];
    }
    for (int d = threadIdx.x; d < HD_G * n; d += blockDim.x) {
      const int ed = d / n, r = d - ed * n;
      sO[ed * nn + r * n + r] = softplus_f(sV[ed * nvec + r]) + min_std;
    }
    __syncthreads();                    // image complete, sV free
    if (threadIdx.x == 0 && g + gridDim.x < groups) {
      mbar_arrive_expect_tx(&bar, in_bytes);
      bulk_copy_g2s(sV, vec + (size_t)(g + gridDim.x) * HD_G * nvec, in_bytes, &bar);
    }
    float4 *dst = reinterpret_cast<float4 *>(L + (size_t)g * HD_G * nn);
    const float4 *src = reinterpret_cast<const float4 *>(sO);
    for (int q = threadIdx.x; q < HD_G * nn / 4; q += blockDim.x) dst[q] = src[q];
    __syncthreads();                    // image read out before the next group overwrites it
  }
}

// grid (ceil(nvec/128), batch chunks); grad_vec zero-initialised by the launcher when reducing
__global__ void head_bwd_kernel(const float *__restrict__ vec, long long ldb_vec, const float *__restrict__ gL,
                                float *__restrict__ gvec, long long B, int n, int chunk) {
  const int nvec = n + n * (n - 1) / 2;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nvec) return;
  int r, c;
  if (e < n) { r = c = e; }
  else {
    const int o = e - n;
    r = (int)((sqrtf(8.0f * (float)o + 1.0f) + 1.0f) * 0.5f);
    while (r * (r - 1) / 2 > o) --r;
    while ((r + 1) * r / 2 <= o) ++r;
    c = o - r * (r - 1) / 2;
  }
  const long long b0 = (long long)blockIdx.y * chunk;
  const long long b1 = b0 + chunk < B ? b0 + chunk : B;
  if (ldb_vec == 0) {
    float acc = 0.f;
    for (long long b = b0; b < b1; ++b) acc += gL[(size_t)b * n * n + r * n + c];
    if (r == c) acc *= 1.f / (1.f + expf(-vec[e]));
    atomicAdd(gvec + e, acc);
  } else {
    for (long long b = b0; b < b1; ++b) {
      float g = gL[(size_t)b * n * n + r * n + c];
      if (r == c) g *= 1.f / (1.f + expf(-vec[b * ldb_vec + e]));
      gvec[b * nvec + e] = g;
    }
  }
}

// Diagonal head (std_only): L = diag(softplus(v) + min_std), zeros elsewhere; one thread per entry of the dense factor
__global__ void __launch_bounds__(256)
head_diag_fwd_kernel(const float *__restrict__ vec, long long ldb_vec, float min_std, float *__restrict__ L,
                     long long B, int n) {
  const long long nn = (long long)n * n, total = B * nn;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long b = e / nn;
    const int r = (int)(e - b * nn), i = r / n;
    L[e] = (r == i * (n + 1)) ? softplus_f(vec[b * ldb_vec + i]) + min_std : 0.f;
  }
}

// grad_vec[b, i] = grad_L[b, i, i] * sigmoid(v[b, i]).  ldb_vec == 0 (one shared vector): CTA per i sums the batch in a
// fixed order (strided partial sums, then a tree) -- deterministic, no atomics.
__global__ void __launch_bounds__(256)
head_diag_bwd_kernel(const float *__restrict__ vec, long long ldb_vec, const float *__restrict__ gL,
                     float *__restrict__ gvec, long long B, int n) {
  const long long nn = (long long)n * n;
  if (ldb_vec != 0) {
    const long long total = B * n;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
      const long long b = e / n;
      const int i = (int)(e - b * n);
      gvec[e] = gL[b * nn + (long long)i * (n + 1)] / (1.f + expf(-vec[b * ldb_vec + i]));
    }
    return;
  }
  __shared__ float red[256];
  const int i = blockIdx.x;
  float acc = 0.f;
  for (long long b = threadIdx.x; b < B; b += blockDim.x) acc += gL[b * nn + (long long)i * (n + 1)];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int s = blockDim.x >> 1; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) gvec[i] = red[0] / (1.f + expf(-vec[i]));
}

}  // namespace

static int gauss_num_sms() {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
  }
  return sms;
}

extern "C" int tce_mvn_rsample(const float *mean, const float *L, int64_t ldb_L, const float *eps, uint64_t seed,
                               uint64_t offset, float *out, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!mean || !L || !out || B < 0 || n < 1 || n > 200) return TCE_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
  int64_t done = 0;
  // contiguous per-episode factors of odd order: bulk-copy kernel on whole groups of RS_G episodes, the rest below
  if ((n & 1) && n <= 64 && ldb_L == (int64_t)n * n && B >= 8 * RS_G && ((uintptr_t)L & 15) == 0) {
    const long long groups = B / RS_G;
    const size_t smem = (size_t)RS_G * n * n * sizeof(float) + RS_G * 64 * sizeof(float);
    const int sms = gauss_num_sms();
    if (smem > 48 * 1024)
      TCE_CUDA(cudaFuncSetAttribute(rsample_bulk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "rsample attr");
    const long long cap = 3LL * sms;
    rsample_bulk_kernel<<<(unsigned)(groups < cap ? groups : cap), RS_G * 64, smem, st>>>(mean, L, eps, seed, offset, out, n, groups);
    TCE_CHECK_LAUNCH("rsample_bulk_kernel");
    done = groups * RS_G;
    if (done == B) return TCE_OK;
  }
  // (the Philox counter is the element index: the tail draws the numbers the single launch would have drawn)
  rsample_kernel<<<(unsigned)(B - done), 128, n * sizeof(float), st>>>(mean, L, ldb_L, eps, seed, offset, out, n, done);
  TCE_CHECK_LAUNCH("rsample_kernel");
  return TCE_OK;
}

extern "C" int tce_chol_fwd(const float *A, float *L, int32_t *info, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!A || !L || B < 0 || n < 1 || n > 128) return TCE_ERR_INVALID_ARGUMENT;
  const size_t smem = (size_t)n * (n + 1) * sizeof(float);
  if (smem > 48 * 1024)
    TCE_CUDA(cudaFuncSetAttribute(chol_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "chol attr");
  chol_fwd_kernel<<<(unsigned)B, 128, smem, (cudaStream_t)stream>>>(A, L, info, n);
  TCE_CHECK_LAUNCH("chol_fwd_kernel");
  return TCE_OK;
}

extern "C" int tce_chol_bwd(const float *L, const float *grad_L, float *grad_A, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!L || !grad_L || !grad_A || B < 0 || n < 1 || n > 96) return TCE_ERR_INVALID_ARGUMENT;
  const size_t smem = 3 * (size_t)n * (n + 1) * sizeof(double);
  TCE_CUDA(cudaFuncSetAttribute(chol_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "cholb attr");
  chol_bwd_kernel<<<(unsigned)B, 128, smem, (cudaStream_t)stream>>>(L, grad_L, grad_A, n);
  TCE_CHECK_LAUNCH("chol_bwd_kernel");
  return TCE_OK;
}

extern "C" int tce_policy_head_fwd(const float *vec, int64_t ldb_vec, float min_std, float *L, int64_t B, int n,
                                   void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!vec || !L || B < 0 || n < 1) return TCE_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
  const int nvec = n + n * (n - 1) / 2;
  int64_t done = 0;
  const size_t smem = (size_t)HD_G * ((size_t)n * n + nvec) * sizeof(float);
  if (ldb_vec == nvec && B >= 8 * HD_G && n >= 8 && smem <= 110 * 1024 && (((uintptr_t)vec | (uintptr_t)L) & 15) == 0) {
    const long long groups = B / HD_G;
    if (smem > 48 * 1024)
      TCE_CUDA(cudaFuncSetAttribute(head_fwd_bulk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "head attr");
    const long long cap = 2LL * gauss_num_sms();
    head_fwd_bulk_kernel<<<(unsigned)(groups < cap ? groups : cap), 256, smem, st>>>(vec, min_std, L, n, groups);
    TCE_CHECK_LAUNCH("head_fwd_bulk_kernel");
    done = groups * HD_G;
    if (done == B) return TCE_OK;
  }
  head_fwd_kernel<<<(unsigned)(B - done), 256, 0, st>>>(vec + done * ldb_vec, ldb_vec, min_std, L + (size_t)done * n * n, n);
  TCE_CHECK_LAUNCH("head_fwd_kernel");
  return TCE_OK;
}

extern "C" int tce_policy_head_bwd(const float *vec, int64_t ldb_vec, const float *grad_L, float *grad_vec,
                                   int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!vec || !grad_L || !grad_vec || B < 0 || n < 1) return TCE_ERR_INVALID_ARGUMENT;
  const int nvec = n + n * (n - 1) / 2;
  cudaStream_t st = (cudaStream_t)stream;
  if (ldb_vec == 0) TCE_CUDA(cudaMemsetAsync(grad_vec, 0, nvec * sizeof(float), st), "head bwd memset");
  const int chunk = 32;
  dim3 grid((nvec + 127) / 128, (unsigned)((B + chunk - 1) / chunk));
  head_bwd_kernel<<<grid, 128, 0, st>>>(vec, ldb_vec, grad_L, grad_vec, B, n, chunk);
  TCE_CHECK_LAUNCH("head_bwd_kernel");
  return TCE_OK;
}

extern "C" int tce_policy_head_diag_fwd(const float *vec, int64_t ldb_vec, float min_std, float *L, int64_t B, int n,
                                        void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!vec || !L || B < 0 || n < 1 || ldb_vec < 0) return TCE_ERR_INVALID_ARGUMENT;
  const long long blocks = (B * n * n + 255) / 256, cap = 8LL * gauss_num_sms();
  head_diag_fwd_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, (cudaStream_t)stream>>>(vec, ldb_vec, min_std,
                                                                                                 L, B, n);
  TCE_CHECK_LAUNCH("head_diag_fwd_kernel");
  return TCE_OK;
}

extern "C" int tce_policy_head_diag_bwd(const float *vec, int64_t ldb_vec, const float *grad_L, float *grad_vec,
                                        int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!vec || !grad_L || !grad_vec || B < 0 || n < 1 || ldb_vec < 0) return TCE_ERR_INVALID_ARGUMENT;
  long long blocks = n;
  if (ldb_vec != 0) {
    const long long cap = 8LL * gauss_num_sms();
    blocks = (B * n + 255) / 256;
    blocks = blocks < cap ? blocks : cap;
  }
  head_diag_bwd_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(vec, ldb_vec, grad_L, grad_vec, B, n);
  TCE_CHECK_LAUNCH("head_diag_bwd_kernel");
  return TCE_OK;
}

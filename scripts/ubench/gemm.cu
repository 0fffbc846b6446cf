// Cycles of the shared-memory fp64 routines of csrc/tce_smem_la.cuh on ONE SM: la_gemm (fp64 tensor cores) against
// the scalar 4x4-register-tile GEMM it replaced, la_tri_inverse against the version whose first merge product
// started its k loop at the output's column, la_chol.  Every pair is checked BIT FOR BIT ("same" = number of
// differing elements is 0).  n = 63 / 36 / 28 (the projection sizes) and tails; 512 and 256 threads.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -I../../tce_rl_b200/csrc gemm.cu -o gemm
#include <cstdio>
#include "tce_smem_la.cuh"

// the scalar la_gemm: thread (I, J) owns rows 4I..4I+3 and the interleaved columns J, J+16, J+32, J+48; each output
// is one accumulator summed in ascending k with one rounded FMA per product
__device__ inline void la_gemm_scalar(Mat C, Mat A, Mat B, int m, int n, int k, int a_tri, int b_tri, double alpha,
                                      double beta) {
  const int TI = (m + 3) >> 2;
  for (int t = threadIdx.x; t < TI * 16; t += blockDim.x) {
    const int I = t >> 4, J = t & 15, i0 = 4 * I;
    int lo = 0, hi = k;
    if (a_tri == TRI_LOWER) hi = min(hi, i0 + 4);
    if (a_tri == TRI_UPPER) lo = max(lo, i0);
    if (b_tri == TRI_LOWER) lo = max(lo, J);
    const double *ap[4], *bp[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) ap[r] = &A(min(i0 + r, m - 1), 0);
#pragma unroll
    for (int c = 0; c < 4; ++c) bp[c] = &B(0, min(J + 16 * c, n - 1));
    double acc[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[r][c] = 0.0;
#pragma unroll 2
    for (int q = lo; q < hi; ++q) {
      double a[4], b[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) a[r] = ap[r][q * A.cs];
#pragma unroll
      for (int c = 0; c < 4; ++c) b[c] = bp[c][q * B.rs];
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] = fma(a[r], b[c], acc[r][c]);
    }
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int i = i0 + r, jj = J + 16 * c;
        if (i < m && jj < n) C(i, jj) = beta == 0.0 ? alpha * acc[r][c] : fma(beta, C(i, jj), alpha * acc[r][c]);
      }
  }
  __syncthreads();
}

// la_tri_inverse as it was: the first merge product starts at k = jj (each lane walks its own diagonal of X)
__device__ inline void la_tri_inverse_diag(Mat L, Mat X, double *dinv, int n) {
  la_diag_block_inverses(L, dinv, n);
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, j = e - i * n;
    X(i, j) = (i >> 3) == (j >> 3) ? dinv[((i >> 3) * LA_NB + (i & 7)) * LA_NB + (j & 7)] : 0.0;
  }
  __syncthreads();
  for (int lw = 3; (1 << lw) < n; ++lw) {
    const int w = 1 << lw, npair = (n + 2 * w - 1) >> (lw + 1), nout = npair << (2 * lw);
    double v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int o = threadIdx.x + u * (int)blockDim.x;
      v[u] = 0.0;
      if (o < nout) {
        const int pr = o >> (2 * lw), rem = o & ((1 << (2 * lw)) - 1), ii = rem >> lw, jj = rem & (w - 1);
        const int c0 = pr << (lw + 1), i = c0 + w + ii, j = c0 + jj;
        if (i < n) {
          double a0 = 0.0, a1 = 0.0;
          int k = jj;
          for (; k + 1 < w; k += 2) { a0 = fma(L(i, c0 + k), X(c0 + k, j), a0); a1 = fma(L(i, c0 + k + 1), X(c0 + k + 1, j), a1); }
          if (k < w) a0 = fma(L(i, c0 + k), X(c0 + k, j), a0);
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

// pure fp64 issue test: 16 independent accumulators per thread, operands in registers
__device__ inline double dfma_only(int iters, double x, double y) {
  double acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = x + i;
  for (int q = 0; q < iters; ++q) {
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = fma(acc[i], y, x);
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += acc[i];
  return s;
}

// number of elements of the n x n views that differ bit for bit (0: identical)
__device__ int count_diff(Mat X, Mat Y, int n, int *red) {
  if (threadIdx.x == 0) *red = 0;
  __syncthreads();
  int c = 0;
  for (int e = threadIdx.x; e < n * n; e += blockDim.x)
    c += __double_as_longlong(X(e / n, e % n)) != __double_as_longlong(Y(e / n, e % n));
  atomicAdd(red, c);
  __syncthreads();
  const int r = *red;
  __syncthreads();
  return r;
}

constexpr int NCASE = 7;
__global__ void __launch_bounds__(512) k(long long *cyc, int *diff, double *sink, int n) {
  extern __shared__ double sd[];
  const int m = (n + 1) & ~1, LD = m + 1, MS = m * LD;
  // b0 lower triangular (well conditioned), b1 full, b2 / b3 / b4 results; padding and b5 hold NaN so that a load
  // outside the operands' [0, n) ranges poisons the result
  Mat b0{sd, LD, 1}, b1{sd + MS, LD, 1}, b2{sd + 2 * MS, LD, 1}, b3{sd + 3 * MS, LD, 1}, b4{sd + 4 * MS, LD, 1};
  double *dinv = sd + 6 * MS;
  __shared__ int red;
  const double nan = __longlong_as_double(0x7ff8000000000001ll);
  for (int e = threadIdx.x; e < 6 * MS; e += blockDim.x) sd[e] = nan;
  __syncthreads();
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, j = e % n;
    b0(i, j) = j <= i ? (i == j ? 1.0 + 0.1 * sin(0.7 * i) : 0.3 * sin(1.3 * i + 2.1 * j + 0.5)) : 0.0;
    b1(i, j) = sin(0.37 * i * i + 1.7 * j + 0.2) / 3.0;
  }
  __syncthreads();
  long long t0, t1;
  int slot = 0;
#define TIME(body) __syncthreads(); t0 = clock64(); body; __syncthreads(); t1 = clock64(); if (threadIdx.x == 0) cyc[slot] = t1 - t0; ++slot;
#define CASE(AA, BB, kk, at, bt, al, be)                                              \
  TIME(la_gemm_scalar(b2, AA, BB, n, n, kk, at, bt, al, be))                           \
  TIME(la_gemm(b3, AA, BB, n, n, kk, at, bt, TRI_FULL, al, be))                        \
  { const int dd = count_diff(b2, b3, n, &red); if (threadIdx.x == 0) diff[slot / 2 - 1] = dd; }
  auto copy_into = [&](Mat X, Mat Y, int nn) {
    for (int e = threadIdx.x; e < nn * nn; e += blockDim.x) X(e / nn, e % nn) = Y(e / nn, e % nn);
    __syncthreads();
  };
  CASE(b0, b1, n, TRI_FULL, TRI_FULL, 1.0, 0.0)                       // 0 full
  CASE(b1.T(), b1, n, TRI_FULL, TRI_FULL, 1.0, 0.0)                   // 1 A transposed
  CASE(b1, b0.T(), n, TRI_FULL, TRI_UPPER, 1.0, 0.0)                  // 2 B transposed
  CASE(b0, b1, n, TRI_LOWER, TRI_FULL, 1.0, 0.0)                      // 3 A lower
  CASE(b0.T(), b0, n, TRI_UPPER, TRI_LOWER, 1.0, 0.0)                 // 4 A^T upper x lower
  CASE(b1, b1.T(), n, TRI_FULL, TRI_FULL, 1.0, 0.0)                   // 5 M M^T
  copy_into(b2, b1, n);
  copy_into(b3, b1, n);
  CASE(b1, b1.T(), min(n, 8), TRI_FULL, TRI_FULL, -1.0, 1.0)         // 6 C - M M^T, k = 8 (la_chol update)
  TIME(la_tri_inverse_diag(b0, b2, dinv, n))                                  // 14
  TIME(la_tri_inverse(b0, b3, dinv, n))                                       // 15
  { const int dd = count_diff(b2, b3, n, &red); if (threadIdx.x == 0) diff[NCASE] = dd; }
  TIME(la_diag_block_inverses(b0, dinv, n))                                   // 16
  double dd = 0.0;
  TIME(dd += dfma_only(63, b0(1, 1), b1(2, 2)))                               // 17: all warps x 63 x 16 DFMA
  if (dd == 123.0) sink[1] = dd;
  __shared__ int bad;
  if (threadIdx.x == 0) bad = 0;
  la_gemm(b4, b1, b1.T(), n, n, n, TRI_FULL, TRI_FULL, TRI_FULL, 1.0, 0.0);
  for (int e = threadIdx.x; e < n; e += blockDim.x) b4(e, e) += 1.0;
  __syncthreads();
  TIME(la_chol(b4, n, &bad))                                                  // 18
  if (threadIdx.x == 0) sink[0] = b2(3, 2) + b3(5, 1) + b4(n - 1, n - 1) + bad;
}

int main() {
  long long *cyc; int *diff; double *sink;
  cudaMalloc(&cyc, 8 * 64); cudaMalloc(&diff, 4 * 16); cudaMalloc(&sink, 64);
  const size_t smem = 200 * 1024;
  cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  const char *names[] = {"full", "A^T", "B^T (upper)", "A lower", "A^T upper x lower", "M M^T", "C - M M^T, k=8"};
  int fails = 0;
  for (int threads : {512, 256}) {
    for (int n : {63, 36, 28, 64, 33, 7, 2}) {
      for (int rep = 0; rep < 2; ++rep) k<<<1, threads, smem>>>(cyc, diff, sink, n);
      long long h[32]; int dh[16];
      cudaMemcpy(h, cyc, sizeof h, cudaMemcpyDeviceToHost);
      cudaMemcpy(dh, diff, sizeof dh, cudaMemcpyDeviceToHost);
      printf("n=%d threads=%d (%s)\n", n, threads, cudaGetErrorString(cudaGetLastError()));
      printf("  %-20s %8s %8s %s\n", "gemm", "scalar", "dmma", "bitwise");
      for (int c = 0; c < NCASE; ++c) {
        printf("  %-20s %8lld %8lld %s\n", names[c], h[2 * c], h[2 * c + 1], dh[c] ? "DIFFER" : "same");
        if (dh[c]) { printf("    %d elements differ\n", dh[c]); ++fails; }
      }
      printf("  tri_inverse          %8lld (k from the diagonal) %8lld (k from 0) %s\n", h[14], h[15], dh[NCASE] ? "DIFFER" : "same");
      fails += dh[NCASE] != 0;
      printf("  diag blocks only %lld, dfma %d warps x 1008 %lld, chol %lld\n", h[16], threads / 32, h[17], h[18]);
    }
  }
  printf("%s\n", fails ? "BITWISE MISMATCHES" : "all bitwise identical");
  return fails != 0;
}

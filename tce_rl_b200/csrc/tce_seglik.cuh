// Device code shared by the segment-likelihood kernels (tce_seglik.cu, tce_seglik_fused.cu): packed lower triangles,
// the ProDMP basis rows and the per-segment step (Cholesky, log-prob, adjoints).
#pragma once
#include <math.h>

#include "tce_common.cuh"

constexpr double LN_2PI = 1.8378770664093453;

__host__ __device__ constexpr int tri(int n) { return n * (n + 1) / 2; }
__device__ __forceinline__ int tri_idx(int r, int c) { return r * (r + 1) / 2 + c; }   // r >= c

// decode a lower-triangular index t -> (I, J), I >= J
__device__ __forceinline__ void tri_decode(int t, int &I, int &J) {
  int i = (int)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
  while (i * (i + 1) / 2 > t) --i;
  while ((i + 1) * (i + 2) / 2 <= t) ++i;
  I = i;
  J = t - i * (i + 1) / 2;
}

// ---- ProDMP basis rows with initial conditions (SURVEY App. A.3), fp64 ----------------------------------------------
// init_row [5 + 2 K1]: y1b, y2b, dy1b, dy2b, 1/det, pos_b[K1], vel_b[K1] at the episode's initial time; entry j <= K1
// (j == K1: the first five)
template <int K1>
__device__ __forceinline__ void init_row_entry(const TabDev &tb, double t_init, int j, double *init_row) {
  int i0; double w;
  time_to_index(tb, t_init, i0, w);
  if (j < K1) {
    init_row[5 + j] = lerp_t(tb.pos[(size_t)i0 * K1 + j], tb.pos[(size_t)(i0 + 1) * K1 + j], w);
    init_row[5 + K1 + j] = lerp_t(tb.vel[(size_t)i0 * K1 + j], tb.vel[(size_t)(i0 + 1) * K1 + j], w);
  } else {
    const double a = lerp_t(tb.y1[i0], tb.y1[i0 + 1], w), b = lerp_t(tb.y2[i0], tb.y2[i0 + 1], w);
    const double c = lerp_t(tb.dy1[i0], tb.dy1[i0 + 1], w), d = lerp_t(tb.dy2[i0], tb.dy2[i0 + 1], w);
    init_row[0] = a; init_row[1] = b; init_row[2] = c; init_row[3] = d;
    init_row[4] = 1.0 / (a * d - b * c);
  }
}
// entry j of the scaled basis row at time t (j < K1) or the pair (xi1, xi2) (j == K1)
template <int K1>
__device__ __forceinline__ void basis_entry(const TabDev &tb, const double *init_row, double t, int j, double *h_row,
                                            double *xi_row) {
  int i0; double w;
  time_to_index(tb, t, i0, w);
  const double y1 = lerp_t(tb.y1[i0], tb.y1[i0 + 1], w), y2 = lerp_t(tb.y2[i0], tb.y2[i0 + 1], w);
  const double idet = init_row[4];
  const double xi1 = (init_row[3] * y1 - init_row[2] * y2) * idet, xi2 = (init_row[0] * y2 - init_row[1] * y1) * idet;
  if (j < K1) {
    const double pj = lerp_t(tb.pos[(size_t)i0 * K1 + j], tb.pos[(size_t)(i0 + 1) * K1 + j], w);
    h_row[j] = (pj - xi1 * init_row[5 + j] - xi2 * init_row[5 + K1 + j]) * tb.scale[j];
  } else {
    xi_row[0] = xi1;
    xi_row[1] = xi2;
  }
}

// ---- per-segment step -------------------------------------------------------------------------------------------
// One thread factors the packed lower triangle c of one segment's n x n gram C (n = N = 2 D, entry (r, q) at
// tri_idx(r, q)) and transforms its residual z; fp64 throughout (cond(C) ~ 1e4: neighbouring time points are almost
// perfectly correlated).
//
// Storage: c, z and the adjoint's output G are register arrays (double[], indexed by compile-time constants, so every
// loop must be fully unrolled: FULL) or Strided views of memory (loops rolled: !FULL).
struct Strided {
  double *p;
  int stride;
  __device__ __forceinline__ double &operator[](int i) const { return p[(size_t)i * stride]; }
};

// for (int i = b; i < e; ++i) f(i), fully unrolled or not at all.  (An unroll count instead of the plain pragma would
// unroll the inner loops, whose trip counts depend on the outer index, at run time rather than completely.)
template <bool FULL, class F>
__device__ __forceinline__ void seg_for(int b, int e, F &&f) {
  if constexpr (FULL) {
#pragma unroll
    for (int i = b; i < e; ++i) f(i);
  } else {
#pragma unroll 1
    for (int i = b; i < e; ++i) f(i);
  }
}

// Cholesky C + reg I = S S^T in place, forward substitution z <- S^-1 z; returns the log-prob -1/2 (n ln 2pi + |z|^2)
// - log det S, bad = index + 1 of the first non-positive pivot (0: none).
// 1/sqrt of a pivot is an fp32 MUFU seed plus two fp64 Newton steps (1e-7 -> 1e-14 -> rounding), and the DIAGONAL
// STORES THE RECIPROCAL 1/S_jj: every later division (substitutions, inverse) becomes a multiplication -- fp64 divide
// and sqrt are ~40-instruction subroutines and there were ~130 of them per segment.
template <int N, bool FULL, class Tri, class Vec>
__device__ __forceinline__ double seg_factor(Tri &c, Vec &z, double reg, int &bad) {
  bad = 0;
  double half_logdet = 0.0, maha = 0.0;
  seg_for<FULL>(0, N, [&](int j) {
    double dj = c[tri_idx(j, j)] + reg;
    seg_for<FULL>(0, j, [&](int k) { dj = fma(-c[tri_idx(j, k)], c[tri_idx(j, k)], dj); });
    if (!(dj > 0.0) && bad == 0) bad = j + 1;
    double inv = (double)rsqrtf((float)dj);
    inv = inv * fma(-0.5 * dj, inv * inv, 1.5);
    inv = inv * fma(-0.5 * dj, inv * inv, 1.5);
    c[tri_idx(j, j)] = inv;
    half_logdet += 0.5 * log(dj);
    seg_for<FULL>(j + 1, N, [&](int i) {
      double v = c[tri_idx(i, j)];
      seg_for<FULL>(0, j, [&](int k) { v = fma(-c[tri_idx(i, k)], c[tri_idx(j, k)], v); });
      c[tri_idx(i, j)] = v * inv;
    });
    double zj = z[j];
    seg_for<FULL>(0, j, [&](int k) { zj = fma(-c[tri_idx(j, k)], z[k], zj); });
    zj *= inv;
    z[j] = zj;
    maha = fma(zj, zj, maha);
  });
  return -0.5 * ((double)N * LN_2PI + maha) - half_logdet;
}

// Per-segment outputs and upstream-gradient inputs, indexed by the segment gid = b P + p.
// grad_mode: 0 = log-probs only, 1 = upstream gradient grad_logp [B, P], 2 = fused surrogate
// loss = -grad_scale sum ratio * adv, ratio = exp(lp - logp_old).
struct SegIO {
  const float *grad_logp, *logp_old, *advantage;
  float *logp;
  int32_t *info;
  double grad_scale, reg;
  int grad_mode;
};

// Upstream gradient g = d loss / d lp (grad_mode 1 or 2); the surrogate adds its partials loss_part += g and
// ratio_part += ratio * grad_scale.
__device__ __forceinline__ double seg_upstream(const SegIO &io, double lp, long long gid, double &loss_part,
                                               double &ratio_part) {
  double g;
  if (io.grad_mode == 2) {
    const double ratio = exp(lp - (double)io.logp_old[gid]);
    g = -ratio * (double)io.advantage[gid] * io.grad_scale;
    loss_part += g;
    ratio_part += ratio * io.grad_scale;
  } else {
    g = (double)io.grad_logp[gid];
  }
  return g;
}

// After seg_factor: z <- alpha = C^-1 r = S^-T z, c <- X = S^-1, and G = g/2 (alpha alpha^T - C^-1) (lower) into G,
// which may be c itself.  The caller forms g alpha.
template <int N, bool FULL, class Tri, class Vec, class Out>
__device__ __forceinline__ void seg_adjoint(Tri &c, Vec &z, double g, Out &G) {
  seg_for<FULL>(0, N, [&](int r) {                         // alpha = S^-T z (back substitution, i = N - 1 .. 0)
    const int i = N - 1 - r;
    double v = z[i];
    seg_for<FULL>(i + 1, N, [&](int k) { v = fma(-c[tri_idx(k, i)], z[k], v); });
    z[i] = v * c[tri_idx(i, i)];
  });
  // S <- S^-1 (lower, in place; the diagonal already holds 1/S_jj = X_jj).  Column j: S[i][k], j <= k < i, are still
  // the Cholesky entries; X[k][j], k < i, are done.
  seg_for<FULL>(0, N, [&](int j) {
    seg_for<FULL>(j + 1, N, [&](int i) {
      double v = 0.0;
      seg_for<FULL>(j, i, [&](int k) { v = fma(c[tri_idx(i, k)], c[tri_idx(k, j)], v); });
      c[tri_idx(i, j)] = -v * c[tri_idx(i, i)];
    });
  });
  // C^-1 = X^T X row by row (entry (i, j) only reads rows k >= i, and within row i the diagonal X[i][i] is consumed
  // last, so G may overwrite X), then G
  const double hg = 0.5 * g;
  seg_for<FULL>(0, N, [&](int i) {
    const double ai = z[i];
    seg_for<FULL>(0, i + 1, [&](int j) {
      double v = 0.0;
      seg_for<FULL>(i, N, [&](int k) { v = fma(c[tri_idx(k, i)], c[tri_idx(k, j)], v); });
      G[tri_idx(i, j)] = hg * (ai * z[j] - v);
    });
  });
}

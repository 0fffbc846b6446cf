// Shared device/host helpers of libtce_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/tce_b200.h"

#define TCE_MAX_K1 16   // max parameters per DoF (num_basis + 1)
#define TCE_MAX_DOF 8
#define TCE_MAX_DP 64   // max parameters per episode (num_dof * K1) of the likelihood and the projections

// CALL with `K1` a compile-time constant for every K1 the tables accept (2..TCE_MAX_K1); returns
// TCE_ERR_UNSUPPORTED_SHAPE for anything else.
#define TCE_DISPATCH_K1(K1v, CALL)                   \
  switch (K1v) {                                     \
    case 2: { constexpr int K1 = 2; CALL; } break;   \
    case 3: { constexpr int K1 = 3; CALL; } break;   \
    case 4: { constexpr int K1 = 4; CALL; } break;   \
    case 5: { constexpr int K1 = 5; CALL; } break;   \
    case 6: { constexpr int K1 = 6; CALL; } break;   \
    case 7: { constexpr int K1 = 7; CALL; } break;   \
    case 8: { constexpr int K1 = 8; CALL; } break;   \
    case 9: { constexpr int K1 = 9; CALL; } break;   \
    case 10: { constexpr int K1 = 10; CALL; } break; \
    case 11: { constexpr int K1 = 11; CALL; } break; \
    case 12: { constexpr int K1 = 12; CALL; } break; \
    case 13: { constexpr int K1 = 13; CALL; } break; \
    case 14: { constexpr int K1 = 14; CALL; } break; \
    case 15: { constexpr int K1 = 15; CALL; } break; \
    case 16: { constexpr int K1 = 16; CALL; } break; \
    default: return TCE_ERR_UNSUPPORTED_SHAPE;       \
  }

// Opaque tables handle (device pointers + the scalars every kernel needs).
struct tce_tables {
  tce_mp_cfg cfg;
  int num_pc;       // N_pc grid points
  int K1;           // num_basis + 1
  int D;            // num_dof
  double scaled_dt; // dt / tau
  double inv_scaled_dt;
  // fp64 tables (device): y1,y2,dy1,dy2 [N_pc]; pos/vel basis [N_pc, K1]; scale [K1]
  double *y1, *y2, *dy1, *dy2, *pos, *vel, *scale;
  // fp32 interleaved copy for the HBM-bound trajectory kernel: row i = [y1,y2,dy1,dy2,pos[K1],vel[K1]]
  float *row32;
  int row32_stride; // 4 + 2*K1
  void *base;       // single allocation behind all of the above
  size_t base_bytes;
};

// POD copy of what device code needs (passed by value to kernels)
struct TabDev {
  const double *y1, *y2, *dy1, *dy2, *pos, *vel, *scale;
  const float *row32;
  int num_pc, K1, D, row32_stride;
  double inv_scaled_dt, tau, inv_tau, delay;
  int relative_goal, relative_goal_scaled;
};

static inline TabDev tab_dev(const tce_tables *t) {
  TabDev d;
  d.y1 = t->y1; d.y2 = t->y2; d.dy1 = t->dy1; d.dy2 = t->dy2; d.pos = t->pos; d.vel = t->vel;
  d.scale = t->scale; d.row32 = t->row32; d.num_pc = t->num_pc; d.K1 = t->K1; d.D = t->D;
  d.row32_stride = t->row32_stride; d.inv_scaled_dt = t->inv_scaled_dt; d.tau = t->cfg.tau; d.inv_tau = 1.0 / t->cfg.tau;
  d.delay = t->cfg.delay; d.relative_goal = t->cfg.relative_goal;
  d.relative_goal_scaled = t->cfg.relative_goal_scaled;
  return d;
}

void tce_set_cuda_error(cudaError_t e, const char *where);

#define TCE_CHECK_LAUNCH(where)                         \
  do {                                                  \
    cudaError_t e__ = cudaGetLastError();               \
    if (e__ != cudaSuccess) {                           \
      tce_set_cuda_error(e__, where);                   \
      return TCE_ERR_CUDA;                              \
    }                                                   \
  } while (0)

#define TCE_CUDA(call, where)                           \
  do {                                                  \
    cudaError_t e__ = (call);                           \
    if (e__ != cudaSuccess) {                           \
      tce_set_cuda_error(e__, where);                   \
      return TCE_ERR_CUDA;                              \
    }                                                   \
  } while (0)

// ---- device helpers -------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
template <typename T>
__device__ __forceinline__ T warp_max(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    T w = __shfl_xor_sync(0xffffffffu, v, o);
    v = w > v ? w : v;
  }
  return v;
}

// torch.lerp(a, b, w): a + w (b - a) for w < 0.5, b - (b - a)(1 - w) otherwise
template <typename T>
__device__ __forceinline__ T lerp_t(T a, T b, T w) {
  T d = b - a;
  return w < T(0.5) ? a + w * d : b - d * (T(1) - w);
}

// float index of a time point in the pre-computed grid + clamped integer base
// (ProDMPBasisGenerator.times_to_indices + indexing_interpolate, util_matrix.py:195-227)
__device__ __forceinline__ void time_to_index(const TabDev &tb, double t, int &i0, double &w) {
  double s = (t - tb.delay) * tb.inv_tau;        // multiply by 1/tau: no fp64 division on the device
  s = s > 0.0 ? s : 0.0;
  double idx = s * tb.inv_scaled_dt;
  int f = (int)idx;                              // idx >= 0: truncation == floor
  f = f > tb.num_pc - 2 ? tb.num_pc - 2 : f;
  i0 = f;
  w = idx - (double)f;
}

// positive doubles order like their bit patterns
__device__ __forceinline__ void atomic_max_pos_double(double *addr, double v) {
  atomicMax(reinterpret_cast<unsigned long long *>(addr), (unsigned long long)__double_as_longlong(v));
}

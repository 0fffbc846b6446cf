// (1) Batched ProDMP trajectory synthesis: params -> pos/vel over T steps.
// Replaces ProDMP.get_traj_pos / get_traj_vel behind TemporalCorrelatedPolicy.sample
// (mprl/rl/policy/temporal_correlated_policy.py:76-100); math: SURVEY App. A.5.
//
// HBM-bound (algorithmic bytes/episode = 4*[Dp + (1+2D) + T + 2D*T]).  General time grids run
// traj_fwd_warp_kernel; a time grid common to the whole batch runs traj_rows_kernel + traj_uniform_kernel.
#include "tce_common.cuh"

namespace {

// index of a time in the pre-computed grid without divisions (inv_tau = 1 / tau, fp64)
__device__ __forceinline__ void time_to_index_fast(const TabDev &tb, double inv_tau, float t, int &i0, float &w) {
  double s = ((double)t - tb.delay) * inv_tau;
  s = s > 0.0 ? s : 0.0;
  const double idx = s * tb.inv_scaled_dt;
  int f = (int)idx;                          // idx >= 0: truncation == floor
  f = f > tb.num_pc - 2 ? tb.num_pc - 2 : f;
  i0 = f;
  w = (float)(idx - (double)f);
}

// Warp-per-slab kernel (any time grid): a warp owns 32 consecutive time points of ONE episode, so everything
// per-episode (basis values at the initial time, parameters, initial conditions) is warp-uniform: the initial-condition
// row is built cooperatively (lane j -> basis column j) and broadcast by shuffles, the parameters are warp-uniform
// (broadcast) loads through L1, the table rows are read through L1 as well (44 KB of fp32 rows: resident).  No shared
// staging of parameters, no CTA barrier, no serial per-episode section; the warp's 32 x 2D results go through a private
// shared tile so that the global stores are contiguous 128-bit.  HBM traffic = the algorithmic bytes (params, initial
// conditions and times are read once, the trajectory is written once).
constexpr int TW_WARPS = 8;
template <int K1, int DMAX>
__global__ void __launch_bounds__(TW_WARPS * 32)
traj_fwd_warp_kernel(TabDev tb, const float *__restrict__ params, const float *__restrict__ times,
                     const float *__restrict__ init_time, const float *__restrict__ init_pos,
                     const float *__restrict__ init_vel, float *__restrict__ traj, long long B, int T) {
  extern __shared__ __align__(16) float tile_all[];
  const int D = tb.D, D2 = 2 * D, Dp = D * K1, stride = tb.row32_stride;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float *tile = tile_all + warp * (32 * D2 + 4);
  const int slabs = (T + 31) >> 5;
  const long long total = B * (long long)slabs;
  const float tau = (float)tb.tau, inv_tau_f = 1.0f / tau;
  const double inv_tau = 1.0 / tb.tau;
  float sc[K1];
#pragma unroll
  for (int j = 0; j < K1; ++j) sc[j] = (float)tb.scale[j];
  const float goal_shift_scale = tb.relative_goal ? (tb.relative_goal_scaled ? 1.0f : 1.0f / sc[K1 - 1]) : 0.0f;
  for (long long w = (long long)blockIdx.x * TW_WARPS + warp; w < total; w += (long long)gridDim.x * TW_WARPS) {
    const long long b = w / slabs;
    const int t0 = (int)(w - b * slabs) << 5, t = t0 + lane;
    const int nt = T - t0 < 32 ? T - t0 : 32;
    // ---- initial-condition row of the episode: lane j < K1 -> (pb_j, vb_j), lane K1 -> y1b, y2b, dy1b, dy2b ----
    int ib; float wb;
    time_to_index_fast(tb, inv_tau, init_time[b], ib, wb);
    const float *q0 = tb.row32 + (size_t)ib * stride, *q1 = q0 + stride;
    float mine0 = 0.f, mine1 = 0.f, y1b = 0.f, y2b = 0.f, dy1b = 0.f, dy2b = 0.f;
    if (lane < K1) {
      mine0 = lerp_t(q0[4 + lane], q1[4 + lane], wb);
      mine1 = lerp_t(q0[4 + K1 + lane], q1[4 + K1 + lane], wb);
    }
    if (lane < 4) y1b = lerp_t(q0[lane], q1[lane], wb);               // lane l < 4 holds the l-th of (y1, y2, dy1, dy2)
    y2b = __shfl_sync(0xffffffffu, y1b, 1); dy1b = __shfl_sync(0xffffffffu, y1b, 2); dy2b = __shfl_sync(0xffffffffu, y1b, 3);
    y1b = __shfl_sync(0xffffffffu, y1b, 0);
    const float inv_det = 1.0f / (y1b * dy2b - y2b * dy1b);
    // ---- this lane's time point ----
    float hp[K1], hv[K1], xi1 = 0.f, xi2 = 0.f, xi3 = 0.f, xi4 = 0.f;
    {
      int i0; float wf;
      time_to_index_fast(tb, inv_tau, lane < nt ? times[b * T + t] : times[b * T + t0], i0, wf);
      const float *r0 = tb.row32 + (size_t)i0 * stride, *r1 = r0 + stride;
      const float y1 = lerp_t(r0[0], r1[0], wf), y2 = lerp_t(r0[1], r1[1], wf);
      const float dy1 = lerp_t(r0[2], r1[2], wf), dy2 = lerp_t(r0[3], r1[3], wf);
      xi1 = (dy2b * y1 - dy1b * y2) * inv_det; xi2 = (y1b * y2 - y2b * y1) * inv_det;
      xi3 = (dy2b * dy1 - dy1b * dy2) * inv_det; xi4 = (y1b * dy2 - y2b * dy1) * inv_det;
#pragma unroll
      for (int j = 0; j < K1; ++j) {
        const float pbj = __shfl_sync(0xffffffffu, mine0, j), vbj = __shfl_sync(0xffffffffu, mine1, j);
        const float pj = lerp_t(r0[4 + j], r1[4 + j], wf), vj = lerp_t(r0[4 + K1 + j], r1[4 + K1 + j], wf);
        hp[j] = (pj - xi1 * pbj - xi2 * vbj) * sc[j];
        hv[j] = (vj - xi3 * pbj - xi4 * vbj) * sc[j];
      }
    }
    const float *th = params + b * Dp;
    float *o = tile + lane * D2;
    for (int d = 0; d < D; ++d) {
      const float y0 = init_pos[b * D + d], v0 = init_vel[b * D + d] * tau;      // warp-uniform loads
      float p = xi1 * y0 + xi2 * v0, v = xi3 * y0 + xi4 * v0;
#pragma unroll
      for (int j = 0; j < K1; ++j) {
        const float thj = th[d * K1 + j];
        p = fmaf(hp[j], thj, p);
        v = fmaf(hv[j], thj, v);
      }
      const float shift = goal_shift_scale * y0;         // relative goal (0 otherwise)
      p = fmaf(hp[K1 - 1], shift, p);
      v = fmaf(hv[K1 - 1], shift, v);
      o[d] = p;
      o[D + d] = v * inv_tau_f;
    }
    __syncwarp();
    const long long g0 = b * T + t0;
    const int n_out = nt * D2;
    float *dst = traj + g0 * D2;
    if ((n_out & 3) == 0 && ((g0 * D2) & 3) == 0) {
      const float4 *s4 = reinterpret_cast<const float4 *>(tile);
      float4 *d4 = reinterpret_cast<float4 *>(dst);
      for (int i = lane; i < n_out / 4; i += 32) d4[i] = s4[i];
    } else {
      for (int i = lane; i < n_out; i += 32) dst[i] = tile[i];
    }
    __syncwarp();
  }
}


// backward: one CTA per episode, thread (d, j) reduces over time.  Low priority path (the reference
// only ever samples under no_grad), kept simple.
template <int K1>
__global__ void traj_bwd_kernel(TabDev tb, const float *__restrict__ grad_traj, const float *__restrict__ times,
                                const float *__restrict__ init_time, float *__restrict__ grad_params,
                                float *__restrict__ grad_init_pos, float *__restrict__ grad_init_vel, int T) {
  const long long b = blockIdx.x;
  const int D = tb.D, D2 = 2 * D;
  const float tau = (float)tb.tau;
  __shared__ float s_pb[TCE_MAX_K1], s_vb[TCE_MAX_K1], s_init[5];
  if (threadIdx.x == 0) {
    int i0; double w;
    time_to_index(tb, (double)init_time[b], i0, w);
    const float wf = (float)w;
    const float *r0 = tb.row32 + (size_t)i0 * tb.row32_stride, *r1 = r0 + tb.row32_stride;
    for (int q = 0; q < 4; ++q) s_init[q] = lerp_t(r0[q], r1[q], wf);
    s_init[4] = 1.0f / (s_init[0] * s_init[3] - s_init[1] * s_init[2]);
    for (int j = 0; j < K1; ++j) {
      s_pb[j] = lerp_t(r0[4 + j], r1[4 + j], wf);
      s_vb[j] = lerp_t(r0[4 + K1 + j], r1[4 + K1 + j], wf);
    }
  }
  __syncthreads();
  // threads [0, D*K1): params; [D*K1, D*K1 + D): init_pos; [.., +D): init_vel
  const int tid = threadIdx.x, nP = D * K1;
  if (tid >= nP + 2 * D) return;
  const int kind = tid < nP ? 0 : (tid < nP + D ? 1 : 2);
  const int d = kind == 0 ? tid / K1 : (tid - nP) % D;
  const int j = kind == 0 ? tid % K1 : 0;
  const float y1b = s_init[0], y2b = s_init[1], dy1b = s_init[2], dy2b = s_init[3], idet = s_init[4];
  const float sc_j = (float)tb.scale[j], sc_g = (float)tb.scale[K1 - 1];
  float acc = 0.f;
  for (int t = 0; t < T; ++t) {
    int i0; double w;
    time_to_index(tb, (double)times[b * T + t], i0, w);
    const float wf = (float)w;
    const float *r0 = tb.row32 + (size_t)i0 * tb.row32_stride, *r1 = r0 + tb.row32_stride;
    const float y1 = lerp_t(r0[0], r1[0], wf), y2 = lerp_t(r0[1], r1[1], wf);
    const float dy1 = lerp_t(r0[2], r1[2], wf), dy2 = lerp_t(r0[3], r1[3], wf);
    const float xi1 = (dy2b * y1 - dy1b * y2) * idet, xi2 = (y1b * y2 - y2b * y1) * idet;
    const float xi3 = (dy2b * dy1 - dy1b * dy2) * idet, xi4 = (y1b * dy2 - y2b * dy1) * idet;
    const float gp = grad_traj[(b * T + t) * D2 + d], gv = grad_traj[(b * T + t) * D2 + D + d] / tau;
    if (kind == 0) {
      const float hp = (lerp_t(r0[4 + j], r1[4 + j], wf) - xi1 * s_pb[j] - xi2 * s_vb[j]) * sc_j;
      const float hv = (lerp_t(r0[4 + K1 + j], r1[4 + K1 + j], wf) - xi3 * s_pb[j] - xi4 * s_vb[j]) * sc_j;
      acc += hp * gp + hv * gv;
    } else if (kind == 1) {
      float a = xi1 * gp + xi3 * gv;
      if (tb.relative_goal) {
        const int g = K1 - 1;
        const float hp = (lerp_t(r0[4 + g], r1[4 + g], wf) - xi1 * s_pb[g] - xi2 * s_vb[g]) * sc_g;
        const float hv = (lerp_t(r0[4 + K1 + g], r1[4 + K1 + g], wf) - xi3 * s_pb[g] - xi4 * s_vb[g]) * sc_g;
        a += (hp * gp + hv * gv) * (tb.relative_goal_scaled ? 1.0f : 1.0f / sc_g);
      }
      acc += a;
    } else {
      acc += (xi2 * gp + xi4 * gv) * tau;
    }
  }
  if (kind == 0 && grad_params) grad_params[b * nP + tid] = acc;
  if (kind == 1 && grad_init_pos) grad_init_pos[b * D + d] = acc;
  if (kind == 2 && grad_init_vel) grad_init_vel[b * D + d] = acc;
}

int g_num_sms = 0;
int num_sms() {
  if (!g_num_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms <= 0) g_num_sms = 148;
  }
  return g_num_sms;
}


// Common time grid (every episode has the same init_time and times row -- all shipped TCE tasks start their
// trajectories at t = 0): the basis rows with initial conditions [xi1, xi2, hp[K1] | xi3, xi4, hv[K1]] are the same for
// all episodes.  traj_rows_kernel evaluates them once (T threads); traj_uniform_kernel is then a batched
// [T x (K1 + 2)] x [(K1 + 2) x D] product per episode: ~250 instructions per (episode, time) point instead of ~1200
// (table lerps, fp64 index arithmetic and the initial-condition algebra are gone from the per-point work), which moves
// the kernel from the issue limit towards the HBM roofline.
template <int K1>
__global__ void traj_rows_kernel(TabDev tb, const float *__restrict__ times_row, const float *__restrict__ init_time,
                                 float *__restrict__ rows, int T) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  constexpr int RW = (2 * (K1 + 2) + 3) & ~3;            // rows padded to 128-bit words (pad = 0)
  const int stride = tb.row32_stride;
  const double inv_tau = 1.0 / tb.tau;
  int ib; float wb;
  time_to_index_fast(tb, inv_tau, init_time[0], ib, wb);
  const float *q0 = tb.row32 + (size_t)ib * stride, *q1 = q0 + stride;
  const float y1b = lerp_t(q0[0], q1[0], wb), y2b = lerp_t(q0[1], q1[1], wb);
  const float dy1b = lerp_t(q0[2], q1[2], wb), dy2b = lerp_t(q0[3], q1[3], wb);
  const float inv_det = 1.0f / (y1b * dy2b - y2b * dy1b);
  int i0; float wf;
  time_to_index_fast(tb, inv_tau, times_row[t], i0, wf);
  const float *r0 = tb.row32 + (size_t)i0 * stride, *r1 = r0 + stride;
  const float y1 = lerp_t(r0[0], r1[0], wf), y2 = lerp_t(r0[1], r1[1], wf);
  const float dy1 = lerp_t(r0[2], r1[2], wf), dy2 = lerp_t(r0[3], r1[3], wf);
  const float xi1 = (dy2b * y1 - dy1b * y2) * inv_det, xi2 = (y1b * y2 - y2b * y1) * inv_det;
  const float xi3 = (dy2b * dy1 - dy1b * dy2) * inv_det, xi4 = (y1b * dy2 - y2b * dy1) * inv_det;
  // stored INTERLEAVED, (position coefficient k, velocity coefficient k) side by side: the consumer multiplies both by
  // the same parameter with one packed FMA
  float *o = rows + (size_t)t * RW;
#pragma unroll
  for (int k = 2 * (K1 + 2); k < RW; ++k) o[k] = 0.f;
  o[0] = xi1; o[1] = xi3; o[2] = xi2; o[3] = xi4;
#pragma unroll
  for (int j = 0; j < K1; ++j) {
    const float pbj = lerp_t(q0[4 + j], q1[4 + j], wb), vbj = lerp_t(q0[4 + K1 + j], q1[4 + K1 + j], wb);
    const float pj = lerp_t(r0[4 + j], r1[4 + j], wf), vj = lerp_t(r0[4 + K1 + j], r1[4 + K1 + j], wf);
    const float scj = (float)tb.scale[j];
    o[2 * (2 + j)] = (pj - xi1 * pbj - xi2 * vbj) * scj;
    o[2 * (2 + j) + 1] = (vj - xi3 * pbj - xi4 * vbj) * scj;
  }
}

// traj_uniform_kernel: thread (e, d) owns one degree of freedom of one episode of the CTA's group: its K1 + 2
// coefficients [y0, tau v0, theta (goal shifted)] stay in registers for the whole trajectory, the basis row of time t is
// read as six 128-bit BROADCAST loads (all lanes the same t), K1 + 2 packed FMAs (FFMA2: position and velocity
// coefficient of the row side by side, the parameter in both halves) give position and velocity.  Results go
// through a shared tile [episode][TU_TT time steps][2 D] so that every episode's TU_TT * 2D floats leave as contiguous
// 128-bit stores (56-byte rows written from registers touch every 32-byte sector several times: L2 write bound).
// ~7 warp instructions and ~2 shared-memory wavefronts per (episode, time) point; at B = 16384 every group has its
// own resident CTA.
constexpr int TU_THREADS = 256;
constexpr int TU_TT = 20;            // time steps per tile pass
template <int K1>
__global__ void __launch_bounds__(TU_THREADS)
traj_uniform_kernel(TabDev tb, const float *__restrict__ rows, const float *__restrict__ params,
                    const float *__restrict__ init_pos, const float *__restrict__ init_vel, float *__restrict__ traj,
                    long long B, int T, int epc, int estride) {
  constexpr int PW = K1 + 2, RWP = (2 * PW + 3) & ~3;
  extern __shared__ __align__(16) float su[];
  const int D = tb.D, D2 = 2 * D, Dp = D * K1;
  float *srow = su;                                   // [T][RWP]
  float *tile = su + (size_t)T * RWP;                 // [epc][estride], estride >= TU_TT * D2 (multiple of 4, = 8 mod 32)
  {                                                   // rows [T][RWP] (padded by traj_rows_kernel): straight 128-bit copy,
    const float4 *src = reinterpret_cast<const float4 *>(rows);          // four loads in flight per thread
    float4 *dst = reinterpret_cast<float4 *>(srow);
    const int n4 = T * (RWP / 4), nth = (int)blockDim.x;
    for (int i0 = threadIdx.x; i0 < n4; i0 += 4 * nth) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) if (i0 + u * nth < n4) v[u] = src[i0 + u * nth];
#pragma unroll
      for (int u = 0; u < 4; ++u) if (i0 + u * nth < n4) dst[i0 + u * nth] = v[u];
    }
  }
  const float tau = (float)tb.tau, inv_tau_f = 1.0f / tau;
  const float sc_g = (float)tb.scale[K1 - 1];
  const float goal_shift_scale = tb.relative_goal ? (tb.relative_goal_scaled ? 1.0f : 1.0f / sc_g) : 0.0f;
  const int e = threadIdx.x / D, d = threadIdx.x - e * D;
  const long long groups = (B + epc - 1) / epc;
  for (long long g = blockIdx.x; g < groups; g += gridDim.x) {
    const long long b0 = g * epc, bb = b0 + e;
    const int ne = (int)((B - b0) < epc ? (B - b0) : epc);
    const bool mine = e < ne;
    float p[PW];
#pragma unroll
    for (int k = 0; k < PW; ++k) p[k] = 0.f;
    if (mine) {
      const float y0 = init_pos[bb * D + d];
      p[0] = y0;
      p[1] = init_vel[bb * D + d] * tau;
#pragma unroll
      for (int j = 0; j < K1; ++j) p[2 + j] = params[bb * Dp + d * K1 + j];
      p[PW - 1] += goal_shift_scale * y0;                                        // relative goal (0 otherwise)
    }
    for (int t0 = 0; t0 < T; t0 += TU_TT) {
      const int nt = T - t0 < TU_TT ? T - t0 : TU_TT;
      __syncthreads();                                 // srow ready (first pass) / previous tile copied out
      if (mine) {
        float *o = tile + (size_t)e * estride + d;
        for (int tl = 0; tl < nt; ++tl) {
          const float4 *row = reinterpret_cast<const float4 *>(srow + (size_t)(t0 + tl) * RWP);
          float2 ac = make_float2(0.f, 0.f);           // (position, velocity * tau): one packed FP32 FMA (FFMA2, sm_100)
#pragma unroll                                         // per coefficient instead of two scalar ones
          for (int q = 0; q < RWP / 4; ++q) {
            const float4 v = row[q];
            if (2 * q < PW) ac = __ffma2_rn(make_float2(v.x, v.y), make_float2(p[2 * q], p[2 * q]), ac);
            if (2 * q + 1 < PW) ac = __ffma2_rn(make_float2(v.z, v.w), make_float2(p[2 * q + 1], p[2 * q + 1]), ac);
          }
          o[tl * D2] = ac.x;
          o[tl * D2 + D] = ac.y * inv_tau_f;
        }
      }
      __syncthreads();
      const int per = nt * D2;                         // contiguous floats per episode in this pass
      const long long g0 = (b0 * T + t0) * (long long)D2;
      if ((per & 3) == 0 && (g0 & 3) == 0 && (((long long)T * D2) & 3) == 0) {
        const int per4 = per >> 2;
        for (int i = threadIdx.x; i < ne * per4; i += blockDim.x) {
          const int ee = i / per4, q = i - ee * per4;
          reinterpret_cast<float4 *>(traj + g0 + (long long)ee * T * D2)[q] =
              reinterpret_cast<const float4 *>(tile + (size_t)ee * estride)[q];
        }
      } else {
        for (int i = threadIdx.x; i < ne * per; i += blockDim.x) {
          const int ee = i / per, q = i - ee * per;
          traj[g0 + (long long)ee * T * D2 + q] = tile[(size_t)ee * estride + q];
        }
      }
    }
  }
}

template <int K1>
int launch_traj_uniform(const tce_tables *t, const float *params, const float *times_row, const float *init_time,
                        const float *init_pos, const float *init_vel, float *rows_ws, float *traj, int64_t B, int64_t T,
                        cudaStream_t st) {
  constexpr int RW = 2 * (K1 + 2), RWP = (RW + 3) & ~3;
  traj_rows_kernel<K1><<<(unsigned)((T + 127) / 128), 128, 0, st>>>(tab_dev(t), times_row, init_time, rows_ws, (int)T);
  TCE_CHECK_LAUNCH("traj_rows_kernel");
  const int D = t->D, D2 = 2 * D;
  if (D > TU_THREADS / 4) return TCE_ERR_UNSUPPORTED_SHAPE;
  // episodes per CTA: up to 16 (<= 256 threads), fewer for small batches so that every SM gets a group
  int epc = TU_THREADS / D;
  if (epc > 16) epc = 16;
  while (epc > 4 && (B + epc - 1) / epc < 2LL * num_sms()) epc >>= 1;
  int estride = (TU_TT * D2 + 3) & ~3;                 // multiple of 4 and = 8 (mod 32): conflict-light tile rows
  while ((estride & 31) != 8) estride += 4;
  const size_t smem = sizeof(float) * ((size_t)T * RWP + (size_t)epc * estride);   // ops.traj_uniform_layout mirrors
  if (smem > 200 * 1024) return TCE_ERR_UNSUPPORTED_SHAPE;                           // epc and smem: keep them in step
  if (smem > 48 * 1024)
    TCE_CUDA(cudaFuncSetAttribute(traj_uniform_kernel<K1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
             "traj uniform smem attr");
  int threads = ((epc * D + 31) / 32) * 32;            // >= 128: the extra threads help with the row copy and the stores
  if (threads < 128) threads = 128;
  long long grid = (B + epc - 1) / epc;
  const long long cap = 8LL * num_sms();
  if (grid > cap) grid = cap;
  traj_uniform_kernel<K1><<<(unsigned)grid, threads, smem, st>>>(tab_dev(t), rows_ws, params, init_pos, init_vel, traj, B,
                                                               (int)T, epc, estride);
  TCE_CHECK_LAUNCH("traj_uniform_kernel");
  return TCE_OK;
}

template <int K1>
int launch_traj_fwd(const tce_tables *t, const float *params, const float *times, const float *init_time,
                    const float *init_pos, const float *init_vel, float *traj, int64_t B, int64_t T,
                    cudaStream_t st) {
  const long long slabs = B * ((T + 31) / 32);
  long long grid = (slabs + TW_WARPS - 1) / TW_WARPS;
  const long long cap = 8LL * num_sms();
  if (grid > cap) grid = cap;
  const size_t smem_w = (size_t)TW_WARPS * (32 * 2 * t->D + 4) * sizeof(float);
  traj_fwd_warp_kernel<K1, TCE_MAX_DOF><<<(unsigned)grid, TW_WARPS * 32, smem_w, st>>>(
      tab_dev(t), params, times, init_time, init_pos, init_vel, traj, B, (int)T);
  TCE_CHECK_LAUNCH("traj_fwd_warp_kernel");
  return TCE_OK;
}

}  // namespace

extern "C" int tce_prodmp_traj_fwd(const tce_tables_t *t, const float *params, const float *times,
                                   const float *init_time, const float *init_pos, const float *init_vel,
                                   float *traj, int64_t B, int64_t T, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!t || !params || !times || !init_time || !init_pos || !init_vel || !traj || B < 0 || T < 1)
    return TCE_ERR_INVALID_ARGUMENT;
  TCE_DISPATCH_K1(t->K1, return launch_traj_fwd<K1>(t, params, times, init_time, init_pos, init_vel, traj, B, T,
                                                    (cudaStream_t)stream));
  return TCE_OK;
}

/* All episodes share ONE time grid: times_row [T] and init_time [1] describe it (episode 0's values); rows_ws
 * [T * (2 * (K1 + 2) rounded up to a multiple of 4)] floats of workspace, 16-byte aligned.  Same results as tce_prodmp_traj_fwd on such inputs.               */
extern "C" int tce_prodmp_traj_fwd_uniform(const tce_tables_t *t, const float *params, const float *times_row,
                                           const float *init_time, const float *init_pos, const float *init_vel,
                                           float *rows_ws, float *traj, int64_t B, int64_t T, void *stream) {
  if (B == 0) return TCE_OK;
  if (!t || !params || !times_row || !init_time || !init_pos || !init_vel || !rows_ws || !traj || B < 0 || T < 1)
    return TCE_ERR_INVALID_ARGUMENT;
  TCE_DISPATCH_K1(t->K1, return launch_traj_uniform<K1>(t, params, times_row, init_time, init_pos, init_vel, rows_ws, traj,
                                                        B, T, (cudaStream_t)stream));
  return TCE_OK;
}

extern "C" int tce_prodmp_traj_bwd(const tce_tables_t *t, const float *grad_traj, const float *times,
                                   const float *init_time, float *grad_params, float *grad_init_pos,
                                   float *grad_init_vel, int64_t B, int64_t T, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!t || !grad_traj || !times || !init_time || B < 0 || T < 1) return TCE_ERR_INVALID_ARGUMENT;
  const int threads = ((t->D * t->K1 + 2 * t->D + 31) / 32) * 32;
  TCE_DISPATCH_K1(t->K1, (traj_bwd_kernel<K1><<<(unsigned)B, threads, 0, (cudaStream_t)stream>>>(
                             tab_dev(t), grad_traj, times, init_time, grad_params, grad_init_pos, grad_init_vel,
                             (int)T)));
  TCE_CHECK_LAUNCH("traj_bwd_kernel");
  return TCE_OK;
}

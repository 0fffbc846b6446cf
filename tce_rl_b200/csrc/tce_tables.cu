// ProDMP pre-computed tables, built on the device in fp64.
// Replaces mp_pytorch ProDMPBasisGenerator.pre_compute (constructed by mprl/util/util_mp.py:11-46);
// algorithm: SURVEY App. A.1-A.4 (ProDMP paper, README.md:221-233).
#include <math.h>
#include <string.h>

#include "tce_common.cuh"

static thread_local char g_cuda_err[256] = "";

void tce_set_cuda_error(cudaError_t e, const char *where) {
  snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", where, cudaGetErrorString(e));
}

extern "C" int tce_version(void) { return 100; }

extern "C" const char *tce_last_cuda_error(void) { return g_cuda_err; }

extern "C" const char *tce_strerror(int status) {
  switch (status) {
    case TCE_OK: return "ok";
    case TCE_ERR_INVALID_ARGUMENT: return "invalid argument";
    case TCE_ERR_UNSUPPORTED_SHAPE: return "unsupported (num_dof, num_basis) combination";
    case TCE_ERR_CUDA: return "CUDA runtime error";
    case TCE_ERR_WORKSPACE: return "workspace too small";
    default: return "unknown status";
  }
}

// One block; thread k < K1 owns basis column k (k == K is the goal column).
__global__ void build_tables_kernel(tce_mp_cfg cfg, int n_pc, int K, double *y1, double *y2, double *dy1,
                                    double *dy2, double *pos, double *vel, double *scale, float *row32) {
  __shared__ double c_p[TCE_MAX_K1], bw[TCE_MAX_K1];
  const int K1 = K + 1;
  const int k = threadIdx.x;
  const double a2 = 0.5 * cfg.alpha;
  const double ds = (double)cfg.pre_compute_length_factor / (double)(n_pc - 1);
  if (k < K) {
    if (K > 1) {
      double dist = cfg.tau / (double)(K - 2 * cfg.num_basis_outside - 1);
      double lo = -cfg.num_basis_outside * dist + cfg.delay;
      double hi = cfg.tau + cfg.num_basis_outside * dist + cfg.delay;
      double ct = lo + (hi - lo) * (double)k / (double)(K - 1);
      c_p[k] = exp(-cfg.alpha_phase * (ct - cfg.delay) / cfg.tau);
    } else {
      c_p[k] = 0.0;
    }
  }
  __syncthreads();
  if (k < K) {
    if (K > 1) {
      double dc = (k < K - 1) ? c_p[k + 1] - c_p[k] : c_p[K - 1] - c_p[K - 2];
      bw[k] = cfg.basis_bandwidth_factor / (dc * dc);
    } else {
      bw[k] = 3.0;
    }
  }
  __syncthreads();
  if (k < K1) {
    double p1 = 0.0, p2 = 0.0, prev1 = 0.0, prev2 = 0.0, mx = -INFINITY;
    for (int i = 0; i < n_pc; ++i) {
      // torch.linspace: start + i*step for the first half, end - (n-1-i)*step for the second
      double s = (i < n_pc / 2) ? ds * i : (double)cfg.pre_compute_length_factor - ds * (n_pc - 1 - i);
      double v1 = exp(-a2 * s), v2 = s * v1;
      double d1 = -a2 * v1, d2 = -a2 * v2 + v1;
      double e = exp(a2 * s);
      double pb, vb;
      if (k < K) {
        double x = exp(-cfg.alpha_phase * s);
        double sum = 0.0, mine = 0.0;
        for (int j = 0; j < K; ++j) {
          double d = x - c_p[j];
          double ph = exp(-0.5 * bw[j] * d * d);
          sum += ph;
          if (j == k) mine = ph;
        }
        double phi = (K > 1) ? mine / sum : mine;
        double f1 = s * e * x * phi, f2 = e * x * phi;
        if (i > 0) {  // cumulative trapezoid
          p1 += 0.5 * (f1 + prev1) * ds;
          p2 += 0.5 * (f2 + prev2) * ds;
        }
        prev1 = f1; prev2 = f2;
        pb = p2 * v2 - p1 * v1;
        vb = p2 * d2 - p1 * d1;
      } else {
        double q1 = (a2 * s - 1.0) * e + 1.0, q2 = a2 * (e - 1.0);
        pb = q2 * v2 - q1 * v1;
        vb = q2 * d2 - q1 * d1;
        y1[i] = v1; y2[i] = v2; dy1[i] = d1; dy2[i] = d2;
      }
      pos[(size_t)i * K1 + k] = pb;
      vel[(size_t)i * K1 + k] = vb;
      mx = pb > mx ? pb : mx;
    }
    double sc = cfg.auto_scale_basis ? 1.0 / mx : 1.0;
    sc *= (k < K) ? cfg.weights_scale : cfg.goal_scale;
    scale[k] = sc;
  }
  __syncthreads();
  // fp32 interleaved rows for the trajectory kernel
  const int stride = 4 + 2 * K1;
  for (int i = threadIdx.x; i < n_pc; i += blockDim.x) {
    float *r = row32 + (size_t)i * stride;
    r[0] = (float)y1[i]; r[1] = (float)y2[i]; r[2] = (float)dy1[i]; r[3] = (float)dy2[i];
    for (int j = 0; j < K1; ++j) {
      r[4 + j] = (float)pos[(size_t)i * K1 + j];
      r[4 + K1 + j] = (float)vel[(size_t)i * K1 + j];
    }
  }
}

extern "C" int tce_prodmp_tables_create(const tce_mp_cfg *cfg, void *stream, tce_tables_t **out) {
  if (!cfg || !out) return TCE_ERR_INVALID_ARGUMENT;
  const int K = cfg->num_basis, K1 = K + 1;
  if (K < 1 || K1 > TCE_MAX_K1 || cfg->num_dof < 1 || cfg->num_dof > TCE_MAX_DOF || cfg->num_dof * K1 > TCE_MAX_TABLE_DP)
    return TCE_ERR_UNSUPPORTED_SHAPE;
  if (cfg->tau <= 0 || cfg->dt <= 0 || cfg->pre_compute_length_factor < 1) return TCE_ERR_INVALID_ARGUMENT;
  if (K > 1 && K - 2 * cfg->num_basis_outside - 1 <= 0) return TCE_ERR_INVALID_ARGUMENT;
  tce_tables *t = new tce_tables();
  t->cfg = *cfg;
  t->K1 = K1;
  t->D = cfg->num_dof;
  t->scaled_dt = cfg->dt / cfg->tau;
  t->inv_scaled_dt = 1.0 / t->scaled_dt;
  t->num_pc = cfg->pre_compute_length_factor * (int)nearbyint(1.0 / t->scaled_dt) + 1;
  const size_t n = (size_t)t->num_pc;
  t->row32_stride = 4 + 2 * K1;
  const size_t n_d = 4 * n + 2 * n * K1 + K1;
  t->base_bytes = n_d * sizeof(double) + n * t->row32_stride * sizeof(float);
  cudaError_t e = cudaMalloc(&t->base, t->base_bytes);
  if (e != cudaSuccess) { tce_set_cuda_error(e, "tables cudaMalloc"); delete t; return TCE_ERR_CUDA; }
  double *p = (double *)t->base;
  t->y1 = p; p += n; t->y2 = p; p += n; t->dy1 = p; p += n; t->dy2 = p; p += n;
  t->pos = p; p += n * K1; t->vel = p; p += n * K1; t->scale = p; p += K1;
  t->row32 = (float *)p;
  build_tables_kernel<<<1, 64, 0, (cudaStream_t)stream>>>(*cfg, t->num_pc, K, t->y1, t->y2, t->dy1, t->dy2,
                                                           t->pos, t->vel, t->scale, t->row32);
  e = cudaGetLastError();
  if (e != cudaSuccess) { tce_set_cuda_error(e, "build_tables_kernel"); cudaFree(t->base); delete t; return TCE_ERR_CUDA; }
  *out = t;
  return TCE_OK;
}

extern "C" void tce_prodmp_tables_destroy(tce_tables_t *t) {
  if (!t) return;
  cudaFree(t->base);
  delete t;
}

extern "C" int tce_prodmp_tables_num_pc(const tce_tables_t *t) { return t ? t->num_pc : TCE_ERR_INVALID_ARGUMENT; }

extern "C" int tce_prodmp_tables_export(const tce_tables_t *t, double *y1, double *y2, double *dy1, double *dy2,
                                        double *pos_basis, double *vel_basis, double *scale) {
  if (!t) return TCE_ERR_INVALID_ARGUMENT;
  TCE_CUDA(cudaDeviceSynchronize(), "tables export sync");
  const size_t n = (size_t)t->num_pc, K1 = (size_t)t->K1;
  struct { double *dst; const double *src; size_t cnt; } c[] = {
      {y1, t->y1, n}, {y2, t->y2, n}, {dy1, t->dy1, n}, {dy2, t->dy2, n},
      {pos_basis, t->pos, n * K1}, {vel_basis, t->vel, n * K1}, {scale, t->scale, K1}};
  for (auto &x : c)
    if (x.dst) TCE_CUDA(cudaMemcpy(x.dst, x.src, x.cnt * sizeof(double), cudaMemcpyDeviceToHost), "tables export");
  return TCE_OK;
}

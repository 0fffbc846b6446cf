// Gaussian scalars, Frobenius / W2 covariance projections and covariance distances for DIAGONAL factors (std_only
// policies).  Each kernel is the dense kernel of tce_proj.cu (gauss_kl_kernel, proj_frob_cov_*, proj_w2_cov_kernel,
// cov_distance_kernel) with L = diag(s), L_o = diag(s_o) substituted: every n x n product is elementwise, so one warp
// per episode and no shared memory, at any n <= 1024.  Standard deviations are strided vectors as for
// tce_proj_kl_diag_*: element i of episode b is s[b * ldb + i * inc] (dense factor, packed [B, n] or one shared vector).
#include "tce_common.cuh"

namespace {

constexpr int DG_WARPS = 4;
constexpr int DG_MAX_N = 1024;
constexpr double DG_LOG_2PI = 1.8378770664093453;

// Stats (s != NULL): out[b] = {maha, tr(Sigma_o^-1 Sigma), logdet Sigma, logdet Sigma_o, entropy}; Mahalanobis only
// (s == NULL): out[b] = maha.  mean == mean_o == NULL: zero mean difference.  Backward (gout != NULL, [B, 5] or [B]):
// grad_mean = 2 g_maha (mean - mean_o) / s_o^2, grad_s = 2 g_tr s / s_o^2 + (2 g_logdet + g_entropy) / s.
__global__ void __launch_bounds__(DG_WARPS * 32)
gauss_stats_diag_kernel(const float *__restrict__ mean, const float *__restrict__ mean_o, const float *__restrict__ s,
                        long long ldb_s, long long inc_s, const float *__restrict__ so, long long ldb_so,
                        long long inc_so, const double *__restrict__ gout, double *__restrict__ out,
                        float *__restrict__ grad_mean, float *__restrict__ grad_s, long long ldb_gs, long long inc_gs,
                        long long B, int n) {
  const int lane = threadIdx.x & 31;
  const long long b = (long long)blockIdx.x * DG_WARPS + (threadIdx.x >> 5);
  if (b >= B) return;                                   // warp-uniform
  const bool stats = s != nullptr;
  const float *sb = stats ? s + b * ldb_s : nullptr, *sob = so + b * ldb_so;
  const float *mb = mean ? mean + b * n : nullptr, *mob = mean ? mean_o + b * n : nullptr;
  if (!gout) {
    double maha = 0.0, tr = 0.0, ld = 0.0, ldo = 0.0;
    for (int i = lane; i < n; i += 32) {
      const double vo = sob[i * inc_so], ivo = 1.0 / vo;
      if (mb) {
        const double z = ((double)mb[i] - (double)mob[i]) * ivo;
        maha = fma(z, z, maha);
      }
      if (stats) {
        const double v = sb[i * inc_s], r = v * ivo;
        tr = fma(r, r, tr);
        ld += log(v);
        ldo += log(vo);
      }
    }
    maha = warp_sum(maha);
    if (!stats) {
      if (lane == 0) out[b] = maha;
      return;
    }
    tr = warp_sum(tr);
    ld = warp_sum(ld);
    ldo = warp_sum(ldo);
    if (lane == 0) {
      double *o = out + b * 5;
      o[0] = maha; o[1] = tr; o[2] = 2.0 * ld; o[3] = 2.0 * ldo; o[4] = 0.5 * n * (1.0 + DG_LOG_2PI) + ld;
    }
    return;
  }
  const double *g = gout + b * (stats ? 5 : 1);
  const double g_maha = g[0];
  const double g_tr = stats ? g[1] : 0.0, g_ld = stats ? g[2] : 0.0, g_ent = stats ? g[4] : 0.0;
  for (int i = lane; i < n; i += 32) {
    const double ivo = 1.0 / (double)sob[i * inc_so];
    if (grad_mean) grad_mean[b * n + i] = mb ? (float)(2.0 * g_maha * ((double)mb[i] - (double)mob[i]) * ivo * ivo) : 0.f;
    if (grad_s) {
      const double v = sb[i * inc_s];
      grad_s[b * ldb_gs + i * inc_gs] = (float)(2.0 * g_tr * v * ivo * ivo + (2.0 * g_ld + g_ent) / v);
    }
  }
}

// One element of the covariance distance of the Frobenius (kind 0) / W2 (kind 1) layers and its derivative w.r.t. s:
//   kind 0: (s_o^2 - s^2)^2;  kind 1: scale_prec ? (s / s_o - 1)^2 : (s_o - s)^2.
__device__ inline double cov_term(int kind, int scale_prec, double v, double vo, double *dterm) {
  if (kind == 0) {
    const double d = vo * vo - v * v;
    *dterm = -4.0 * d * v;
    return d * d;
  }
  if (scale_prec) {
    const double ivo = 1.0 / vo, r = v * ivo - 1.0;
    *dterm = 2.0 * r * ivo;
    return r * r;
  }
  const double d = vo - v;
  *dterm = -2.0 * d;
  return d * d;
}

// MODE 0: distance val[b] = cp, or grad_s = gval[b] d cp / d s.
// MODE 1: projection forward.  cp > eps_cov: eta = sqrt(cp / eps_cov) - 1, a = 1 / (1 + eta);
//   kind 0 (Frobenius, on the variances): out = sqrt((s^2 + eta s_o^2) a);  kind 1 (W2, on the factors): out = (s + eta s_o) a;
//   save_sc[b] = {eta, active, cp, 0}, info[b] = 1 if a projected variance is not positive.
// MODE 2: projection backward from gout = d loss / d out and save_sc: with y the projected variable (s^2 / s),
//   d y / d y_in = a, d y / d eta = a (y_o - y), d eta / d cp = 1 / (2 sqrt(cp eps_cov)).
template <int MODE>
__global__ void __launch_bounds__(DG_WARPS * 32)
cov_diag_kernel(int kind, int scale_prec, const float *__restrict__ s, long long ldb_s, long long inc_s,
                const float *__restrict__ so, long long ldb_so, long long inc_so, double eps_cov,
                const double *__restrict__ gval, double *__restrict__ val, const float *__restrict__ gout,
                long long ldb_g, long long inc_g, float *__restrict__ out, long long ldb_o, long long inc_o,
                double *__restrict__ save_sc, int32_t *__restrict__ info, long long B, int n) {
  const int lane = threadIdx.x & 31;
  const long long b = (long long)blockIdx.x * DG_WARPS + (threadIdx.x >> 5);
  if (b >= B) return;                                   // warp-uniform
  const float *sb = s + b * ldb_s, *sob = so + b * ldb_so;
  float *ob = out ? out + b * ldb_o : nullptr;
  if (MODE == 2) {
    const double *sc = save_sc + b * 4;
    const float *gb = gout + b * ldb_g;
    if (sc[1] == 0.0) {
      for (int i = lane; i < n; i += 32) ob[i * inc_o] = gb[i * inc_g];
      return;
    }
    const double eta = sc[0], cp = sc[2], a = 1.0 / (1.0 + eta + 1e-16);
    double dot = 0.0;
    for (int i = lane; i < n; i += 32) {
      const double v = sb[i * inc_s], vo = sob[i * inc_so], g = gb[i * inc_g];
      if (kind == 0) {                                  // d out / d y = 1 / (2 out)
        const double y = (v * v + eta * vo * vo) * a;
        dot = fma(0.5 * g / sqrt(y), a * a * (vo * vo - v * v), dot);
      } else {
        dot = fma(g, a * (vo - (v + eta * vo) * a), dot);
      }
    }
    const double coef = warp_sum(dot) / (2.0 * sqrt(cp * eps_cov));
    for (int i = lane; i < n; i += 32) {
      const double v = sb[i * inc_s], vo = sob[i * inc_so], g = gb[i * inc_g];
      double dterm;
      cov_term(kind, scale_prec, v, vo, &dterm);
      const double gy = kind == 0 ? v * a * g / sqrt((v * v + eta * vo * vo) * a) : a * g;
      ob[i * inc_o] = (float)(gy + coef * dterm);
    }
    return;
  }
  double cp = 0.0;
  for (int i = lane; i < n; i += 32) {
    double dterm;
    cp += cov_term(kind, scale_prec, sb[i * inc_s], sob[i * inc_so], &dterm);
  }
  cp = warp_sum(cp);
  if (MODE == 0) {
    if (gval) {
      const double g = gval[b];
      for (int i = lane; i < n; i += 32) {
        double dterm;
        cov_term(kind, scale_prec, sb[i * inc_s], sob[i * inc_so], &dterm);
        ob[i * inc_o] = (float)(g * dterm);
      }
    }
    if (val && lane == 0) val[b] = cp;
    return;
  }
  const bool active = cp > eps_cov;
  const double eta = active ? fabs(sqrt(cp / eps_cov) - 1.0) : 0.0, a = 1.0 / (1.0 + eta + 1e-16);
  int bad = 0;
  for (int i = lane; i < n; i += 32) {
    const double v = sb[i * inc_s], vo = sob[i * inc_so];
    double y = v;
    if (active && kind == 0) {
      const double var = (v * v + eta * vo * vo) * a;
      if (!(var > 0.0)) bad = 1;
      y = sqrt(var);
    } else if (active) {
      y = (v + eta * vo) * a;
    }
    ob[i * inc_o] = (float)y;
  }
  bad = __any_sync(0xffffffffu, bad);
  if (lane == 0) {
    double *sc = save_sc + b * 4;
    sc[0] = eta; sc[1] = active ? 1.0 : 0.0; sc[2] = cp; sc[3] = 0.0;
    if (info) info[b] = bad;
  }
}

unsigned dg_grid(int64_t B) { return (unsigned)((B + DG_WARPS - 1) / DG_WARPS); }

bool dg_bad_common(const float *s, int64_t ldb_s, const float *so, int64_t ldb_so, int64_t B, int n) {
  return !s || !so || B < 0 || n < 1 || n > DG_MAX_N || ldb_s < 0 || ldb_so < 0;
}

// an output written per episode must not be shared by the batch
bool dg_bad_out(const void *p, int64_t ldb, int64_t B) { return !p || ldb < 0 || (ldb == 0 && B > 1); }

template <int MODE>
int cov_diag_launch(int kind, int scale_prec, const float *s, int64_t ldb_s, int64_t inc_s, const float *so,
                    int64_t ldb_so, int64_t inc_so, double eps_cov, const double *gval, double *val,
                    const float *gout, int64_t ldb_g, int64_t inc_g, float *out, int64_t ldb_o, int64_t inc_o,
                    double *save_sc, int32_t *info, int64_t B, int n, void *stream, const char *what) {
  cov_diag_kernel<MODE><<<dg_grid(B), DG_WARPS * 32, 0, (cudaStream_t)stream>>>(
      kind, scale_prec, s, ldb_s, inc_s, so, ldb_so, inc_so, eps_cov, gval, val, gout, ldb_g, inc_g, out, ldb_o, inc_o,
      save_sc, info, B, n);
  TCE_CHECK_LAUNCH(what);
  return TCE_OK;
}

}  // namespace

extern "C" int tce_gauss_stats_diag(const float *mean, const float *mean_o, const float *s, int64_t ldb_s,
                                    int64_t inc_s, const float *s_old, int64_t ldb_so, int64_t inc_so, double *out,
                                    int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!s_old || !out || B < 0 || n < 1 || n > DG_MAX_N || ldb_s < 0 || ldb_so < 0 || (!mean != !mean_o) ||
      (!s && !mean))
    return TCE_ERR_INVALID_ARGUMENT;
  gauss_stats_diag_kernel<<<dg_grid(B), DG_WARPS * 32, 0, (cudaStream_t)stream>>>(
      mean, mean_o, s, ldb_s, inc_s, s_old, ldb_so, inc_so, nullptr, out, nullptr, nullptr, 0, 0, B, n);
  TCE_CHECK_LAUNCH("gauss_stats_diag_kernel");
  return TCE_OK;
}

extern "C" int tce_gauss_stats_diag_bwd(const float *mean, const float *mean_o, const float *s, int64_t ldb_s,
                                        int64_t inc_s, const float *s_old, int64_t ldb_so, int64_t inc_so,
                                        const double *grad_out, float *grad_mean, float *grad_s, int64_t ldb_gs,
                                        int64_t inc_gs, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (!s_old || !grad_out || B < 0 || n < 1 || n > DG_MAX_N || ldb_s < 0 || ldb_so < 0 || (!mean != !mean_o) ||
      (!grad_mean && !grad_s) || (grad_s && (!s || dg_bad_out(grad_s, ldb_gs, B))) || (!s && !mean))
    return TCE_ERR_INVALID_ARGUMENT;
  gauss_stats_diag_kernel<<<dg_grid(B), DG_WARPS * 32, 0, (cudaStream_t)stream>>>(
      mean, mean_o, s, ldb_s, inc_s, s_old, ldb_so, inc_so, grad_out, nullptr, grad_mean, grad_s, ldb_gs, inc_gs, B, n);
  TCE_CHECK_LAUNCH("gauss_stats_diag_kernel(bwd)");
  return TCE_OK;
}

extern "C" int tce_proj_frob_diag_fwd(const float *s, int64_t ldb_s, int64_t inc_s, const float *s_old, int64_t ldb_so,
                                      int64_t inc_so, double eps_cov, float *out, int64_t ldb_o, int64_t inc_o,
                                      double *save_sc, int32_t *info, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (dg_bad_common(s, ldb_s, s_old, ldb_so, B, n) || !(eps_cov > 0) || dg_bad_out(out, ldb_o, B) || !save_sc)
    return TCE_ERR_INVALID_ARGUMENT;
  return cov_diag_launch<1>(0, 0, s, ldb_s, inc_s, s_old, ldb_so, inc_so, eps_cov, nullptr, nullptr, nullptr, 0, 0, out,
                            ldb_o, inc_o, save_sc, info, B, n, stream, "cov_diag_kernel(frob fwd)");
}

extern "C" int tce_proj_frob_diag_bwd(const float *s, int64_t ldb_s, int64_t inc_s, const float *s_old, int64_t ldb_so,
                                      int64_t inc_so, double eps_cov, const double *save_sc, const float *grad_out,
                                      int64_t ldb_g, int64_t inc_g, float *grad_s, int64_t ldb_gs, int64_t inc_gs,
                                      int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (dg_bad_common(s, ldb_s, s_old, ldb_so, B, n) || !(eps_cov > 0) || !save_sc || !grad_out || ldb_g < 0 ||
      dg_bad_out(grad_s, ldb_gs, B))
    return TCE_ERR_INVALID_ARGUMENT;
  return cov_diag_launch<2>(0, 0, s, ldb_s, inc_s, s_old, ldb_so, inc_so, eps_cov, nullptr, nullptr, grad_out, ldb_g,
                            inc_g, grad_s, ldb_gs, inc_gs, const_cast<double *>(save_sc), nullptr, B, n, stream,
                            "cov_diag_kernel(frob bwd)");
}

extern "C" int tce_proj_w2_diag_fwd(const float *s, int64_t ldb_s, int64_t inc_s, const float *s_old, int64_t ldb_so,
                                    int64_t inc_so, double eps_cov, int scale_prec, float *out, int64_t ldb_o,
                                    int64_t inc_o, double *save_sc, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (dg_bad_common(s, ldb_s, s_old, ldb_so, B, n) || !(eps_cov > 0) || dg_bad_out(out, ldb_o, B) || !save_sc)
    return TCE_ERR_INVALID_ARGUMENT;
  return cov_diag_launch<1>(1, scale_prec, s, ldb_s, inc_s, s_old, ldb_so, inc_so, eps_cov, nullptr, nullptr, nullptr, 0,
                            0, out, ldb_o, inc_o, save_sc, nullptr, B, n, stream, "cov_diag_kernel(w2 fwd)");
}

extern "C" int tce_proj_w2_diag_bwd(const float *s, int64_t ldb_s, int64_t inc_s, const float *s_old, int64_t ldb_so,
                                    int64_t inc_so, double eps_cov, int scale_prec, const double *save_sc,
                                    const float *grad_out, int64_t ldb_g, int64_t inc_g, float *grad_s, int64_t ldb_gs,
                                    int64_t inc_gs, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (dg_bad_common(s, ldb_s, s_old, ldb_so, B, n) || !(eps_cov > 0) || !save_sc || !grad_out || ldb_g < 0 ||
      dg_bad_out(grad_s, ldb_gs, B))
    return TCE_ERR_INVALID_ARGUMENT;
  return cov_diag_launch<2>(1, scale_prec, s, ldb_s, inc_s, s_old, ldb_so, inc_so, eps_cov, nullptr, nullptr, grad_out,
                            ldb_g, inc_g, grad_s, ldb_gs, inc_gs, const_cast<double *>(save_sc), nullptr, B, n, stream,
                            "cov_diag_kernel(w2 bwd)");
}

extern "C" int tce_cov_distance_diag(int kind, const float *s, int64_t ldb_s, int64_t inc_s, const float *s_old,
                                     int64_t ldb_so, int64_t inc_so, int scale_prec, const double *grad_val, double *val,
                                     float *grad_s, int64_t ldb_gs, int64_t inc_gs, int64_t B, int n, void *stream) {
  if (B == 0) return TCE_OK;              /* empty shard: pointers may be NULL */
  if (kind < 0 || kind > 1 || dg_bad_common(s, ldb_s, s_old, ldb_so, B, n) || (!grad_val && !val) ||
      (grad_val && dg_bad_out(grad_s, ldb_gs, B)))
    return TCE_ERR_INVALID_ARGUMENT;
  return cov_diag_launch<0>(kind, scale_prec, s, ldb_s, inc_s, s_old, ldb_so, inc_so, 0.0, grad_val, val, nullptr, 0, 0,
                            grad_val ? grad_s : nullptr, ldb_gs, inc_gs, nullptr, nullptr, B, n, stream,
                            "cov_diag_kernel(distance)");
}

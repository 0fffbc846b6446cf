/* tce_b200.h -- C ABI of libtce_b200.so: the B200-native (sm_100a) kernels of TCE's episodic
 * policy-update path.
 *
 * The reference (BruceGeLi/TCE_RL) has no FFI: the seam this library sits behind is the duck-typed
 * Python method surface of mprl.rl (policy / projection / agent classes created by the string
 * factories, mprl/rl/policy/__init__.py:19, mprl/rl/projection/__init__.py:40,
 * mprl/rl/agent/__init__.py:19).  Each entry point below cites the reference call it replaces.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer to a contiguous row-major array unless a stride is passed;
 *    float = fp32, double = fp64, indices int64, flags uint8 (torch.bool);
 *  - every call is asynchronous on `stream` (a cudaStream_t passed as void*), allocates nothing,
 *    never synchronises the host and is CUDA-graph capturable; the only allocation is the tables
 *    handle (explicit create / destroy);
 *  - return value: 0 = TCE_OK, negative = tce_status; numerical failures (non positive pivots) are
 *    reported LAPACK-style in device `info` arrays, never by aborting;
 *  - "L" is a lower-triangular Cholesky factor stored as a dense [n, n] matrix; only the lower
 *    triangle is read, gradients are written for the lower triangle (upper = 0);
 *  - `ldb` arguments are batch strides in elements; 0 broadcasts one matrix over the batch (the
 *    non-contextual covariance of every shipped TCE config, black_box_policy.py:53-55).
 */
#ifndef TCE_B200_H
#define TCE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  TCE_OK = 0,
  TCE_ERR_INVALID_ARGUMENT = -1,
  TCE_ERR_UNSUPPORTED_SHAPE = -2, /* (num_dof, num_basis+1) not in the instantiated kernel list */
  TCE_ERR_CUDA = -3,              /* a CUDA runtime call failed; see tce_last_cuda_error()        */
  TCE_ERR_WORKSPACE = -4          /* workspace too small                                          */
} tce_status;

int tce_version(void);
const char *tce_strerror(int status);
const char *tce_last_cuda_error(void);

/* ---- ProDMP configuration and pre-computed tables ------------------------------------------------
 * Replaces mp_pytorch's ExpDecayPhaseGenerator + ProDMPBasisGenerator(pre_compute_length_factor=5)
 * + ProDMP construction done by get_mp (mprl/util/util_mp.py:11-46).                              */
typedef struct {
  int32_t num_dof;
  int32_t num_basis;            /* K; parameters per DoF = K + 1 (weights + goal)                 */
  int32_t num_basis_outside;
  int32_t pre_compute_length_factor; /* 5 in the reference (util_mp.py:33)                         */
  int32_t auto_scale_basis;
  int32_t relative_goal;
  int32_t relative_goal_scaled; /* ambiguity switch, SURVEY App. A.4; 0 = g_eff = scale*g + y0    */
  int32_t reserved;
  double tau, delay, dt, alpha, alpha_phase, basis_bandwidth_factor, weights_scale, goal_scale;
} tce_mp_cfg;

typedef struct tce_tables tce_tables_t;

int tce_prodmp_tables_create(const tce_mp_cfg *cfg, void *stream, tce_tables_t **out);
void tce_prodmp_tables_destroy(tce_tables_t *tables);
int tce_prodmp_tables_num_pc(const tce_tables_t *tables);
/* copy the fp64 tables to HOST buffers (any pointer may be NULL): y1,y2,dy1,dy2 [N_pc];
 * pos_basis, vel_basis [N_pc, K+1]; scale [K+1] (= weights_goal_scale).  Synchronises.           */
int tce_prodmp_tables_export(const tce_tables_t *tables, double *y1, double *y2, double *dy1,
                             double *dy2, double *pos_basis, double *vel_basis, double *scale);

/* ---- (1) trajectory synthesis ---------------------------------------------------------------------
 * ProDMP.get_traj_pos / get_traj_vel as used by TemporalCorrelatedPolicy.sample
 * (mprl/rl/policy/temporal_correlated_policy.py:76-100).
 * params [B, D*(K+1)] (already sampled parameters, or the mean), times [B, T], init_time [B],
 * init_pos / init_vel [B, D] -> traj [B, T, 2*D] (pos | vel).                                     */
int tce_prodmp_traj_fwd(const tce_tables_t *tables, const float *params, const float *times,
                        const float *init_time, const float *init_pos, const float *init_vel,
                        float *traj, int64_t B, int64_t T, void *stream);
/* backward: grad_traj [B,T,2D] -> grad_params [B,Dp], grad_init_pos [B,D], grad_init_vel [B,D]
 * (any output may be NULL).  API-permitted, never exercised by the reference (sample runs under
 * no_grad, temporal_correlated_sampler.py:91,200).                                                */
/* tce_prodmp_traj_fwd for a batch whose episodes share ONE time grid (same init_time and times row: every shipped TCE
 * task): the basis rows are evaluated once (rows_ws: T * (2 * (K1 + 2) rounded up to a multiple of 4) floats of 16-byte
 * aligned workspace) and the batch becomes a
 * small matrix product per episode.  times_row [T] / init_time [1]: episode 0's values.                        */
int tce_prodmp_traj_fwd_uniform(const tce_tables_t *tables, const float *params, const float *times_row,
                                const float *init_time, const float *init_pos, const float *init_vel,
                                float *rows_ws, float *traj, int64_t B, int64_t T, void *stream);
int tce_prodmp_traj_bwd(const tce_tables_t *tables, const float *grad_traj, const float *times,
                        const float *init_time, float *grad_params, float *grad_init_pos,
                        float *grad_init_vel, int64_t B, int64_t T, void *stream);

/* ---- (2) Gaussian policy over the MP parameters -----------------------------------------------------
 * out = mean + L eps : MultivariateNormal(loc, scale_tril).rsample (black_box_policy.py:82-84 and
 * mp_pytorch sample_trajectories).  eps [B, n] is injected when not NULL, otherwise drawn in-kernel
 * from Philox4x32-10 (seed, offset) with Box-Muller (counter = element index: the draws do not depend on
 * which kernel serves an episode).  Per-episode factors of odd order n <= 64 that are contiguous
 * (ldb_L == n*n) and 16-byte aligned are streamed four episodes at a time by bulk asynchronous copies
 * (cp.async.bulk + mbarrier); everything else (stride 0, even n, the last B % 4 episodes) row by row.  */
int tce_mvn_rsample(const float *mean, const float *L, int64_t ldb_L, const float *eps, uint64_t seed,
                    uint64_t offset, float *out, int64_t B, int n, void *stream);
/* Batched Cholesky A = L L^T, one CTA per matrix in shared memory, n <= 128
 * (torch.linalg.cholesky via util_matrix.py:133 / the Frobenius + KL projections).                */
int tce_chol_fwd(const float *A, float *L, int32_t *info, int64_t B, int n, void *stream);
/* grad_A = sym(L^-T Phi(L^T grad_L) L^-1)  (SURVEY App. F)                                         */
int tce_chol_bwd(const float *L, const float *grad_L, float *grad_A, int64_t B, int n, void *stream);
/* policy head: covariance vector [B or 1, n + n(n-1)/2] -> L [B, n, n]
 * diag = softplus(v) + min_std, strictly lower filled row-major (abstract_policy.py:166-187,
 * util_numerical.py:44-68, util_matrix.py:12-33); ldb_vec = 0 broadcasts one vector.  Contiguous
 * 16-byte-aligned per-episode vectors (ldb_vec == n + n(n-1)/2, B >= 32) take the bulk-copy kernel.  */
int tce_policy_head_fwd(const float *vec, int64_t ldb_vec, float min_std, float *L, int64_t B, int n,
                        void *stream);
/* grad_vec [Bv, nvec]: Bv = B (ldb_vec != 0) or 1 (sum over the batch, ldb_vec == 0)               */
int tce_policy_head_bwd(const float *vec, int64_t ldb_vec, const float *grad_L, float *grad_vec,
                        int64_t B, int n, void *stream);
/* diagonal policy head (std_only): vec [B or 1, n] -> L [B, n, n] = diag(softplus(v) + min_std), zeros
 * elsewhere; ldb_vec = 0 broadcasts one vector.  The backward reads the diagonal of grad_L; grad_vec [Bv, n]
 * with Bv = 1 (ldb_vec == 0: summed over the batch in a fixed order) or B.                             */
int tce_policy_head_diag_fwd(const float *vec, int64_t ldb_vec, float min_std, float *L, int64_t B, int n,
                             void *stream);
int tce_policy_head_diag_bwd(const float *vec, int64_t ldb_vec, const float *grad_L, float *grad_vec,
                             int64_t B, int n, void *stream);
/* per-episode Gaussian scalars used by every projection / KL / entropy call
 * (black_box_policy.py:130-224, projection_utils.gaussian_kl):
 *   out[b, 0] = maha(mean, mean_o, L_o) = |L_o^-1 (mean - mean_o)|^2
 *   out[b, 1] = tr(Sigma_o^-1 Sigma)     = |L_o^-1 L|_F^2
 *   out[b, 2] = logdet Sigma = 2 sum log L_ii ;  out[b, 3] = logdet Sigma_o
 *   out[b, 4] = entropy(mean, L) = n/2 (1 + ln 2 pi) + sum log L_ii
 * L == NULL computes the Mahalanobis part only (out[b, 1] = out[b, 2] = 0).                          */
int tce_gauss_stats(const float *mean, const float *L, int64_t ldb_L, const float *mean_o,
                    const float *L_o, int64_t ldb_Lo, double *out, int64_t B, int n, void *stream);
/* gradient of the five scalars w.r.t. (mean, L) given grad_out [B,5] (the "other" distribution is data):
 * grad_mean [B,n] (may be NULL), grad_L [B,n,n] lower (NULL = mean part only).                       */
int tce_gauss_stats_bwd(const float *mean, const float *L, int64_t ldb_L, const float *mean_o,
                        const float *L_o, int64_t ldb_Lo, const double *grad_out, float *grad_mean,
                        float *grad_L, int64_t B, int n, void *stream);

/* maha [B] = |L_o^-1 (mean - mean_o)|^2 (policy.maha, black_box_policy.py:205-224) when grad_out == NULL;
 * otherwise grad_mean [B,n] = grad_out[b] * 2 Sigma_o^-1 (mean - mean_o) (maha may also be written).
 * n <= 64: one warp per episode (solves in registers); contiguous 16-byte-aligned factors of odd order are
 * fetched four episodes at a time by one bulk asynchronous copy; ldb_Lo = 0 broadcasts one factor.         */
int tce_gauss_maha(const float *mean, const float *mean_o, const float *L_o, int64_t ldb_Lo,
                   const double *grad_out, double *maha, float *grad_mean, int64_t B, int n, void *stream);
/* backward of tce_gauss_maha w.r.t. ALL arguments (BlackBoxPolicy.log_prob differentiates the Mahalanobis term w.r.t.
 * the distribution's own mean and factor, black_box_policy.py:95-128):  grad_mean [B,n] = 2 g L_o^-T L_o^-1 d
 * (d maha / d mean_o is its negative), grad_L [B,n,n] = -2 g tril(u z^T), z = L_o^-1 d, u = L_o^-T z; either may be
 * NULL.                                                                                                   */
int tce_gauss_maha_bwd_full(const float *mean, const float *mean_o, const float *L_o, int64_t ldb_Lo,
                            const double *grad_out, float *grad_mean, float *grad_L, int64_t B, int n,
                            void *stream);
/* Non-contextual policy: ONE L_o for all episodes (the reference repeats it B times,
 * black_box_policy.py:50-53).  tce_tri_inverse writes Linv [B,n,n] = L^-1 (fp64, B is normally 1);
 * tce_gauss_maha_shared is tce_gauss_maha with the two triangular solves per episode replaced by products
 * with that shared inverse; with grad_out == NULL and grad_mean != NULL it also writes d maha / d mean
 * (so that a backward pass is one elementwise product).                                                 */
int tce_tri_inverse(const float *L, int64_t ldb, double *Linv, int64_t B, int n, void *stream);
int tce_gauss_maha_shared(const float *mean, const float *mean_o, const double *Linv, const double *grad_out,
                          double *maha, float *grad_mean, int64_t B, int n, void *stream);

/* ---- (4a) differentiable trust-region projections ------------------------------------------------------
 * Replace the trust_region_projections layers (BruceGeLi/trust-region-layers@TCE_ICLR24) created by
 * projection_factory (mprl/rl/projection/__init__.py:19-40) and called at
 * temporal_correlated_agent.py:530-533; KL covariance part replaces cpp_projection (ITPAL).  n <= 64.
 *
 * mean projection (all layers): mean_part [B] fp64 is the layer's mean distance (1/2 maha for KL, maha or
 * squared Euclidean otherwise); proj = (mean + w mean_o) / (1 + w), w = sqrt(mean_part / eps) - 1 where
 * mean_part > eps, identity elsewhere.  bwd returns the gradient w.r.t. mean and w.r.t. mean_part.      */
int tce_proj_mean_fwd(const float *mean, const float *mean_o, const double *mean_part, double eps,
                      float *proj_mean, int64_t B, int n, void *stream);
int tce_proj_mean_bwd(const float *mean, const float *mean_o, const double *mean_part, double eps,
                      const float *grad_out, float *grad_mean, double *grad_mean_part, int64_t B, int n,
                      void *stream);
/* entropy projection: L * exp((beta - H(L)) / n) where H(L) < beta (always if equality); beta [B] fp64
 * (ldb_beta = 0 broadcasts one value); entropy [B] (optional) receives H(L) before the projection.       */
int tce_proj_entropy_fwd(const float *L, const double *beta, int64_t ldb_beta, int equality, float *out,
                         double *entropy, int64_t B, int n, void *stream);
int tce_proj_entropy_bwd(const float *L, const double *beta, int64_t ldb_beta, int equality,
                         const float *grad_out, float *grad_L, int64_t B, int n, void *stream);
/* Diagonal KL covariance projection (std_only policies), optionally followed by the entropy control of
 * tce_proj_entropy_fwd (beta == NULL: none).  Every diagonal is a strided vector: element i of episode b is
 * s[b * ldb + i * inc] (dense factor: ldb = n*n, inc = n+1; packed [B, n]: inc = 1; one shared vector: ldb = 0
 * on the inputs).  With lam_i = (s_old,i / s_i)^2 the projected variance is s_old,i^2 (1+eta) / (lam_i+eta), eta
 * the root of KL_cov(eta) = eps_cov where the KL before the projection exceeds eps_cov.  state [B, 4] fp64
 * {eta, active, alpha, entropy active} feeds the backward; info [B] (optional): 1 if a standard deviation is not
 * positive and finite.  The backward returns d loss / d s (s_old is a constant).  One warp per episode, n <= 1024. */
int tce_proj_kl_diag_fwd(const float *s, int64_t ldb_s, int64_t inc_s, const float *s_old, int64_t ldb_so,
                         int64_t inc_so, double eps_cov, const double *beta, int64_t ldb_beta, int equality,
                         float *out, int64_t ldb_o, int64_t inc_o, double *state, int32_t *info, int64_t B, int n,
                         void *stream);
int tce_proj_kl_diag_bwd(const float *s, int64_t ldb_s, int64_t inc_s, const float *s_old, int64_t ldb_so,
                         int64_t inc_so, const double *state, const float *grad_out, int64_t ldb_g, int64_t inc_g,
                         float *grad_s, int64_t ldb_gs, int64_t inc_gs, int64_t B, int n, void *stream);
/* KL covariance projection: min KL(N(.,S)||N(.,S~)) s.t. KL_cov(S||S_old) <= eps_cov, solved exactly on
 * the generalised eigenvalues (CTA-per-matrix one-sided Jacobi + Newton for eta); proj_L = chol(S_proj).
 * `save` (tce_proj_kl_save_doubles(B, n) doubles) carries M = L_old Q, U = L~^-1 M, L~^-1, Sigma_proj, lambda,
 * {eta, active, kl0, fingerprint, alpha, ent_active, alpha^2, -} to the backward (implicit differentiation of eta*).  warm_start != 0: `save` still holds the state of a previous call;
 * it is used to start the eigen-solve when it was produced with the same L_o (checked by a fingerprint),
 * e.g. across the epochs of one update_policy.  info [B]: non positive pivot of the final Cholesky.     */
size_t tce_proj_kl_save_doubles(int64_t B, int n);
int tce_proj_kl_cov_fwd(const float *L, const float *L_o, double eps_cov, float *proj_L, double *save,
                        int32_t *info, int warm_start, int64_t B, int n, void *stream);
int tce_proj_kl_cov_bwd(const float *L, const float *proj_L, const float *grad_out, const double *save,
                        float *grad_L, int64_t B, int n, void *stream);
/* The same projection followed by the entropy control of tce_proj_entropy_fwd in ONE launch (the two are
 * consecutive single-CTA kernels on the critical path of an epoch with a non-contextual covariance):
 * proj_L = KL projection (kept for the backward), out_L = alpha(proj_L) * proj_L.  The backward takes the
 * gradient w.r.t. out_L.                                                                                  */
int tce_proj_kl_entropy_fwd(const float *L, const float *L_o, double eps_cov, const double *beta,
                            int64_t ldb_beta, int equality, float *proj_L, float *out_L, double *save,
                            int32_t *info, int warm_start, int64_t B, int n, void *stream);
int tce_proj_kl_entropy_bwd(const float *L, const float *proj_L, const float *grad_out, const double *save,
                            float *grad_L, int64_t B, int n, void *stream);
/* tce_proj_kl_entropy_bwd when out_inv [B,n,n] = out_L^-1 (fp64, lower) is already known -- the trust-region loss
 * inverts the layer's output for its Mahalanobis term (tce_tri_inverse) -- so that the backward need not invert
 * proj_L itself (the largest single phase of that kernel).                                                */
int tce_proj_kl_entropy_bwd_inv(const float *L, const float *proj_L, const float *grad_out, const double *save,
                                const double *out_inv, float *grad_L, int64_t B, int n, void *stream);
/* Backward of tce_proj_kl_cov_fwd (fused_entropy = 0) / tce_proj_kl_entropy_fwd* (fused_entropy = 1) when the consumer
 * returns the gradient w.r.t. the output COVARIANCE Sigma_out = alpha^2 Sigma_proj [B,n,n] (symmetric, fp64) -- e.g.
 * grad_sigma of tce_seglik_uniform_finish / tce_seglik_dsigma_reduce -- instead of w.r.t. the factor: no Cholesky
 * adjoint, and the forward's factor (tce_proj_kl_entropy_fwd_chol) is off the critical path.
 * tr_coeff != 0 additionally adds the gradient of tr_coeff * KL_cov(N(., L L^T) || N(., Sigma_out)) with Sigma_out
 * DETACHED -- the covariance term of the trust-region regression loss (get_trust_region_loss,
 * temporal_correlated_agent.py:561-567), whose VALUE the forward leaves in the state (scalar 7 of a matrix): both
 * are closed forms on the saved eigen-system, so the loss term needs no kernel of its own.                      */
/* tce_proj_kl_entropy_bwd that also adds the gradient of the trust-region regression term
 * tr_coeff * KL_cov(N(L L^T) || N(Sigma_out)), Sigma_out = the layer's own (detached) output (closed form on the saved
 * eigen-system; get_trust_region_loss, temporal_correlated_agent.py:561-567).                              */
int tce_proj_kl_entropy_bwd_tr(const float *L, const float *proj_L, const float *grad_out, const double *save,
                               double tr_coeff, float *grad_L, int64_t B, int n, void *stream);
int tce_proj_kl_bwd_sigma(const float *L, const double *grad_sigma, const double *save, int fused_entropy,
                          double tr_coeff, float *grad_L, int64_t B, int n, void *stream);
/* tce_proj_kl_bwd_prep: K = L~^-T U~ into the state -- the part of the covariance-space backward that does not depend
 * on the incoming gradient; run it after the forward while the consumer of the covariance is busy.
 * tce_proj_kl_bwd_sigma_k: tce_proj_kl_bwd_sigma using that K (4 GEMMs instead of 5, one matrix load less).    */
/* Policy head fused into the projection (shipped configuration: one covariance vector for the batch):
 * tce_proj_kl_entropy_fwd_sigma_vec = tce_policy_head_fwd + tce_proj_kl_entropy_fwd_sigma in one launch (the factor is
 * also written to L_built); tce_proj_kl_bwd_sigma_k_vec = tce_proj_kl_bwd_sigma_k + tce_policy_head_bwd (gradient
 * w.r.t. the covariance vector, overwritten).  abstract_policy.py:166-187, black_box_policy.py:30-56.           */
int tce_proj_kl_entropy_fwd_sigma_vec(const float *vec, int64_t ldb_vec, float min_std, float *L_built,
                                      const float *L_o, double eps_cov, const double *beta, int64_t ldb_beta,
                                      int equality, float *proj_L, float *out_L, double *save, int32_t *info,
                                      int warm_start, int64_t B, int n, void *stream);
int tce_proj_kl_bwd_sigma_k_vec(const float *L, const float *vec, int64_t ldb_vec, const double *grad_sigma,
                                const double *save, int fused_entropy, double tr_coeff, float *grad_vec, int64_t B,
                                int n, void *stream);
int tce_proj_kl_bwd_prep(double *save, int64_t B, int n, void *stream);
int tce_proj_kl_bwd_sigma_k(const float *L, const double *grad_sigma, const double *save, int fused_entropy,
                            double tr_coeff, float *grad_L, int64_t B, int n, void *stream);
/* tce_proj_kl_entropy_fwd in two launches: _sigma writes the state (Sigma_proj, alpha = entropy scale from the
 * closed-form log-determinant, ...; for an inactive projection also the outputs); _chol forms
 * proj_L = chol(Sigma_proj) and out_L = alpha proj_L from the state.  What only needs the covariance
 * (the likelihood's Sigma0 inputs) can be ordered after the first launch alone.                            */
int tce_proj_kl_entropy_fwd_sigma(const float *L, const float *L_o, double eps_cov, const double *beta,
                                  int64_t ldb_beta, int equality, float *proj_L, float *out_L, double *save,
                                  int32_t *info, int warm_start, int64_t B, int n, void *stream);
/* out_inv (optional) [B,n,n] fp64: inverse of out_L (lower), for the Mahalanobis term of the trust-region loss   */
int tce_proj_kl_entropy_fwd_chol(const double *save, float *proj_L, float *out_L, double *out_inv, int32_t *info,
                                 int64_t B, int n, void *stream);
/* Frobenius: S_new = (S + eta S_old) / (1 + eta), eta = sqrt(|S_old - S|_F^2 / eps_cov) - 1; save_sc [B,4] */
int tce_proj_frob_cov_fwd(const float *L, const float *L_o, int64_t ldb_Lo, double eps_cov, float *proj_L,
                          double *save_sc, int32_t *info, int64_t B, int n, void *stream);
int tce_proj_frob_cov_bwd(const float *L, const float *L_o, int64_t ldb_Lo, double eps_cov,
                          const float *proj_L, const float *grad_out, const double *save_sc, float *grad_L,
                          int64_t B, int n, void *stream);
/* W2 (commutative): proj = (L + eta L_old) / (1 + eta) on the factors that are passed; save_sc [B,4]      */
int tce_proj_w2_cov_fwd(const float *L, const float *L_o, int64_t ldb_Lo, double eps_cov, int scale_prec,
                        float *proj_L, double *save_sc, int64_t B, int n, void *stream);
int tce_proj_w2_cov_bwd(const float *L, const float *L_o, int64_t ldb_Lo, double eps_cov, int scale_prec,
                        const float *grad_out, float *grad_L, int64_t B, int n, void *stream);
/* covariance distances of the Frobenius (kind 0) / W2 (kind 1) layers: val [B] when grad_val == NULL,
 * otherwise grad_L [B,n,n] = grad_val[b] * d val / d L (used by get_trust_region_loss).                 */
int tce_cov_distance(int kind, const float *L, const float *L_o, int64_t ldb_Lo, int scale_prec,
                     const double *grad_val, double *val, float *grad_L, int64_t B, int n, void *stream);

/* ---- (3) TCE segment-wise trajectory likelihood -----------------------------------------------------
 * TemporalCorrelatedPolicy.log_prob (temporal_correlated_policy.py:104-203) = mp.update_inputs +
 * get_traj_pos(flat) + get_traj_pos_cov + MultivariateNormal(covariance_matrix).log_prob.
 *
 * Stage 1 (gram):  per episode, C_bp = H_bp (L_b L_b^T) H_bp^T  (no regulariser) and the residual
 *                  r_bp = x_bp - mu_bp, both fp64 into `work`; max_b,p,i C_bp[i,i] is folded into
 *                  *diag_max (device double, caller zero-initialises) with an atomic max.
 * (collective)     at >1 GPU the caller all-reduces(MAX) *diag_max here.
 * Stage 2 (chol):  per segment, C += reg_rel * *diag_max * I, Cholesky, log-prob.  With grad_logp
 *                  [B,P] != NULL it writes the per-segment adjoints used by stage 3 to `adj` (same
 *                  size as `work`; may alias it).
 *                  With logp_old/advantage [B,P] != NULL instead, the surrogate loss of
 *                  temporal_correlated_agent.py:718-739 is fused: the upstream gradient is
 *                  -exp(lp - lp_old) * adv * grad_scale; its sum is added to loss_acc[0] and the sum of
 *                  ratio * grad_scale to loss_acc[1] (grad_scale = 1 / (B * P) gives loss = -mean(ratio *
 *                  adv) and the mean importance ratio).  loss_acc: 2 device doubles, caller zeroes.
 * Stage 3 (bwd):   per episode, from `adj`: grad_mean [B, Dp] and grad_L [B, Dp, Dp] (lower triangle),
 *                  both multiplied by *upstream (device float) when upstream != NULL.
 *
 * smp_traj [B, T, 2D] (only [:, pairs, :D] is read), mean [B, Dp], L [B, Dp, Dp] (batch stride
 * ldb_L, 0 = shared), times [B, T], init_* as above, pred_pairs [P, 2] int64.                       */
size_t tce_seglik_work_bytes(const tce_tables_t *tables, int64_t B, int64_t P);
int tce_seglik_gram(const tce_tables_t *tables, const float *smp_traj, const float *mean, const float *L,
                    int64_t ldb_L, const float *times, const float *init_time, const float *init_pos,
                    const float *init_vel, const int64_t *pred_pairs, void *work, double *diag_max,
                    int64_t B, int64_t T, int64_t P, void *stream);
int tce_seglik_chol(const tce_tables_t *tables, const void *work, void *adj, const double *diag_max, double reg_rel,
                    const float *grad_logp, const float *logp_old, const float *advantage,
                    double grad_scale, double *loss_acc, float *logp, int32_t *info, int64_t B,
                    int64_t P, void *stream);
int tce_seglik_bwd(const tce_tables_t *tables, const void *work, const float *L, int64_t ldb_L,
                   const float *times, const float *init_time, const int64_t *pred_pairs,
                   const float *upstream, float *grad_mean, float *grad_L, int64_t B, int64_t T, int64_t P,
                   void *stream);
/* Shapes.  The staged entry points above and below (and the diagonal likelihood) serve every supported shape:
 * 1 <= num_dof <= 8, 2 <= K1 <= 16, Dp = num_dof K1 <= 64.  The five (num_dof, K1) pairs (7, 9), (4, 9), (7, 4), (3, 4)
 * and (2, 3) have kernels specialised on num_dof and are the only shapes of the fused and uniform-grid entry points
 * (tce_seglik_fused_config ... tce_seglik_uniform_finish); other shapes run the staged kernels with num_dof read from
 * the tables.  Anything else returns TCE_ERR_UNSUPPORTED_SHAPE.
 * tce_seglik_compiled: 1 = one of the five specialised shapes, 0 = supported by the staged path only,
 * TCE_ERR_UNSUPPORTED_SHAPE = outside the supported set.  Host only, no launch.                                      */
int tce_seglik_compiled(const tce_tables_t *tables);
/* Stage 1 for ONE covariance shared by the batch, given as Sigma = (*sigma_scale) * Sigma0 [Dp, Dp] fp64 (device
 * pointers; sigma_scale may be NULL = 1) instead of its factor -- e.g. straight out of tce_proj_kl_entropy_fwd's
 * state.  Stages 2 and 3 as for tce_seglik_gram (stage 3 through tce_seglik_bwd_shared).                       */
int tce_seglik_gram_sigma(const tce_tables_t *tables, const float *smp_traj, const float *mean,
                          const double *Sigma0, const double *sigma_scale, const float *times,
                          const float *init_time, const float *init_pos, const float *init_vel,
                          const int64_t *pred_pairs, void *work, double *diag_max, int64_t B, int64_t T, int64_t P,
                          void *stream);
/* Stage 3 for ONE covariance shared by the batch (a factor L [Dp, Dp] given to tce_seglik_gram with ldb_L = 0, or
 * tce_seglik_gram_sigma): grad_mean [B, Dp] (may be NULL) per episode as tce_seglik_bwd; the gradient w.r.t. the
 * covariance is summed over the batch in a fixed order (per-CTA partials, then one reduce; no atomics), so two calls
 * on the same inputs give the same bits.  grad_sigma [Dp, Dp] fp64 = upstream * sum_b d lp_b / d Sigma (symmetric),
 * grad_L [Dp, Dp] fp32 = 2 tril(grad_sigma L) (needs L); either may be NULL, not both.  part: workspace of
 * tce_seglik_shared_part_doubles(tables, B) doubles (0: unsupported shape or B < 1).  Three launches.        */
size_t tce_seglik_shared_part_doubles(const tce_tables_t *tables, int64_t B);
int tce_seglik_bwd_shared(const tce_tables_t *tables, const void *work, const float *L, const float *times,
                          const float *init_time, const int64_t *pred_pairs, const float *upstream, float *grad_mean,
                          double *part, float *grad_L, double *grad_sigma, int64_t B, int64_t T, int64_t P,
                          void *stream);
/* Diagonal covariance (std_only policies, per-episode standard deviations s, strided as for tce_proj_kl_diag_*):
 * C is block diagonal with one 2 x 2 block per (pair, DoF), C_d[k,k'] = sum_j h_kj h_k'j s_{d,j}^2 + reg.
 * tce_seglik_diag_max: the regulariser seed diag_max = max over the batch of diag C (atomic max into *diag_max,
 * zero it first; all-reduce(MAX) it between the launches at > 1 GPU).  tce_seglik_diag_fwd: logp [B, P], info [B, P]
 * (optional; first non-positive pivot as in tce_seglik_chol).  tce_seglik_diag_bwd: from grad_logp [B, P],
 * grad_mean [B, Dp] and grad_s (strided, ldb_gs > 0), either may be NULL.  fp64 arithmetic, fixed summation order. */
int tce_seglik_diag_max(const tce_tables_t *tables, const float *s, int64_t ldb_s, int64_t inc_s,
                        const float *times, const float *init_time, const int64_t *pred_pairs, double *diag_max,
                        int64_t B, int64_t T, int64_t P, void *stream);
int tce_seglik_diag_fwd(const tce_tables_t *tables, const float *smp_traj, const float *mean, const float *s,
                        int64_t ldb_s, int64_t inc_s, const float *times, const float *init_time,
                        const float *init_pos, const float *init_vel, const int64_t *pred_pairs,
                        const double *diag_max, double reg_rel, float *logp, int32_t *info, int64_t B, int64_t T,
                        int64_t P, void *stream);
int tce_seglik_diag_bwd(const tce_tables_t *tables, const float *smp_traj, const float *mean, const float *s,
                        int64_t ldb_s, int64_t inc_s, const float *times, const float *init_time,
                        const float *init_pos, const float *init_vel, const int64_t *pred_pairs,
                        const double *diag_max, double reg_rel, const float *grad_logp, float *grad_mean,
                        float *grad_s, int64_t ldb_gs, int64_t inc_gs, int64_t B, int64_t T, int64_t P,
                        void *stream);

/* ---- (3') the same likelihood, fused: product path of TemporalCorrelatedPolicy.log_prob / segment_surrogate --------
 * (temporal_correlated_policy.py:104-203 + temporal_correlated_agent.py:718-739).
 *
 * tce_seglik_prepass : per episode the basis rows of its distinct time points and the residuals r = x - mu into `pre`
 *                      (tce_seglik_fused_config: pre_doubles_per_episode doubles per episode, ~5 KB for box pushing --
 *                      the only HBM intermediate of the path), and max_{b,p,i} C_bp[i,i] folded into *diag_max (caller
 *                      zeroes it; at >1 GPU the caller all-reduces(MAX) it before the next call).  Covariance either
 *                      as factors L (batch stride ldb_L, 0 = one shared factor) or as Sigma = (*sigma_scale) * Sigma0
 *                      [Dp,Dp] fp64 (Sigma0 != NULL; sigma_scale may be NULL = 1).
 * tce_seglik_fused   : ONE persistent kernel: gram, per-segment Cholesky, log-prob, and for grad_mode != 0 the whole
 *                      backward.  grad_mode 0: logp / info only.  1: upstream gradient grad_logp [B,P].  2: fused
 *                      surrogate: g = -exp(lp - logp_old) * advantage * grad_scale, loss_acc[0] += sum g,
 *                      loss_acc[1] += sum ratio * grad_scale (loss_acc: 2 device doubles, caller zeroes).
 *                      Outputs (any may be NULL): logp [B,P], info [B,P] (first non-positive pivot + 1), grad_mean
 *                      [B,Dp]; per-episode factors: grad_L [B,Dp,Dp] (lower, upper = 0); shared covariance:
 *                      dsigma_part (part_floats floats from tce_seglik_fused_config: one partial d loss / d Sigma per
 *                      CTA in DoF-block layout, then the reduce kernel's sum and ticket), to be finished by
 *                      tce_seglik_dsigma_reduce(nparts = grid): grad_L [Dp,Dp] = 2 tril((sum partials) L) * (*upstream)
 *                      and / or grad_sigma [Dp,Dp] (dense symmetric).
 *                      `chained` != 0 claims pred_pairs[p][1] == pred_pairs[p+1][0] for all p (the fixed-interval
 *                      selection of every TCE config: P + 1 distinct time points instead of 2 P); a wrong claim is
 *                      refused (info[0] = -7, nothing computed).  The same value must be given to both calls.
 * Uniform time grid (every episode has the same init_time and times row) + shared covariance: C_p, its Cholesky
 * factor and its inverse are identical for all episodes.  tce_seglik_uniform_prep (what & 1: basis rows + C_p + diag
 * max from episode 0's grid; what & 2: factor / inverse / logdet per segment; a multi-GPU caller may all-reduce
 * *diag_max between two calls), tce_seglik_uniform_main (per episode: residual, log-prob, grad_mean; per CTA the sums
 * of g alpha alpha^T into `apart`, sizes from tce_seglik_uniform_parts) and tce_seglik_uniform_finish (one CTA:
 * adjoints -> dSigma -> grad_L / grad_sigma) replace pre-pass + fused kernel + reduce in that case.
 * ws: tce_seglik_uniform_ws_doubles(P) doubles.                                                                 */
int tce_seglik_fused_config(const tce_tables_t *tables, int64_t B, int64_t P, int chained, int32_t *episodes_per_iter,
                            int32_t *grid, int64_t *part_floats, int64_t *pre_doubles_per_episode);
int tce_seglik_prepass(const tce_tables_t *tables, const float *smp_traj, const float *mean, const float *L,
                       int64_t ldb_L, const double *Sigma0, const double *sigma_scale, const float *times,
                       const float *init_time, const float *init_pos, const float *init_vel,
                       const int64_t *pred_pairs, double *pre, double *diag_max, int chained, int64_t B, int64_t T,
                       int64_t P, void *stream);
int tce_seglik_fused(const tce_tables_t *tables, const double *pre, const float *L, int64_t ldb_L,
                     const double *Sigma0, const double *sigma_scale, const int64_t *pred_pairs,
                     const double *diag_max, double reg_rel, int grad_mode, const float *grad_logp,
                     const float *logp_old, const float *advantage, double grad_scale, double *loss_acc, float *logp,
                     int32_t *info, float *grad_mean, float *grad_L, float *dsigma_part, int chained, int64_t B,
                     int64_t P, void *stream);
int tce_seglik_dsigma_reduce(const tce_tables_t *tables, float *dsigma_part, int nparts, const float *L,
                             const float *upstream, float *grad_L, double *grad_sigma, void *stream);
size_t tce_seglik_uniform_ws_doubles(const tce_tables_t *tables, int64_t P);
int tce_seglik_uniform_parts(const tce_tables_t *tables, int64_t B, int64_t P, int32_t *nparts,
                             int64_t *apart_doubles);
int tce_seglik_uniform_prep(const tce_tables_t *tables, const float *L, const double *Sigma0,
                            const double *sigma_scale, const float *times, const float *init_time,
                            const int64_t *pred_pairs, double *ws, double *diag_max, double reg_rel, int what,
                            int64_t P, void *stream);
int tce_seglik_uniform_main(const tce_tables_t *tables, const double *ws, const float *smp_traj, const float *mean,
                            const float *init_pos, const float *init_vel, const int64_t *pred_pairs, int grad_mode,
                            const float *grad_logp, const float *logp_old, const float *advantage,
                            double grad_scale, double *loss_acc, float *logp, int32_t *info, float *grad_mean,
                            double *apart, int64_t B, int64_t T, int64_t P, void *stream);
int tce_seglik_uniform_finish(const tce_tables_t *tables, double *ws, const double *apart, int nparts,
                              const float *L, const float *upstream, float *grad_L, double *grad_sigma, int64_t P,
                              void *stream);

/* ---- (4b) GAE and segment advantages ------------------------------------------------------------------
 * TemporalCorrelatedAgent.get_advantage_return (temporal_correlated_agent.py:118-181).
 * rewards [B,T], values [B,T+1], dones / time_limit_dones [B,T] uint8 -> adv, ret [B,T].            */
int tce_gae(const float *rewards, const float *values, const uint8_t *dones, const uint8_t *tl_dones,
            float gamma, float lam, int use_gae, float *adv, float *ret, int64_t B, int64_t T,
            void *stream);
/* get_segment_advantage (temporal_correlated_agent.py:183-321); mode 0 = accumulate (expects
 * `advantages`), 1 = value_subtraction, 2 = accumulated_rewards (un-normalised part only).
 * Writes raw segment advantages [B,P] and adds {count, sum, sum of squares} to stats[3] (device
 * doubles, caller zero-initialises; all-reduced(SUM) by the caller at >1 GPU).                      */
int tce_segment_advantage_raw(int mode, const float *rewards, const float *values, const float *advantages,
                              const int64_t *pred_pairs, float gamma, float *seg, double *stats, int64_t B,
                              int64_t T, int64_t P, void *stream);
/* adds {count, sum, sum of squares} of x[N] to stats[3] */
int tce_sum_stats(const float *x, double *stats, int64_t N, void *stream);
/* (x - mean) / (std_unbiased + 1e-8) with mean/std from stats[3] (temporal_correlated_agent.py:281-284) */
int tce_normalize_by_stats(float *x, const double *stats, int64_t N, void *stream);

/* ---- optimiser step of the policy epoch (temporal_correlated_agent.py:561-589: clip_grad_norm_, Adam.step) ----
 * All gradients live in ONE flat fp32 buffer (16-byte aligned) in the order of `params`.
 * tce_grad_sumsq: state[0] += 1 (step counter), state[1] += sum g^2 (caller zeroes state[1] beforehand).
 * tce_adam_step : torch.optim.Adam (L2 weight decay, bias correction with t = state[0], no amsgrad) on the
 *                 gradient scaled by min(1, max_norm / (sqrt(state[1]) + 1e-6)) (max_norm <= 0: no clipping).
 *                 A non-finite gradient norm skips the update (parameters and moments stay intact: the reference
 *                 raises BEFORE backward/step on a NaN loss, temporal_correlated_agent.py:569-577).
 * `params` / `sizes` are HOST arrays (count <= 32) of device pointers and element counts; m, v are flat fp32
 * moment buffers of sum(sizes) elements.                                                                   */
int tce_grad_sumsq(const float *grad_flat, int64_t n, double *state, void *stream);
int tce_adam_step(int count, float *const *params, const int64_t *sizes, const float *grad_flat, float *m,
                  float *v, const double *state, double max_norm, double lr, double beta1, double beta2,
                  double eps, double weight_decay, void *stream);

/* ---- data-parallel gradient exchange fused with the gradient norm, over NVLink peer memory (csrc/tce_p2p.cu) ----
 * Replaces ncclAllReduce(AVG) of the flat gradient + tce_grad_sumsq per optimiser step (SURVEY 8(e) collective (1)).
 * peer_bufs[r] / peer_pads[r] (HOST arrays of `world` device pointers): rank r's flat gradient buffer (n floats,
 * 16-byte aligned) and signal pad (>= 2 * world uint64, zero-initialised once) as mapped into THIS process
 * (symmetric memory: torch.distributed._symmetric_memory rendezvous, or cudaIpc / cuMem mappings).
 * avg_out [n] (local) receives (1/world) * sum_r peer_bufs[r] summed in rank order (bit-identical on all ranks);
 * state3 = {step += 1, sum of squares of avg_out += , error flag (1 = a peer did not arrive within ~2 s)};
 * local2 = two uint64 of local device memory, zero-initialised once (launch sequence number, block ticket).
 * Every rank must launch it the same number of times.  On return (stream order) every peer has finished reading
 * this rank's buffer, which may then be overwritten.                                                         */
int tce_p2p_allreduce_sumsq(int world, int rank, const void *const *peer_bufs, void *const *peer_pads, int64_t n,
                            float *avg_out, void *local2, double *state3, void *stream);
/* The same exchange restricted to elements [offset, offset + n) of the buffers (offset a multiple of 4), so that an
 * update can exchange the gradient in up to two ranges as they become final (the mean network's slice while the
 * covariance chain is still in its backward, the covariance slice last): `phase` in {0, 1} selects the 2 * world
 * signal-pad slots [2 * world * phase, ...) and the two uint64 local2[2 * phase ..]; pads need >= 4 * world uint64 and
 * local2 four uint64 when phase 1 is used.  `bump_step`: this call increments state3[0] (once per optimiser step).
 * Sums of squares of all ranges accumulate in state3[1].                                                     */
int tce_p2p_allreduce_sumsq_range(int world, int rank, const void *const *peer_bufs, void *const *peer_pads,
                                  int64_t offset, int64_t n, int phase, int bump_step, float *avg_out, void *local2,
                                  double *state3, void *stream);

/* Push variant (the one the agent uses): no arrival / departure barriers.  peer_xchg[r]: rank r's exchange area
 * (tce_p2p_push_xchg_bytes(world, n_total) bytes of symmetric memory, zero-initialised once: per-block flags followed by
 * receive slots [2 parities][world][n_total rounded up to 4]) as mapped into this process; grad: this rank's LOCAL flat
 * gradient (n_total floats, padded with zeros to a multiple of 4, 16-byte aligned).  Each block stores its slice of
 * grad[offset, offset + n) into every peer's slot, releases a per-block flag, waits for the peers' flags of the same
 * block and reduces from local memory in rank order.  offset, n multiples of 4; phase / bump_step / local2 / state3 as
 * for tce_p2p_allreduce_sumsq_range.  Every rank must launch the same sequence of calls.                       */
size_t tce_p2p_push_xchg_bytes(int world, int64_t n_total);
int tce_p2p_push_allreduce_sumsq(int world, int rank, void *const *peer_xchg, const float *grad, int64_t n_total,
                                 int64_t offset, int64_t n, int phase, int bump_step, float *avg_out, void *local2,
                                 double *state3, void *stream);

/* ---- mean chain of a policy epoch with ONE shared covariance (csrc/tce_epoch.cu) -----------------------------
 * Replaces, for the non-contextual policies of every shipped config, the per-episode pieces between the policy
 * network and the segment likelihood: the mean part of the KL metric and the mean projection
 * (trust_region_projections mean_projection via temporal_correlated_agent.py:530-533), its backward, the mean part of
 * the trust-region regression loss with its gradient (get_trust_region_loss, :561-567) and the batch means of the
 * logging decomposition (:641-686).
 * tce_epoch_mean_fwd : Linv_old = L_old^-1 [n,n] fp64 (tce_tri_inverse) -> proj_mean [B,n], maha_old [B] =
 *                      |L_old^-1 (mean - mean_old)|^2, u_old [B,n] = Sigma_old^-1 (mean - mean_old);
 *                      acc[0] += sum_b 1/2 maha_old, acc[1] += sum_b 1/2 maha(proj_mean, mean_old).
 * tce_epoch_tr_mean  : Linv_new = L~^-1 [n,n] fp64 and kl_scalars [16] as left in the state by
 *                      tce_proj_kl_entropy_fwd(_sigma) -> tr_grad [B,n] = tr_coeff / B * Sigma_out^-1 (mean - proj_mean),
 *                      Sigma_out^-1 = (Sigma~^-1 + eta Sigma_old^-1) / (alpha^2 (1 + eta));  acc[2] += sum_b 1/2
 *                      maha(mean, proj_mean; Sigma_out).  Needs nothing of the likelihood: runs beside it.
 * tce_epoch_mean_combine : g_proj_mean = d loss / d proj_mean [B,n] -> grad_mean [B,n] = mean-projection adjoint of g
 *                      + tr_grad (may be NULL).
 * tce_epoch_metrics  : out19 = the 7 loss values + 12 KL logging means of one epoch (rl/agent.py key order) from
 *                      acc[3], lik_stats {surrogate, mean ratio}, kl_scalars, adam_stats {step, sum g^2} (may be NULL).
 * acc is zero-initialised by the caller; everything is asynchronous on `stream`.                                */
int tce_epoch_mean_fwd(const float *mean, const float *mean_old, const double *Linv_old, double eps_mean,
                       float *proj_mean, double *maha_old, float *u_old, double *acc, int64_t B, int n,
                       void *stream);
int tce_epoch_tr_mean(const float *mean, const float *mean_old, const double *maha_old, const float *u_old,
                      const double *Linv_new, const double *kl_scalars, double eps_mean, double tr_coeff,
                      float *tr_grad, double *acc, int64_t B, int n, void *stream);
int tce_epoch_mean_combine(const float *g_proj_mean, const float *mean, const float *mean_old, const double *maha_old,
                           const float *u_old, const float *tr_grad, double eps_mean, float *grad_mean, int64_t B,
                           int n, void *stream);
int tce_epoch_metrics(const double *acc, const double *lik_stats, const double *kl_scalars, const double *adam_stats,
                      int64_t B, double tr_coeff, int with_cov, double ent_coef, double *out19, void *stream);

/* ---- measurement helper ---------------------------------------------------------------------------------
 * One register-resident FMA-chain kernel (fp32 or fp64) over the whole chip; *flops (host) receives the
 * FLOPs executed.  bench.py times it to obtain the FMA-pipe roofline denominators.                      */
/* Profiling aids, functional only when the library is built with -DTCE_PROFILE (otherwise they return
 * TCE_ERR_UNSUPPORTED_SHAPE and the kernels contain no stamps): SM-clock stamps taken between the phases of the last
 * KL forward ([0..15]) / covariance-space backward ([16..31]) launch                                              */
int tce_debug_kl_phase_cycles(long long *out32);
/* same for block 0 of the last tce_seglik_gram ([0..6]) / tce_seglik_bwd ([16..21]) launches */
int tce_debug_seglik_phase_cycles(long long *out32);
int tce_bench_fma(int fp64, int iters, void *scratch, double *flops, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* TCE_B200_H */

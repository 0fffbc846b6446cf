"""Gaussian policies over ProDMP parameters with the reference's API, evaluated by the CUDA kernels.

Reference: mprl/rl/policy/abstract_policy.py:10-328, black_box_policy.py:30-224,
temporal_correlated_policy.py:34-203; factory mprl/rl/policy/__init__.py:8-19.
"""
from __future__ import annotations

import torch

from .. import ops, util
from ..mp import get_mp


class AbstractGaussianPolicy:
    def __init__(self, dim_in, dim_out, mean_net_args, variance_net_args, init_method, out_layer_gain,
                 act_func_hidden, act_func_last, dtype="torch.float32", device="cuda", **kwargs):
        self.dim_in, self.dim_out = dim_in, dim_out
        variance_net_args = dict(variance_net_args)
        self.contextual_cov = variance_net_args.pop("contextual")
        self.std_only = variance_net_args.pop("std_only")
        self.mean_net_args, self.variance_net_args = mean_net_args, variance_net_args
        self.init_method, self.out_layer_gain = init_method, out_layer_gain
        self.act_func_hidden, self.act_func_last = act_func_hidden, act_func_last
        self.dtype, self.device = util.parse_dtype_device(dtype, device)
        if self.dtype != torch.float32:
            raise NotImplementedError("the sm_100a kernels take fp32 tensors (fp64 is used internally where "
                                      "the arithmetic is ill conditioned); pass dtype=float32")
        self.num_dof = dim_out
        self.min_std = float(kwargs.get("min_std", 1e-2))
        self.mean_net = self.variance_net = None
        self._create_network()

    def _create_network(self):
        mk = lambda name, dim_out, args: util.MLP(name=name, dim_in=self.dim_in, dim_out=dim_out,
                                                  hidden_layers=util.mlp_arch_3_params(**args),
                                                  init_method=self.init_method, out_layer_gain=self.out_layer_gain,
                                                  act_func_hidden=self.act_func_hidden,
                                                  act_func_last=self.act_func_last, dtype=self.dtype,
                                                  device=self.device)
        cls = self.__class__.__name__
        self.mean_net = mk(cls + "_mean", self.dim_out, self.mean_net_args)
        dim_var = self.dim_out if self.std_only else self.dim_out + self.dim_out * (self.dim_out - 1) // 2
        if self.contextual_cov:
            self.variance_net = mk(cls + "_variance", dim_var, self.variance_net_args)
        else:
            vec = torch.zeros(dim_var, dtype=self.dtype, device=self.device)
            # abstract_policy.py:113-116: inverse softplus of 1 with the DEFAULT bound (1e-2), not min_std
            vec[:self.dim_out] += util.reverse_from_softplus_space(
                torch.ones(self.dim_out, dtype=self.dtype, device=self.device), lower_bound=None)
            self.variance_net = util.TrainableVariable(cls + "_variance", vec)

    @property
    def network(self):
        return self.mean_net, self.variance_net

    @property
    def parameters(self):
        return list(self.mean_net.parameters()) + list(self.variance_net.parameters())

    @property
    def contextual_std(self):
        return self.contextual_cov

    @property
    def contextual(self):
        return True

    @property
    def is_diag(self):
        return self.std_only

    def save_weights(self, log_dir: str, epoch: int):
        """abstract_policy.py:140-151, files in the reference's layout (rollout.save_mlp / save_variable)."""
        from .. import rollout
        rollout.save_net(self.mean_net, log_dir, epoch)
        rollout.save_net(self.variance_net, log_dir, epoch)

    def load_weights(self, log_dir: str, epoch: int):
        from .. import rollout
        rollout.load_net(self.mean_net, log_dir, epoch)
        rollout.load_net(self.variance_net, log_dir, epoch)

    def _vector_to_cholesky(self, cov_val: torch.Tensor, batch: int | None = None):
        """softplus(diag) + min_std, strictly-lower row-major fill (std_only: diagonal only) -- one fused kernel
        (``tce::policy_head`` / ``tce::policy_head_diag``)."""
        head = ops.policy_head_diag if self.std_only else ops.policy_head
        if cov_val.dim() == 1:
            return head(cov_val, int(batch), self.dim_out, self.min_std)
        return head(cov_val, cov_val.shape[0], self.dim_out, self.min_std)

    def _cholesky_to_vector(self, params_L: torch.Tensor):
        diag, off = util.reverse_build_matrix(params_L, not self.std_only)
        diag = util.reverse_from_softplus_space(diag, self.min_std)
        return diag if self.std_only else torch.cat([diag, off], dim=-1)

    def set_cov_variable(self, param_L: torch.Tensor):
        assert self.contextual_std is False, "Variance is a net instead of a variable."
        self.variance_net.variable.data = self._cholesky_to_vector(param_L).detach()


class BlackBoxPolicy(AbstractGaussianPolicy):
    def policy(self, obs):
        """-> (params_mean [B, Dp], params_L [B, Dp, Dp])   (black_box_policy.py:30-56)."""
        if self.contextual_cov:
            return self.mean_net(obs), self._vector_to_cholesky(self.variance_net(obs))
        return self.mean_net(obs), self.shared_params_L(obs.shape[0])

    def shared_params_L(self, batch: int):
        """The ONE factor of a non-contextual policy, broadcast over the batch with stride 0.  The reference
        expands the parameter vector and materialises B equal factors (black_box_policy.py:50-53); every
        consumer here reads the first one (``rl/projection.py:_first``) or a stride-0 view."""
        first = self._vector_to_cholesky(self.variance_net.variable, 1)
        params_L = first.expand(batch, -1, -1)
        params_L._tce_first = first
        return params_L

    def sample(self, require_grad, params_mean, params_L, use_mean=False, eps=None):
        if use_mean:
            smp = params_mean
        else:
            seed = int(torch.randint(0, 2 ** 62, [], device="cpu").item()) if eps is None else 0
            with torch.set_grad_enabled(bool(require_grad) and torch.is_grad_enabled()):   # nothing saved for a backward
                smp = ops.mvn_rsample(params_mean, params_L, eps, seed, 0)
        return smp if require_grad else smp.detach()

    def log_prob(self, smp_params, params_mean, params_L, **kwargs):
        """MVN(loc, scale_tril).log_prob (black_box_policy.py:95-128) = -1/2 (k ln 2pi + maha) - 1/2 logdet."""
        k = params_mean.shape[-1]
        maha = ops.gauss_maha(smp_params, params_mean, params_L)
        return (-0.5 * (k * 1.8378770664093453 + maha) - 0.5 * self.log_determinant(params_L)).to(params_mean.dtype)

    def entropy(self, params):
        """1/2 k (1 + ln 2 pi) + sum log L_ii (MultivariateNormal.entropy, black_box_policy.py:130-154)."""
        L = params[1]
        k = L.shape[-1]
        return 0.5 * k * (1.0 + 1.8378770664093453) + torch.diagonal(L, dim1=-2, dim2=-1).log().sum(-1)

    def covariance(self, params_L):
        return torch.einsum('...ij,...kj->...ik', params_L, params_L)

    def log_determinant(self, params_L):
        return 2 * torch.diagonal(params_L, dim1=-2, dim2=-1).log().sum(-1)

    def precision(self, params_L):
        eye = torch.eye(params_L.shape[-1], dtype=params_L.dtype, device=params_L.device)
        return torch.cholesky_solve(eye, params_L, upper=False)

    def maha(self, params, params_other, params_L):
        return ops.gauss_maha(params, params_other, params_L).to(params.dtype)


class TemporalCorrelatedPolicy(BlackBoxPolicy):
    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.mp = get_mp(**kwargs["mp"])
        self.num_dof = self.mp.num_dof

    def sample(self, require_grad, params_mean, params_L, times, init_time, init_pos, init_vel, use_mean=False,
               eps=None):
        """Trajectory [B, T, 2 D] (pos | vel) of sampled (or mean) ProDMP parameters
        (temporal_correlated_policy.py:34-102); ``eps`` [B, Dp] injects the normal draw."""
        with torch.set_grad_enabled(bool(require_grad) and torch.is_grad_enabled()):      # nothing saved for a backward
            if use_mean:
                theta = params_mean
            else:
                seed = int(torch.randint(0, 2 ** 62, [], device="cpu").item()) if eps is None else 0
                theta = ops.mvn_rsample(params_mean, params_L, eps, seed, 0)
            traj = ops.prodmp_traj(theta, times, init_time, init_pos, init_vel, self.mp.tables.handle, self.num_dof)
        return traj if require_grad else traj.detach()

    def log_prob(self, smp_traj, params_mean, params_L, times, init_time, init_pos, init_vel, **kwargs):
        """TCE segment-wise likelihood [B, P] (temporal_correlated_policy.py:104-203)."""
        pred_pairs = kwargs["pred_pairs"]
        if self._per_episode_diag(params_L, times.shape[0]):
            return ops.seg_logprob_diag(smp_traj, params_mean, params_L, times, init_time, init_pos, init_vel,
                                        pred_pairs, self.mp.tables)
        return ops.seg_logprob(smp_traj, params_mean, params_L, times, init_time, init_pos, init_vel, pred_pairs,
                               self.mp.tables)

    def _per_episode_diag(self, params_L, batch):
        """std_only with one factor per episode: the block-diagonal (2 x 2 per DoF) likelihood.  A factor shared by
        the batch keeps the shared-covariance path, which forms the trajectory covariance once per batch."""
        return self.is_diag and ops.shared_factor(params_L, batch) is None

    def segment_surrogate(self, smp_traj, params_mean, params_L, times, init_time, init_pos, init_vel, pred_pairs,
                          log_prob_old, advantages):
        """Fused ``log_prob`` + ``surrogate_loss`` (temporal_correlated_agent.py:538-550,718-739): returns
        (-mean(exp(lp_new - lp_old) * adv), mean importance ratio, lp_new) from two kernels, backward = one.
        Per-episode diagonal factors: the diagonal likelihood, then the surrogate formula of the agent on its log-probs."""
        if self._per_episode_diag(params_L, times.shape[0]):
            lp = ops.seg_logprob_diag(smp_traj, params_mean, params_L, times, init_time, init_pos, init_vel, pred_pairs,
                                      self.mp.tables)
            ratio = (lp - log_prob_old).exp()
            return -(ratio * advantages).mean(), ratio.mean().detach(), lp.detach()
        return ops.seg_surrogate(smp_traj, params_mean, params_L, times, init_time, init_pos, init_vel, pred_pairs,
                                 log_prob_old, advantages, self.mp.tables)


def policy_factory(typ: str, **kwargs):
    """mprl/rl/policy/__init__.py:8-19."""
    return {"TemporalCorrelatedPolicy": TemporalCorrelatedPolicy, "BlackBoxPolicy": BlackBoxPolicy}[typ](**kwargs)

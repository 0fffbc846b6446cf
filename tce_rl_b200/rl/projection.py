"""Differentiable trust-region projection layers with the API of ``trust_region_projections``.

Reference: factory mprl/rl/projection/__init__.py:19-40; call sites
mprl/rl/agent/temporal_correlated_agent.py:439-441 (initial_entropy), :530-533 (projection),
:561-567 (get_trust_region_loss), black_box_agent.py:359-363 (compute_metrics).  The layer classes
themselves live in the unvendored BruceGeLi/trust-region-layers@TCE_ICLR24 (+ C++ cpp_projection); their
behaviour follows SURVEY App. B.  All arithmetic runs in the hand-written kernels of csrc/tce_proj.cu; the
Python below only routes tensors (per-episode scalars stay on the device, no host synchronisation).
"""
from __future__ import annotations

import math

import torch

from .. import ops, util


# (the covariance chain deliberately runs forward and backward on a side stream, see _call_overlapped; torch's
# accumulate-grad stream-mismatch warning is switched off only inside the agent's update scope: rl/agent.py)


def _expand_first(t, batch):
    """Broadcast ONE factor [1, n, n] over the batch (stride 0) and remember the original: ``_first`` then hands it
    back without a slice node (the backward of ``expanded[:1]`` materialises and reduces a [B, n, n] gradient,
    and -- worse -- queues on the main stream behind the covariance chain, see DESIGN.md section 4)."""
    e = t.expand(batch, -1, -1)
    e._tce_first = t
    return e


def _first(L):
    base = getattr(L, "_tce_first", None)
    return base if base is not None else L[:1]


def _shared(policy, L):
    """A non-contextual policy carries ONE covariance (every batch entry equal): evaluate the covariance
    terms once and broadcast, as the KL layer of the reference does for the projection itself."""
    return not policy.contextual_std and L.dim() == 3 and L.shape[0] > 1


_HELPER_STREAMS = {}


def _helper_stream(device):
    """One helper stream PER PARENT stream: the trust-region branch and the logging branch both fork their mean part
    off; on a shared helper the (critical) mean gradient of the first would queue behind logging kernels."""
    key = (str(device), torch.cuda.current_stream(device).cuda_stream)
    if key not in _HELPER_STREAMS:
        _HELPER_STREAMS[key] = torch.cuda.Stream(device=device)
    return _HELPER_STREAMS[key]


def _maha(policy, mean, mean_o, L_o, linv=None):
    """|L_o^-1 (mean - mean_o)|^2 [B] fp64.  Diagonal factors: elementwise.  One shared covariance (non-contextual
    policy): invert the factor once (``linv``: an inverse already formed in this epoch, see ``shared_inverse``) and use
    matrix-vector products per episode instead of two triangular solves."""
    if policy.is_diag:
        return ops.gauss_maha_diag(mean, mean_o, L_o)
    if not (_shared(policy, L_o) and L_o.is_cuda):
        return ops.gauss_maha(mean, mean_o, L_o)
    return ops.gauss_maha_shared(mean, mean_o, linv if linv is not None else shared_inverse(L_o))


def shared_inverse(L_o):
    """fp64 inverse [n, n] of the ONE factor behind a broadcast covariance (not differentiable)."""
    return ops.tri_inverse(_first(L_o).detach().contiguous())[0]


def _factor_stats(policy, L, L_o):
    """gauss_stats of the covariance factors only (zero mean difference) [Bc, 5]."""
    if policy.is_diag:
        return ops.gauss_stats_diag(None, L, None, L_o)
    zeros = torch.zeros(L.shape[0], L.shape[-1], device=L.device)
    return ops.gauss_stats(zeros, L.contiguous(), zeros, L_o)


def _cov_stats(policy, L, L_o):
    """gauss_stats on the covariance factors only (zero mean difference), broadcast when shared."""
    B = L.shape[0]
    if _shared(policy, L):
        L, L_o = _first(L), _first(L_o)
    st = _factor_stats(policy, L, L_o)
    return st.expand(B, -1) if st.shape[0] != B else st


def gaussian_kl_details(policy, p, q, mean_part=None, q_linv=None):
    """(mean, cov, shape, volume) parts of KL(p || q), each [B] fp64, cov = shape + volume
    (gaussian_kl_details of the fork, used for logging at temporal_correlated_agent.py:641-686).
    ``mean_part`` may carry an already computed 1/2 maha (avoids a second batch-sized launch), ``q_linv`` the
    inverse factor of a shared q covariance formed earlier in the epoch (``shared_inverse``)."""
    helper = None
    if mean_part is None and p[0].is_cuda and _shared(policy, q[1]):
        # shared covariance: the mean part (factor inverse + batch kernel) and the covariance part (one
        # latency-bound CTA) are independent chains -- fork the first onto a helper stream
        cur, helper = torch.cuda.current_stream(), _helper_stream(p[0].device)
        helper.wait_stream(cur)
        with torch.cuda.stream(helper):
            mean_part = 0.5 * _maha(policy, p[0], q[0], q[1], linv=q_linv)
            mean_part.record_stream(cur)
    st = _cov_stats(policy, p[1], q[1])
    k = p[0].shape[-1]
    shape, volume = 0.5 * (st[:, 1] - k), 0.5 * (st[:, 3] - st[:, 2])
    if helper is not None:
        torch.cuda.current_stream().wait_stream(helper)
    if mean_part is None:
        mean_part = 0.5 * _maha(policy, p[0], q[0], q[1], linv=q_linv)
    return mean_part, shape + volume, shape, volume


def gaussian_kl(policy, p, q):
    """(mean part, covariance part) of KL(p || q), each [B] fp64 (projection_utils.gaussian_kl)."""
    mean_part, cov_part, _, _ = gaussian_kl_details(policy, p, q)
    return mean_part, cov_part


_KL_LOSS_CONST = {}


def _kl_loss_consts(B, coeff, with_cov, dev):
    """Cached constant gradients of the shared-covariance KL trust-region loss: (w [1,5], d loss / d maha [B],
    d loss / d stats [1,5])."""
    key = (B, coeff, with_cov, str(dev))
    if key not in _KL_LOSS_CONST:
        w = torch.tensor([[0.0, 0.5, -0.5, 0.5, 0.0]], dtype=torch.float64, device=dev)
        _KL_LOSS_CONST[key] = (w, torch.full((B,), 0.5 * coeff / B, dtype=torch.float64, device=dev),
                               w * (coeff if with_cov else 0.0))
    return _KL_LOSS_CONST[key]


class _SharedKLLoss(torch.autograd.Function):
    """loss = coeff * (mean_b 1/2 maha_b + [with_cov] (shape + volume)),  shape = 1/2 (tr - k),
    volume = 1/2 (logdet_q - logdet_p), from maha [B] and the five scalars st [1, 5] of ``gauss_stats``.
    Also returns the detached per-term values for the logging branch."""

    @staticmethod
    def forward(ctx, maha, st, coeff, with_cov, k, out_dtype):
        B, dev = maha.shape[0], maha.device
        w, ctx.g_maha, ctx.g_st = _kl_loss_consts(B, coeff, with_cov, dev)
        mean_diff = 0.5 * maha
        shape, volume = 0.5 * (st[:, 1] - k), 0.5 * (st[:, 3] - st[:, 2])
        cov_diff = shape + volume
        loss = mean_diff.mean() + cov_diff[0] if with_cov else mean_diff.mean()
        ctx.mark_non_differentiable(mean_diff, cov_diff, shape, volume)
        return (loss * coeff).to(out_dtype), mean_diff, cov_diff, shape, volume

    @staticmethod
    def backward(ctx, g, *_unused):
        if g is ops.unit_seed(g.device, g.dtype):                          # the usual case: no kernel at all
            return ctx.g_maha, ctx.g_st, None, None, None, None
        g = g.to(torch.float64)
        return ctx.g_maha * g, ctx.g_st * g, None, None, None, None


class _FoldedKLLoss(torch.autograd.Function):
    """loss = coeff * (mean_b 1/2 maha_b + [with_cov] (shape + volume)) with shape / volume read from the KL state
    scalars [1, 10] (slots 7, 8; constants for autograd: their gradient is applied by the projection's backward)."""

    @staticmethod
    def forward(ctx, maha, sc, coeff, with_cov, out_dtype):
        B = maha.shape[0]
        _, ctx.g_maha, _ = _kl_loss_consts(B, coeff, with_cov, maha.device)
        mean_diff = 0.5 * maha
        shape, volume = sc[:, 7].expand(B), sc[:, 8].expand(B)       # [1] (shared covariance) or [B] (per episode)
        cov_diff = shape + volume
        loss = mean_diff.mean() + cov_diff.mean() if with_cov else mean_diff.mean()
        ctx.mark_non_differentiable(mean_diff, cov_diff, shape, volume)
        return (loss * coeff).to(out_dtype), mean_diff, cov_diff, shape, volume

    @staticmethod
    def backward(ctx, g, *_unused):
        if g is ops.unit_seed(g.device, g.dtype):
            return ctx.g_maha, None, None, None, None
        raise RuntimeError("a folded trust-region loss must be back-propagated with the unit seed "
                           "(ops.unit_seed): its covariance gradient was added to the projection's backward")


def _entropy_schedule(kind, total_train_steps, dim):
    if kind == "linear":
        return lambda init, target, temp, step: step * (target * dim - init) / total_train_steps + init
    if kind == "exp":
        return lambda init, target, temp, step: dim * target + (init - dim * target) * temp ** (
            10 * step / total_train_steps)
    return None


class BaseProjectionLayer:
    def __init__(self, proj_type="", mean_bound=0.03, cov_bound=1e-3, trust_region_coeff=0.0, scale_prec=True,
                 entropy_schedule=None, action_dim=None, total_train_steps=None, target_entropy=0.0,
                 temperature=0.5, entropy_eq=False, entropy_first=False, do_regression=False, cpu=False,
                 dtype=torch.float32, **kwargs):
        if cpu:
            raise NotImplementedError("tce_rl_b200 projections run on the GPU only (no CPU path)")
        if do_regression:
            raise NotImplementedError("do_regression is false in every TCE config and is not built")
        self.proj_type = proj_type
        self.mean_bound, self.cov_bound = float(mean_bound), float(cov_bound)
        self.trust_region_coeff = trust_region_coeff
        self.scale_prec = bool(scale_prec)
        assert (action_dim and total_train_steps) if entropy_schedule else True
        self.entropy_eq, self.entropy_first = bool(entropy_eq), bool(entropy_first)
        self.entropy_schedule = _entropy_schedule(entropy_schedule, total_train_steps, action_dim)
        self.target_entropy, self.temperature = float(target_entropy), temperature
        self._initial_entropy = None
        # detached by-products of the last projection / trust-region-loss call, reused by the agent's logging
        # (temporal_correlated_agent.py:641-686 recomputes them): {"new_old_mean": [B], "new_proj": 4 x [B]}
        self.cache = {}
        self.overlap = bool(kwargs.get("overlap", True))      # run independent chains on a side stream
        self._side = None
        self._beta_cache = None

    @property
    def initial_entropy(self):
        return self._initial_entropy

    @initial_entropy.setter
    def initial_entropy(self, entropy):
        if self._initial_entropy is None:                     # write once
            self._initial_entropy = entropy

    # ---- pieces ---------------------------------------------------------------------------------------
    def _entropy_bound(self, step, device):
        if self.entropy_schedule is None:
            return None                                        # bound -inf: the projection is the identity
        key = (step, str(device), id(self._initial_entropy))
        if self._beta_cache is None or self._beta_cache[0] != key:     # constant over the epochs of one update:
            beta = self.entropy_schedule(self.initial_entropy, self.target_entropy, self.temperature, step)
            self._beta_cache = (key, torch.as_tensor(beta, device=device).to(torch.float64).reshape(1))
        return self._beta_cache[1]                                     # five tiny kernels once, not per epoch

    def _entropy_projection(self, policy, p, beta):
        if beta is None:
            return p
        mean, L = p
        shared = L.dim() == 3 and L.stride(0) == 0
        L_in = _first(L) if shared else L
        out, _ = ops.proj_entropy(L_in.contiguous(), beta, self.entropy_eq)
        return mean, (_expand_first(out, mean.shape[0]) if shared else out)

    projects = False        # the base layer only applies the entropy control (its trust-region step is the identity)

    def _mean_part(self, policy, p, q):
        raise NotImplementedError

    def _cov_projection(self, policy, L, L_old):
        return L

    def _cov_projection_with_entropy(self, policy, L, L_old, beta):
        """Covariance projection and entropy control as one op, or None if the layer has no fused kernel."""
        return None

    def _shared_sigma(self, proj_L1):
        return None

    def _trust_region_projection(self, policy, p, q):
        if not self.projects:
            return p
        mean, L = p
        old_mean, old_L = q
        mean_part = self._mean_part(policy, p, q)
        self.cache = {"new_old_mean": mean_part.detach()}
        proj_mean = ops.proj_mean(mean, old_mean, mean_part, self.mean_bound)
        if not policy.contextual_std:                          # one shared covariance: project the first only
            proj_L = _expand_first(self._cov_projection(policy, _first(L), _first(old_L)), mean.shape[0])
        else:
            proj_L = self._cov_projection(policy, L, old_L)
        return proj_mean, proj_L

    def _trust_region_projection_with_entropy(self, policy, p, q, beta):
        """Trust-region step + entropy control as fused kernels, or None (then the two steps run separately)."""
        return None

    def _side_stream(self, device):
        if self._side is None:
            self._side = torch.cuda.Stream(device=device, priority=-1)     # the covariance chain is the critical path
        return self._side

    def _overlappable(self, policy, L):
        return (self.projects and self.overlap and not policy.contextual_std and not self.entropy_first
                and L.is_cuda)

    def __call__(self, policy, p, q, step, *args, cov_projected=None, defer_factor=False, **kwargs):
        """``defer_factor``: return as soon as the covariance ITSELF (``_tce_sigma``) is available; the caller then
        calls ``join_covariance`` on every stream that reads the projected factor."""
        if self._overlappable(policy, p[1]):
            return self._call_overlapped(policy, p, q, step, cov_projected, defer_factor)
        beta = self._entropy_bound(step, p[0].device)
        if self.entropy_first:
            p = self._entropy_projection(policy, p, beta)
        elif beta is not None:
            fused = self._trust_region_projection_with_entropy(policy, p, q, beta)
            if fused is not None:
                return fused
        proj = self._trust_region_projection(policy, p, q)
        return proj if self.entropy_first else self._entropy_projection(policy, proj, beta)

    def start_cov_projection(self, policy, L, old_L, step):
        """Non-contextual covariance: the covariance chain (ONE matrix: projection + entropy scaling, a
        latency-bound single-CTA sequence) depends neither on the observations nor on the mean net, so it can
        be started on a side stream (a parallel branch when captured in a CUDA graph) BEFORE the mean net is
        evaluated; pass the returned handle to ``__call__(..., cov_projected=handle)``.  Calling it first also
        fixes the order of the backward: autograd runs nodes in reverse creation order, so the mean-net
        backward is queued on the main stream before the (long) covariance backward is joined into it.
        Returns None when the layer would not overlap (contextual covariance, CPU tensors, ...)."""
        if not self._overlappable(policy, L):
            return None
        main = torch.cuda.current_stream()
        side = self._side_stream(L.device)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            beta = self._entropy_bound(step, L.device)
            fused = self._cov_projection_with_entropy(policy, _first(L), _first(old_L), beta) if beta is not None else None
            if fused is not None:                               # one kernel each way (KL layer)
                proj_L1 = fused
            else:
                proj_L1 = self._cov_projection(policy, _first(L), _first(old_L))
                if beta is not None:
                    proj_L1 = ops.proj_entropy(proj_L1.contiguous(), beta, self.entropy_eq)[0]
            proj_L1.record_stream(main)
            # broadcast here: the backward of the expand (a [B, n, n] -> [n, n] reduction) then runs on the side
            # stream in front of the covariance backward instead of delaying the mean chain on the main stream
            out = _expand_first(proj_L1, L.shape[0])
            if fused is not None:
                out._tce_sigma = self._shared_sigma(proj_L1)       # Sigma for the likelihood's stage 1 (or None)
            return out

    def _call_overlapped(self, policy, p, q, step, cov_projected=None, defer_factor=False):
        mean, L = p
        old_mean, old_L = q
        proj_L = cov_projected if cov_projected is not None else self.start_cov_projection(policy, L, old_L, step)
        mean_part = self._mean_part(policy, p, q)
        self.cache = {"new_old_mean": mean_part.detach()}
        proj_mean = ops.proj_mean(mean, old_mean, mean_part, self.mean_bound)
        sig = getattr(proj_L, "_tce_sigma", None)
        if defer_factor and sig is not None and sig[2] is not None:
            # the likelihood's first stage only needs Sigma: wait for the first half of the covariance forward; whoever
            # reads the FACTOR on another stream joins the covariance stream first (`join_covariance`)
            torch.cuda.current_stream().wait_event(sig[2])
            self._cov_pending = True
        else:
            torch.cuda.current_stream().wait_stream(self._side_stream(mean.device))
            self._cov_pending = False
        return proj_mean, proj_L

    _cov_pending = False

    def join_covariance(self, stream=None):
        """Order ``stream`` (default: the current one) after the covariance chain of the last ``__call__`` (needed
        before the projected FACTOR is read when the call returned after the Sigma half of a split forward)."""
        if self._side is not None:
            (stream or torch.cuda.current_stream()).wait_stream(self._side)

    def trust_region_value(self, policy, p, q):
        return gaussian_kl(policy, p, q)

    def _with_cov(self, policy, set_variance):
        return policy.contextual_std or (set_variance is not None and not set_variance)

    def get_trust_region_loss(self, policy, p, proj_p, set_variance=None, fold=False):
        """coeff * mean(mean_diff [+ cov_diff]) between p and the DETACHED projection (SURVEY App. B.5).
        ``fold`` (KL layer, one shared covariance, ``proj_p`` = the output of the last projection of ``p``): the
        covariance term is taken in closed form from the projection's eigen-system and its GRADIENT is added inside
        the projection's own backward kernel; valid when the loss is back-propagated exactly once with unit weight
        together with that projection (TemporalCorrelatedAgent.policy_epoch does) -- otherwise leave it False."""
        target = (proj_p[0].detach(), proj_p[1].detach())
        kl_metric = type(self).trust_region_value is BaseProjectionLayer.trust_region_value
        if kl_metric and fold and p[0].is_cuda and not _shared(policy, p[1]) and self._can_fold(p, proj_p):
            return self._folded_kl_trust_region_loss(policy, p, target, set_variance)
        if kl_metric and p[0].is_cuda and _shared(policy, p[1]):
            if fold and self._can_fold(p, proj_p):
                return self._folded_kl_trust_region_loss(policy, p, target, set_variance)
            return self._shared_kl_trust_region_loss(policy, p, target, set_variance)
        if kl_metric:      # KL metric
            mean_diff, cov_diff, shape, volume = gaussian_kl_details(policy, p, target)
            self.cache["new_proj"] = tuple(x.detach() for x in (mean_diff, cov_diff, shape, volume))
        else:
            mean_diff, cov_diff = self.trust_region_value(policy, p, target)
        loss = (mean_diff + cov_diff if self._with_cov(policy, set_variance) else mean_diff).mean()
        return (loss * self.trust_region_coeff).to(p[0].dtype)

    def _can_fold(self, p, proj_p):
        return False

    def _shared_kl_trust_region_loss(self, policy, p, target, set_variance):
        """KL metric, ONE covariance for the batch: same value as the generic path, but the loss arithmetic is one
        autograd node (``_SharedKLLoss``) whose backward hands out cached constant gradients -- the generic
        formulation costs ~12 small launches each way, and in the backward they sit between the loss seed and
        the single-CTA covariance kernel / the mean gradient the mean net is waiting for."""
        cur, helper = torch.cuda.current_stream(), _helper_stream(p[0].device)
        helper.wait_stream(cur)
        with torch.cuda.stream(helper):                                    # mean part beside the covariance part
            linv = None
            if not policy.is_diag:
                linv = shared_inverse(target[1])
                ready = torch.cuda.Event()
                ready.record()
                # the KL layer's backward needs the inverse of exactly this factor (its own output): hand it over
                self._output_inverse = (linv, ready, _first(target[1]).data_ptr())
            maha = _maha(policy, p[0], target[0], target[1], linv=linv)
            maha.record_stream(cur)
        with_cov = self._with_cov(policy, set_variance)
        st = _factor_stats(policy, _first(p[1]), _first(target[1]))      # [1, 5]
        cur.wait_stream(helper)
        loss, mean_diff, cov_diff, shape, volume = _SharedKLLoss.apply(
            maha, st, float(self.trust_region_coeff), bool(with_cov), int(p[0].shape[-1]), p[0].dtype)
        self.cache["new_proj"] = (mean_diff, cov_diff, shape, volume)
        return loss

    def compute_metrics(self, policy, p, q, step=None):
        with torch.no_grad():
            ent, ent_q = policy.entropy(p), policy.entropy(q)
            mean_kl, cov_kl = gaussian_kl(policy, p, q)
            mean_diff, cov_diff = self.trust_region_value(policy, p, q)
            kl, con = mean_kl + cov_kl, mean_diff + cov_diff
            return {"kl": kl.mean(), "constraint": con.mean(), "mean_constraint": mean_diff.mean(),
                    "cov_constraint": cov_diff.mean(), "entropy": ent.mean(), "entropy_diff": (ent_q - ent).mean(),
                    "kl_max": kl.max(), "constraint_max": con.max(), "mean_constraint_max": mean_diff.max(),
                    "cov_constraint_max": cov_diff.max(), "entropy_max": ent.max()}


class KLProjectionLayer(BaseProjectionLayer):
    projects = True
    __doc__ = """KL projection.  ``warm_start`` (default on): the eigen-basis found by the previous call is handed to the
    next one; the kernel uses it only when the old covariance is bit-identical (fingerprint), i.e. across the
    epochs of one ``update_policy`` -- results are unchanged, the Jacobi solve needs 2-3 sweeps instead of ~9."""

    def __init__(self, *args, warm_start=True, **kwargs):
        super().__init__(*args, **kwargs)
        self.warm_start = bool(warm_start)
        self._kl_state = None

    fuse_entropy = True      # KL projection + entropy control in one launch (start_cov_projection)
    sigma_to_likelihood = True   # hand Sigma (already formed inside the projection kernel) to the likelihood
    # Forward in two launches (Sigma / Cholesky) so that the likelihood's stage 1 starts ~20 us earlier.  Measured
    # at B = 1024: no net gain -- the trust-region branch, which needs the factor, then collides with stage 3 of the
    # likelihood instead of stage 1 (profiles/README.md) -- so it is off by default.
    split_forward = True     # (round 2: the uniform-grid likelihood leaves most SMs free, the collision is gone, and the
    #                          gradient returns in covariance space, so nothing on the critical path needs the factor)

    def _shared_sigma(self, proj_L1):
        """(Sigma0 [n, n] fp64, alpha^2 [1]) views of the state written by the fused kernel: the covariance of the
        layer's output is alpha^2 * Sigma0.  Valid until the next forward of this layer."""
        state = getattr(self, "_last_state", None)
        sig = getattr(self, "_last_sigma", None)
        if not self.sigma_to_likelihood or state is None or sig is None or proj_L1.shape[0] != 1:
            return None
        # sig[0]: Sigma0 [1, n, n] fp64, a DIFFERENTIABLE output of the projection op (gradient in covariance space)
        return sig[0], sig[1], (ops.SIGMA_READY.get(id(state)) if self.split_forward else None)

    def _state_for(self, Lc):
        state = self._kl_state
        if (not self.warm_start or state is None or state.device != Lc.device
                or state.numel() != ops.kl_state_size(Lc.shape[0], Lc.shape[-1])):
            state = ops.kl_state(Lc.shape[0], Lc.shape[-1], Lc.device)
            if self.warm_start:
                self._kl_state = state
        return state

    def _can_fold(self, p, proj_p):
        last = getattr(self, "_last_call", None)
        if last is None:
            return False
        if last.get("per_episode"):
            return p[1] is last["L_in"] and proj_p[1] is last["out"]
        return last["out_inv"] is not None and _first(p[1]) is last["L_in"] and _first(proj_p[1]) is last["out"]

    def _trust_region_projection_with_entropy(self, policy, p, q, beta):
        """Per-episode covariance factors (contextual policy): KL projection + entropy control of all B matrices in ONE
        kernel each way (instead of projection + entropy-scaling kernels), and the eigen-system of every matrix stays
        in the state: the covariance terms of the trust-region loss and of the logging decomposition are closed forms
        of it (``cache``: no gauss_stats launches), the trust-region covariance gradient is added inside the backward
        kernel (``get_trust_region_loss(fold=True)``)."""
        if not policy.contextual_std or not self.fuse_entropy or not p[1].is_cuda:
            return None
        mean, L = p
        old_mean, old_L = q
        mean_part = self._mean_part(policy, p, q)
        proj_mean = ops.proj_mean(mean, old_mean, mean_part, self.mean_bound)
        if policy.is_diag:
            self.cache = {"new_old_mean": mean_part.detach()}
            return proj_mean, self._diag_projection(L, old_L, beta)
        Lc = L.contiguous()
        state = self._state_for(Lc)
        self._last_state = state
        self._output_inverse = None
        out, _proj, _info, _sigma, _scale, _inv = ops.proj_kl_entropy(
            Lc, old_L.contiguous(), self.cov_bound, state, self.warm_start, beta, self.entropy_eq, False, self,
            return_sigma=True)
        sc = ops.kl_state_scalars(state, Lc.shape[0], Lc.shape[-1]).detach()
        self.cache = {"new_old_mean": mean_part.detach(),
                      "new_old_cov": (sc[:, 10] + sc[:, 11], sc[:, 10], sc[:, 11]),
                      "proj_old_cov": (sc[:, 12] + sc[:, 13], sc[:, 12], sc[:, 13])}
        self._last_call = dict(L_in=L, out=out, out_inv=None, state=state, per_episode=True)
        self._tr_fold = 0.0
        return proj_mean, out

    def _folded_kl_trust_region_loss(self, policy, p, target, set_variance):
        """Shared covariance, target = this layer's last output: Mahalanobis term with the inverse the forward's
        second launch already formed; covariance term = two scalars of the state (closed form on the eigen-system),
        its gradient is added by the projection's backward kernel (``_tr_fold``)."""
        last = self._last_call
        n = p[0].shape[-1]
        with_cov = self._with_cov(policy, set_variance)
        if last.get("per_episode"):                        # B matrices: mean term per episode, covariance terms from the state
            B = p[0].shape[0]
            maha = ops.gauss_maha(p[0], target[0], target[1])
            sc = ops.kl_state_scalars(last["state"], B, n)
            self._tr_fold = float(self.trust_region_coeff) / B if with_cov else 0.0     # loss = mean over the B matrices
        else:
            linv = last["out_inv"][0]
            self._output_inverse = None
            maha = _maha(policy, p[0], target[0], target[1], linv=linv)
            sc = ops.kl_state_scalars(last["state"], 1, n)
            self._tr_fold = float(self.trust_region_coeff) if with_cov else 0.0
        loss, mean_diff, cov_diff, shape, volume = _FoldedKLLoss.apply(
            maha, sc, float(self.trust_region_coeff), bool(with_cov), p[0].dtype)
        self.cache["new_proj"] = (mean_diff, cov_diff, shape, volume)
        return loss

    def _mean_part(self, policy, p, q):
        linv = shared_inverse(q[1]) if (_shared(policy, q[1]) and q[1].is_cuda and not policy.is_diag) else None
        self._old_linv = linv                                   # reused by the logging branch of the same epoch
        return 0.5 * _maha(policy, p[0], q[0], q[1], linv=linv)

    def _diag_projection(self, L, L_old, beta):
        """Diagonal factors (std_only policy): closed-form projection [+ entropy control], one warp per matrix.  No
        eigen-system is kept, so nothing can be folded into its backward and no Sigma is handed to the likelihood."""
        self._last_state = self._last_call = None
        return ops.proj_kl_diag(L, L_old, self.cov_bound, beta, self.entropy_eq)[0]

    def _cov_projection(self, policy, L, L_old):
        if policy.is_diag:
            return self._diag_projection(L, L_old, None)
        Lc = L.contiguous()
        state = self._state_for(Lc)
        return ops.proj_kl_cov(Lc, L_old.contiguous(), self.cov_bound, state, self.warm_start, self)[0]

    def _cov_projection_with_entropy(self, policy, L, L_old, beta):
        if not self.fuse_entropy:
            return None
        if policy.is_diag:
            return self._diag_projection(L, L_old, beta)
        Lc = L.contiguous()
        state = self._state_for(Lc)
        self._last_state = state
        self._output_inverse = None            # only an inverse formed AFTER this forward can belong to it
        split = bool(self.split_forward and self.sigma_to_likelihood and Lc.shape[0] == 1)
        out, _proj, _info, sigma, scale, out_inv = ops.proj_kl_entropy(
            Lc, L_old.contiguous(), self.cov_bound, state, self.warm_start, beta, self.entropy_eq, split, self,
            return_sigma=True)
        self._last_sigma = (sigma, scale)
        # what a folded trust-region loss (get_trust_region_loss(..., fold=True)) needs from THIS forward
        self._last_call = dict(L_in=L, out=out, out_inv=out_inv if split else None, state=state)
        self._tr_fold = 0.0
        return out


class FrobeniusProjectionLayer(BaseProjectionLayer):
    projects = True

    def _mean_dist(self, policy, p, q):
        if self.scale_prec:
            return ops.gauss_maha_diag(p[0], q[0], q[1]) if policy.is_diag else ops.gauss_maha(p[0], q[0], q[1])
        return ((q[0] - p[0]) ** 2).sum(-1).to(torch.float64)

    def _mean_part(self, policy, p, q):
        return self._mean_dist(policy, p, q)

    def _cov_projection(self, policy, L, L_old):
        if policy.is_diag:
            return ops.proj_frob_diag(L, L_old, self.cov_bound)[0]
        return ops.proj_frob_cov(L.contiguous(), L_old, self.cov_bound)[0]

    def _cov_dist(self, policy, kind, L, L_o, scale_prec):
        """Covariance distance [B]; a shared (non-contextual) covariance is evaluated once and broadcast."""
        B = L.shape[0]
        if _shared(policy, L):
            L, L_o = _first(L), _first(L_o)
        if policy.is_diag:
            val = ops.cov_distance_diag(kind, L, L_o, scale_prec)
        else:
            val = ops.cov_distance(kind, L.contiguous(), L_o, scale_prec)
        return val.expand(B) if val.shape[0] != B else val

    def trust_region_value(self, policy, p, q):
        return self._mean_dist(policy, p, q), self._cov_dist(policy, 0, p[1], q[1], False)

    def get_trust_region_loss(self, policy, p, proj_p, set_variance=None):
        target = (proj_p[0].detach(), proj_p[1].detach())
        diff = self._mean_dist(policy, p, target)
        if self._with_cov(policy, set_variance):               # squared L difference instead of the Frobenius metric
            Lp, Lt = (_first(p[1]), _first(target[1])) if _shared(policy, p[1]) else (p[1], target[1])
            if policy.is_diag:                                 # (zero off the diagonal)
                Lp, Lt = Lp.diagonal(dim1=-2, dim2=-1), Lt.diagonal(dim1=-2, dim2=-1)
                diff = diff + (Lp - Lt).pow(2).sum(-1).to(torch.float64)
            else:
                diff = diff + (Lp - Lt).pow(2).sum([-1, -2]).to(torch.float64)
        return (diff.mean() * self.trust_region_coeff).to(p[0].dtype)


class WassersteinProjectionLayer(FrobeniusProjectionLayer):
    def _cov_projection(self, policy, L, L_old):
        if policy.is_diag:
            return ops.proj_w2_diag(L, L_old, self.cov_bound, self.scale_prec)[0]
        return ops.proj_w2_cov(L.contiguous(), L_old, self.cov_bound, self.scale_prec)[0]

    def trust_region_value(self, policy, p, q):
        return self._mean_dist(policy, p, q), self._cov_dist(policy, 1, p[1], q[1], self.scale_prec)

    def get_trust_region_loss(self, policy, p, proj_p, set_variance=None):
        return BaseProjectionLayer.get_trust_region_loss(self, policy, p, proj_p, set_variance)


def projection_factory(typ: str, **kwargs):
    """mprl/rl/projection/__init__.py:19-40 (device -> ``cpu`` flag, dtype parsing)."""
    kwargs = dict(kwargs)
    dtype, device = util.parse_dtype_device(kwargs.get("dtype", "float32"), kwargs.pop("device", "cuda"))
    kwargs["cpu"] = device == torch.device("cpu")
    kwargs["dtype"] = dtype
    layers = {"BaseProjectionLayer": BaseProjectionLayer, "KLProjectionLayer": KLProjectionLayer,
              "FrobeniusProjectionLayer": FrobeniusProjectionLayer,
              "WassersteinProjectionLayer": WassersteinProjectionLayer}
    if typ not in layers:
        raise NotImplementedError(f"{typ} is not on the TCE policy-update path (SURVEY section 2, row 7)")
    return layers[typ](**kwargs)

"""Oracle of the KL covariance projection for diagonal factors (``policy.is_diag``, std_only policies).

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__``).  The dense restatement in ``oracle.projection`` goes through an
eigen-decomposition of N = W^T W; for diagonal factors N = diag(lam), lam = (sigma_old / sigma)^2, and a fresh std_only
policy has all sigma equal, i.e. repeated eigenvalues, where ``eigh`` has no usable gradient.  Here the projection is
the elementwise closed form of the same dual: sigma_proj^2 = (1 + eta) / (1 / sigma^2 + eta / sigma_old^2), with eta
from ``kl_cov_solve_eta`` on lam and the same one-Newton-step implicit re-attachment.  Everything else (the other
layers, the distances, the entropy control) is ``oracle.projection`` unchanged.
"""
from __future__ import annotations

import torch

from . import projection as op


def kl_cov_projection_diag(chol, chol_old, eps_cov):
    """Sigma_proj [B,k,k] (diagonal) and active mask of diagonal factors, differentiable w.r.t. ``chol``."""
    sig = chol.diagonal(dim1=-2, dim2=-1)
    sig_o = chol_old.diagonal(dim1=-2, dim2=-1)
    lam = (sig_o / sig) ** 2
    zero = torch.zeros(lam.shape[:-1], dtype=lam.dtype)
    kl0 = op.kl_cov_eta_function(lam, zero)
    active = kl0 > eps_cov
    eta = torch.zeros_like(kl0)
    if active.any():
        eta_star = op.kl_cov_solve_eta(lam, eps_cov)
        # one differentiable Newton step re-attaches the implicit gradient d eta*/d lam
        e = eta_star.clone().requires_grad_(True)
        with torch.enable_grad():
            f = op.kl_cov_eta_function(lam.detach(), e)
            dfde, = torch.autograd.grad(f.sum(), e)
        eta_impl = eta_star - (op.kl_cov_eta_function(lam, eta_star) - eps_cov) / dfde.detach()
        eta = torch.where(active, eta_impl, eta)
    eta = eta[..., None]
    var = torch.where(active[..., None], (1 + eta) / (1 / sig ** 2 + eta / sig_o ** 2), sig ** 2)
    return torch.diag_embed(var), active


class KLProjectionLayer(op.KLProjectionLayer):
    """``oracle.projection.KLProjectionLayer`` with the diagonal branch for ``policy.is_diag``."""

    def _trust_region_projection(self, policy, p, q, eps, eps_cov, **kwargs):
        if not policy.is_diag:
            return super()._trust_region_projection(policy, p, q, eps, eps_cov, **kwargs)
        mean, chol = p
        old_mean, old_chol = q
        mean_part, _ = op.gaussian_kl(policy, p, q)
        proj_mean = op.mean_projection(mean, old_mean, mean_part, eps)
        if not policy.contextual_std:              # one shared covariance: project the first only
            chol, old_chol = chol[:1], old_chol[:1]
        cov_proj, _ = kl_cov_projection_diag(chol, old_chol, eps_cov)
        proj_chol = torch.diag_embed(cov_proj.diagonal(dim1=-2, dim2=-1).sqrt())
        if not policy.contextual_std:
            proj_chol = proj_chol.expand(mean.shape[0], -1, -1)
        return proj_mean, proj_chol


def projection_factory(typ: str, **kwargs):
    """``oracle.projection.projection_factory`` with the KL layer above."""
    if typ != "KLProjectionLayer":
        return op.projection_factory(typ, **kwargs)
    kwargs = dict(kwargs)
    dtype = kwargs.get("dtype", torch.float32)
    kwargs["dtype"] = getattr(torch, dtype.replace("torch.", "")) if isinstance(dtype, str) else dtype
    kwargs["cpu"] = True
    kwargs.pop("device", None)
    return KLProjectionLayer(**kwargs)

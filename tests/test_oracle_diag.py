"""The diagonal KL covariance projection of the oracle (``oracle.projection_diag``, std_only policies): agrees with the
dense projection where that one is well posed, meets the bound, solves the dual and has usable gradients where the
dense one (eigh on repeated eigenvalues) does not.  CPU only."""
import torch
from scipy.optimize import minimize_scalar

from oracle import projection as op
from oracle import projection_diag as opd
from oracle.policy import BlackBoxPolicy

F64 = torch.float64


def diag_factors(B, n, seed, spread=0.3):
    g = torch.Generator().manual_seed(seed)
    s = torch.exp(spread * torch.randn(B, n, generator=g, dtype=F64))
    s_old = torch.exp(spread * torch.randn(B, n, generator=g, dtype=F64))
    return torch.diag_embed(s), torch.diag_embed(s_old)


def kl_cov(cov, L_old):
    """KL_cov(N(cov) || N(L_old L_old^T)) in closed form for diagonal matrices."""
    v, vo = cov.diagonal(dim1=-2, dim2=-1), (L_old.diagonal(dim1=-2, dim2=-1)) ** 2
    return 0.5 * (v / vo - 1 + torch.log(vo / v)).sum(-1)


def test_equals_dense_projection_on_distinct_eigenvalues():
    L, L_old = diag_factors(6, 63, 0)
    eps = 5e-4
    dense, act_d = op.kl_cov_projection(L, L_old, eps)
    diag, act = opd.kl_cov_projection_diag(L, L_old, eps)
    assert act.all() and torch.equal(act, act_d)
    assert (diag - dense).abs().max().item() <= 1e-12 * dense.abs().max().item()
    off = diag - torch.diag_embed(diag.diagonal(dim1=-2, dim2=-1))
    assert off.abs().max().item() == 0.0


def test_bound_where_active_identity_where_inactive():
    L, L_old = diag_factors(8, 14, 1)
    L = L.clone()
    L[:3] = L_old[:3] * 1.001                              # close to the old policy: inactive
    eps = 5e-4
    cov, act = opd.kl_cov_projection_diag(L, L_old, eps)
    assert not act[:3].any() and act[3:].all()
    assert torch.allclose(cov[:3], L[:3] @ L[:3].transpose(-1, -2), rtol=0, atol=1e-15)
    kl = kl_cov(cov[3:], L_old[3:])
    assert (kl - eps).abs().max().item() <= 1e-12


def test_eta_solves_the_dual():
    """The stationarity condition of the dual of the KL projection is KL_cov(eta) = eps: eta* minimises
    (KL_cov(eta) - eps)^2 on eta >= 0, found here independently by scipy's bounded scalar minimiser."""
    L, L_old = diag_factors(3, 21, 2)
    eps = 1e-3
    lam = (L_old.diagonal(dim1=-2, dim2=-1) / L.diagonal(dim1=-2, dim2=-1)) ** 2
    eta = op.kl_cov_solve_eta(lam, eps)
    for b in range(3):
        f = lambda e: float((op.kl_cov_eta_function(lam[b:b + 1], torch.tensor([e], dtype=F64)) - eps) ** 2)
        ref = minimize_scalar(f, bounds=(0.0, 10 * float(eta[b]) + 10.0), method="bounded",
                              options=dict(xatol=1e-12)).x
        assert abs(ref - float(eta[b])) <= 1e-5 * max(1.0, float(eta[b]))
    assert (op.kl_cov_eta_function(lam, eta) - eps).abs().max().item() <= 1e-12


def test_gradcheck_including_equal_sigma():
    eps = 5e-4
    L, L_old = diag_factors(2, 5, 3)
    Ls = [L, 0.9 * torch.eye(5, dtype=F64).expand(2, 5, 5).clone()]      # second: all-equal sigma (a fresh policy)
    olds = [L_old, torch.eye(5, dtype=F64).expand(2, 5, 5).clone()]
    for L0, Lo in zip(Ls, olds):
        s = L0.diagonal(dim1=-2, dim2=-1).clone().requires_grad_(True)
        fn = lambda x: opd.kl_cov_projection_diag(torch.diag_embed(x), Lo, eps)[0].diagonal(dim1=-2, dim2=-1)
        assert opd.kl_cov_projection_diag(torch.diag_embed(s), Lo, eps)[1].all()
        assert torch.autograd.gradcheck(fn, (s,), eps=1e-7, atol=1e-7, rtol=1e-5)
    # the dense projection has no usable gradient at equal sigma: that is why the diagonal branch exists
    s = (0.9 * torch.ones(1, 5, dtype=F64)).requires_grad_(True)
    dense, act = op.kl_cov_projection(torch.diag_embed(s), torch.eye(5, dtype=F64)[None], eps)
    assert act.all()
    g, = torch.autograd.grad(dense.diagonal(dim1=-2, dim2=-1).sum(), s)
    sd = s.detach().clone().requires_grad_(True)
    diag, _ = opd.kl_cov_projection_diag(torch.diag_embed(sd), torch.eye(5, dtype=F64)[None], eps)
    gd, = torch.autograd.grad(diag.diagonal(dim1=-2, dim2=-1).sum(), sd)
    assert torch.isfinite(gd).all() and not torch.isfinite(g).all()


def test_kl_layer_dispatches_on_is_diag():
    pol = BlackBoxPolicy(7, std_only=True, contextual=True)
    layer = opd.projection_factory("KLProjectionLayer", mean_bound=0.05, cov_bound=5e-4, dtype="float64")
    assert isinstance(layer, opd.KLProjectionLayer) and layer.dtype == torch.float64
    assert type(opd.projection_factory("FrobeniusProjectionLayer")) is op.FrobeniusProjectionLayer
    L, L_old = diag_factors(4, 7, 4)
    mean = torch.zeros(4, 7, dtype=F64)
    pm, pL = layer._trust_region_projection(pol, (mean, L), (mean, L_old), 0.05, 5e-4)
    assert torch.equal(pL, torch.diag_embed(pL.diagonal(dim1=-2, dim2=-1)))
    assert (kl_cov(pL @ pL.transpose(-1, -2), L_old) - 5e-4).abs().max().item() <= 1e-12

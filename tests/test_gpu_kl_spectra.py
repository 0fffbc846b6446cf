"""KL covariance projection on the spectra where an eigen-solver and a dual solve go wrong, at every Jacobi shape.

The generalised eigenvalues lam of N = W^T W, W = L~^-1 L_old, are placed on purpose: all equal (a fresh policy,
L~ = c L_old), tight clusters, several decades wide, a step barely inside / outside the bound, and eta far above the
first search grid.  The kernels (csrc/tce_proj.cu on csrc/tce_smem_la.cuh) are compared with an fp64 reference that
needs no eigenvectors (DESIGN §4):

    Sigma(eta) = (1 + eta) (Sigma~^-1 + eta Sigma_old^-1)^-1 = (1 + eta) L_old (N + eta I)^-1 L_old^T ,

built from Cholesky factorisations and triangular solves only, so its gradient is finite where eigenvalues repeat
(the oracle's goes through ``torch.linalg.eigh`` and has no usable value there).  The reference itself is checked on
the CPU against the oracle, a closed form and ``gradcheck``.
"""
import math

import pytest
import torch

from oracle import projection as oproj

if torch.cuda.is_available():
    from tce_rl_b200 import _lib, ops

F64 = torch.float64
LOG_2PI = 1.8378770664093453
EPS = 5e-4
NS = [1, 2, 3, 7, 28, 31, 32, 33, 36, 63, 64]
LAYOUTS = ["one_cta_per_matrix", "more_matrices_than_sms"]


# ---------------------------------------------------------------------------------------------------------------------
# fp64 reference
# ---------------------------------------------------------------------------------------------------------------------
def _tsolve(A, B):
    return torch.linalg.solve_triangular(A, B, upper=False)


def _logdiag(C):
    return torch.log(torch.diagonal(C, dim1=-2, dim2=-1)).sum(-1)


def kl_of_eta_lam(lam, eta):
    """KL_cov(eta) = 1/2 sum_i g(r_i), g(r) = 1/r - 1 + ln r, r_i = 1 + x_i, x_i = (lam_i - 1) / (1 + eta): written
    without the cancellation of 1/r - 1 against ln r near r = 1."""
    x = (lam - 1.0) / (1.0 + eta)[..., None]
    return 0.5 * (torch.log1p(x) - x / (1.0 + x)).sum(-1)


def solve_eta(lam, eps):
    """Root of KL_cov(eta) = eps (decreasing in eta): bracket by doubling, then bisect to the last bit."""
    lo = torch.zeros(lam.shape[:-1], dtype=F64)
    hi = torch.ones_like(lo)
    for _ in range(2000):
        big = kl_of_eta_lam(lam, hi) > eps
        if not bool(big.any()):
            break
        lo, hi = torch.where(big, hi, lo), torch.where(big, 2.0 * hi, hi)
    for _ in range(200):
        mid = 0.5 * (lo + hi)
        big = kl_of_eta_lam(lam, mid) > eps
        lo, hi = torch.where(big, mid, lo), torch.where(big, hi, mid)
    return 0.5 * (lo + hi)


def kl_of_eta_chol(N, eta):
    """KL(N(Sigma(eta)) || N(Sigma_old)) with K = chol(N + eta I):
    tr(Sigma_old^-1 Sigma) = (1 + eta) |K^-1|_F^2,
    logdet Sigma_old - logdet Sigma = logdet(N + eta I) - n ln(1 + eta)."""
    n = N.shape[-1]
    eye = torch.eye(n, dtype=F64)
    K = torch.linalg.cholesky(N + eta[..., None, None] * eye)
    Ki = _tsolve(K, eye.expand_as(K))
    return 0.5 * ((1.0 + eta) * (Ki * Ki).sum((-2, -1)) - n - n * torch.log1p(eta) + 2.0 * _logdiag(K))


def kl_of_sigma(S, Lo):
    """KL(N(S) || N(Lo Lo^T)), covariance part, from traces and logdets of Cholesky factors."""
    n = S.shape[-1]
    C = torch.linalg.cholesky(S)
    X = _tsolve(Lo, C)
    return 0.5 * ((X * X).sum((-2, -1)) - n + 2.0 * _logdiag(Lo) - 2.0 * _logdiag(C))


def kl_reference(Lt, Lo, eps, beta=None, equality=False):
    """The KL covariance projection of L~ = ``Lt`` against ``Lo`` ([B, n, n] fp64, lower), optionally followed by the
    entropy control (``beta`` [B]).  Differentiable w.r.t. ``Lt``: eta* is re-attached by one implicit Newton step
    with a detached derivative (as ``oracle.projection.kl_cov_projection`` does) on the Cholesky form of KL(eta).
    ``eps``: a float or [B].  -> dict of eta, active, kl0, sigma (Sigma_proj), proj (its factor), alpha, ent, out and
    ``scalars`` [B, 16] laid out as ``ops.kl_state_scalars`` documents (slot 3, the fingerprint, and 14/15 are NaN)."""
    B, n = Lt.shape[0], Lt.shape[-1]
    eps_t = torch.as_tensor(eps, dtype=F64).expand(B)
    ld_old = 2.0 * _logdiag(Lo)
    W = _tsolve(Lt, Lo)
    N = W.transpose(-1, -2) @ W
    X = _tsolve(Lo, Lt)                                                   # tr(Sigma_old^-1 Sigma~) = |Lo^-1 L~|_F^2
    ld_in = 2.0 * _logdiag(Lt)
    kl0 = 0.5 * ((X * X).sum((-2, -1)) - n + ld_old - ld_in)
    active = kl0.detach() > eps_t
    lam = torch.linalg.eigvalsh(N.detach())                              # eigenvalues only: the root, never autograd
    eta_star = torch.where(active, solve_eta(lam, eps_t), torch.zeros_like(eps_t))
    dfde = -0.5 * ((lam - 1.0) ** 2 / ((1.0 + eta_star)[:, None] * (lam + eta_star[:, None]) ** 2)).sum(-1)
    dfde = torch.where(active, dfde, -torch.ones_like(dfde))
    eta_impl = eta_star - (kl_of_eta_chol(N, eta_star) - eps_t) / dfde
    eta = torch.where(active, eta_impl, torch.zeros_like(eta_impl))
    K = torch.linalg.cholesky(N + eta[:, None, None] * torch.eye(n, dtype=F64))
    Y = _tsolve(K, Lo.transpose(-1, -2))
    sig_eta = (1.0 + eta)[:, None, None] * (Y.transpose(-1, -2) @ Y)
    sigma = torch.where(active[:, None, None], sig_eta, Lt @ Lt.transpose(-1, -2))
    P = torch.linalg.cholesky(sigma)
    H = 0.5 * n * (1.0 + LOG_2PI) + _logdiag(P)
    if beta is None:
        ent = torch.zeros(B, dtype=torch.bool)
        alpha = torch.ones(B, dtype=F64)
    else:
        ent = torch.ones(B, dtype=torch.bool) if equality else (H.detach() < beta)
        alpha = torch.where(ent, torch.exp((beta - H) / n), torch.ones_like(H))
    out = alpha[:, None, None] * P
    # state scalars straight from Sigma~, Sigma_old and Sigma_out = (alpha P)(alpha P)^T
    la = torch.log(alpha)
    ld_out = 2.0 * _logdiag(P) + 2.0 * n * la
    tr_out_in = (_tsolve(P, Lt) ** 2).sum((-2, -1)) / alpha ** 2         # tr(Sigma_out^-1 Sigma~)
    tr_old_out = alpha ** 2 * (_tsolve(Lo, P) ** 2).sum((-2, -1))        # tr(Sigma_old^-1 Sigma_out)
    nan = torch.full_like(kl0, float("nan"))
    sc = torch.stack([eta, active.to(F64), kl0, nan, alpha, ent.to(F64), alpha ** 2,
                      0.5 * (tr_out_in - n), 0.5 * (ld_out - ld_in), 0.5 * n * (1.0 + LOG_2PI) + 0.5 * ld_out,
                      0.5 * ((X * X).sum((-2, -1)) - n), 0.5 * (ld_old - ld_in),
                      0.5 * (tr_old_out - n), 0.5 * (ld_old - ld_out), nan, nan], -1)
    return dict(eta=eta, eta_star=eta_star, active=active, kl0=kl0, lam=lam, sigma=sigma, proj=P, alpha=alpha, ent=ent,
                out=out, scalars=sc, dfde=dfde)


# ---------------------------------------------------------------------------------------------------------------------
# spectra
# ---------------------------------------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _l_old(n, g):
    """Well-conditioned old factor (condition number of Sigma_old below ~10, standard deviations ~0.3-0.8)."""
    A = torch.randn(n, n, generator=g, dtype=F64)
    S = 0.2 * (torch.eye(n, dtype=F64) + 0.6 * A @ A.T / n)
    return torch.linalg.cholesky(S)


def _orth(n, g):
    Q, R = torch.linalg.qr(torch.randn(n, n, generator=g, dtype=F64))
    return Q * torch.sign(torch.diagonal(R))


def _clusters(n, gap, k):
    centres = torch.tensor([0.55, 1.6, 3.1], dtype=F64)[:k]
    i = torch.arange(n)
    return centres[i % k] * (1.0 + gap * (i // k).to(F64))


def _log_uniform(n, lo, hi, g):
    return torch.exp(math.log(lo) + (math.log(hi) - math.log(lo)) * torch.rand(n, generator=g, dtype=F64))


def _for_eta(n, eta, g):
    """lam with KL_cov(eta) ~ eps at about ``eta`` (for eta >> lam: KL ~ sum (lam - 1)^2 / (4 eta^2))."""
    lam0 = 1.0 + eta * math.sqrt(4.0 * EPS / n)
    return lam0 * torch.exp(0.05 * (2.0 * torch.rand(n, generator=g, dtype=F64) - 1.0))


# label -> lam (None: L~ = c L_old with the power of two c, exact in fp32)
CASES = {
    "equal_c0.5": 0.5, "equal_c2": 2.0, "equal_c1": 1.0,
    "clustered_3x1e-6": lambda n, g: _clusters(n, 1e-6, 3),
    "clustered_2x1e-4": lambda n, g: _clusters(n, 1e-4, 2),
    "clustered_3x1e-3": lambda n, g: _clusters(n, 1e-3, 3),
    "wide_1e-3_1e3": lambda n, g: _log_uniform(n, 1e-3, 1e3, g),
    "wide_1e-4_1e5": lambda n, g: _log_uniform(n, 1e-4, 1e5, g),
    "eta_1e6": lambda n, g: _for_eta(n, 1e6, g),
    "eta_5e6": lambda n, g: _for_eta(n, 5e6, g),
    "eta_1.2e7": lambda n, g: _for_eta(n, 1.2e7, g),
    "eta_1e8": lambda n, g: _for_eta(n, 1e8, g),
}


def make_pair(label, n, seed):
    """(L~, L_old) fp32-rounded (returned as fp64, exact) with L~ = chol(L_old Q diag(1 / lam) Q^T L_old^T)."""
    g = _gen(seed)
    Lo = _l_old(n, g)
    spec = CASES[label] if label in CASES else label
    if isinstance(spec, float):
        Lt = spec * Lo
    else:
        lam = spec(n, g)
        Q = _orth(n, g)
        M = Lo @ Q
        Lt = torch.linalg.cholesky((M / lam) @ M.T)
    return torch.tril(Lt).float().double(), torch.tril(Lo).float().double()


def make_batch(labels, n, seed):
    pairs = [make_pair(lb, n, seed + 7919 * k) for k, lb in enumerate(labels)]
    return torch.stack([p[0] for p in pairs]), torch.stack([p[1] for p in pairs])


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference itself
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [7, 28])
def test_reference_matches_oracle_on_distinct_eigenvalues(n):
    labels = ["wide_1e-3_1e3", "clustered_3x1e-3", "eta_1e6", "wide_1e-4_1e5"]
    Lt0, Lo = make_batch(labels, n, seed=3)
    # break the 1e-3 clusters: the oracle's eigenvector gradient needs distinct eigenvalues
    Lt0[1] = make_pair(lambda n_, g: torch.linspace(0.5, 3.0, n_, dtype=F64), n, 5)[0]
    S = torch.randn(Lt0.shape, generator=_gen(1), dtype=F64)
    S = S + S.transpose(-1, -2)
    res = []
    for fn in ("ref", "oracle"):
        Lt = Lt0.clone().requires_grad_(True)
        if fn == "ref":
            r = kl_reference(Lt, Lo, EPS)
            sig, act = r["sigma"], r["active"]
        else:
            sig, act = oproj.kl_cov_projection(Lt, Lo, EPS)
        (sig * S).sum().backward()
        res.append((sig.detach(), act, Lt.grad))
    (s1, a1, g1), (s2, a2, g2) = res
    assert torch.equal(a1, a2) and bool(a1.all())
    for b in range(len(labels)):
        assert (s1[b] - s2[b]).abs().max() <= 1e-10 * s2[b].abs().max(), labels[b]
        assert (g1[b] - g2[b]).abs().max() <= 1e-9 * g2[b].abs().max(), labels[b]
    assert (kl_of_sigma(s1, Lo) - EPS).abs().max() <= 1e-12


@pytest.mark.parametrize("c", [0.5, 2.0, 0.125])
def test_reference_closed_form_for_a_scaled_factor(c):
    """L~ = c L_old: lam = 1 / c^2 (all equal), Sigma_proj = s Sigma_old with s = (1 + eta) / (lam + eta)."""
    n = 9
    Lo = make_pair("equal_c1", n, 11)[1][None]
    r = kl_reference(c * Lo, Lo, EPS)
    lam = 1.0 / c ** 2
    eta = r["eta"].item()
    assert abs(0.5 * n * (1.0 / ((lam + eta) / (1.0 + eta)) - 1.0 + math.log((lam + eta) / (1.0 + eta))) - EPS) <= 1e-14
    s = (1.0 + eta) / (lam + eta)
    ref = s * Lo @ Lo.transpose(-1, -2)
    assert (r["sigma"] - ref).abs().max() <= 1e-13 * ref.abs().max()
    assert (r["lam"] - lam).abs().max() <= 1e-12 * lam


def test_reference_gradcheck_on_degenerate_spectra():
    """Equal eigenvalues (L~ = L_old / 2) and a 1e-6 cluster: the gradient of the output factor (entropy control on)
    and of Sigma_proj exists and matches finite differences."""
    n = 4
    Lo = make_pair("equal_c1", n, 2)[1][None]
    Lc = make_pair("clustered_3x1e-6", n, 4)
    for Lt0, Lo_ in ((0.5 * Lo, Lo), (Lc[0][None], Lc[1][None])):
        H = 0.5 * n * (1.0 + LOG_2PI) + _logdiag(Lo_)
        beta = H + 0.2

        def f(x):
            r = kl_reference(torch.tril(x), Lo_, EPS, beta, False)
            return r["out"], r["sigma"]
        assert bool(kl_reference(Lt0, Lo_, EPS)["active"].all())
        assert torch.autograd.gradcheck(f, (Lt0.clone().requires_grad_(True),), eps=1e-6, atol=1e-6, rtol=1e-5)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the kernels against the reference
# ---------------------------------------------------------------------------------------------------------------------
DEV = "cuda"
MAIN = list(CASES)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _layout_batch(layout, labels, n, seed):
    """``labels`` once (B <= number of SMs: one 512-thread CTA per matrix), or cycled with fresh draws to more matrices
    than SMs (the two-CTAs-per-SM `compact` variant)."""
    if layout == "one_cta_per_matrix":
        assert len(labels) <= _sms()
        lab = list(labels)
    else:
        lab = [labels[k % len(labels)] for k in range(_sms() + 5)]
    Lt, Lo = make_batch(lab, n, seed)
    return lab, Lt, Lo


class Bounds:
    """Collects every violated bound of a test (with the case that violated it) and fails once, listing them all."""

    def __init__(self, labels):
        self.labels, self.fails = labels, []

    def per_matrix(self, what, err, tol, mask=None):
        err, tol = torch.as_tensor(err, dtype=F64).cpu(), torch.as_tensor(tol, dtype=F64).cpu().expand_as(err)
        bad = ~(err <= tol)
        if mask is not None:
            bad &= mask.cpu()
        for b in torch.nonzero(bad).flatten().tolist():
            self.fails.append(f"{what} [{b}:{self.labels[b]}]: {err[b].item():.3g} > {tol[b].item():.3g}")

    def check(self):
        assert not self.fails, f"{len(self.fails)} bound(s) missed:\n" + "\n".join(self.fails[:60])


def _amax(x):
    return x.abs().flatten(1).max(1).values


# Bounds that follow from the Jacobi stopping rule (csrc/tce_smem_la.cuh, LA_JACOBI_TOL2) rather than from fp64
# rounding; the numbers are documented there.  The factors: measured up to 6e-6 of max|.| (a 2x1e-4-clustered
# spectrum at n = 7).  The scalars that are sums over the eigenvalues (kl0 and the KL decompositions) see the residual
# of the last sweep in second order: measured up to 1e-6 relative on 1e-6 clusters.  eta, Sigma_proj and the
# constraint are held to the bounds the projection promises its users; the gradients see check_grad.
FACTOR_OF_MAX = 1e-5
EIGEN_SUM_REL = 2e-6


def kernel_lam(state, B, n):
    """The generalised eigenvalues the forward kernel found (a view of its state)."""
    o = 4 * B * n * n
    return state[o:o + B * n].view(B, n)


def check_forward(bd, ref, state, n, proj=None, out=None, info=None, eps=EPS, eta_vs_reference=True):
    """Everything the forward leaves behind, against the reference.  eta is checked twice: against the root of
    KL_cov(eta) = eps on the kernel's own eigenvalues (the dual solve alone) and against the reference's eta (the
    eigenvalues as well; ``eta_vs_reference=False`` where that root is ill-conditioned: test_kl_cov_at_the_bound)."""
    B = len(bd.labels)
    sc = ops.kl_state_scalars(state, B, n).cpu()
    sigma = ops.kl_state_sigma(state, B, n)[0].cpu()
    act = ref["active"]
    eps_t = torch.as_tensor(eps, dtype=F64).expand(B)
    if info is not None:
        bd.per_matrix("info", info.cpu().abs().to(F64), 0.0)
    bd.per_matrix("active flag", (sc[:, 1] - act.to(F64)).abs(), 0.0)
    root = solve_eta(kernel_lam(state, B, n).cpu(), eps_t)
    bd.per_matrix("eta vs the root on the kernel's eigenvalues (rel)", (sc[:, 0] - root).abs(), 1e-6 * root, act)
    eta_r = ref["eta"].detach()
    if eta_vs_reference:
        bd.per_matrix("eta (rel)", (sc[:, 0] - eta_r).abs(), 1e-6 * eta_r, act)
    kl_state = kl_of_sigma(sigma, ref["Lo"])
    bd.per_matrix("KL(Sigma_proj || Sigma_old) - eps", (kl_state - eps_t).abs(), 1e-7 * eps_t, act)
    sig_r = ref["sigma"].detach()
    bd.per_matrix("Sigma_proj", _amax(sigma - sig_r), 1e-5 * _amax(sig_r))
    scale = torch.maximum(ref["scalars"].detach().abs(), torch.ones(1, dtype=F64) * eps_t[:, None])
    for k, name, rel in [(2, "kl0", EIGEN_SUM_REL), (4, "alpha", 1e-8), (5, "entropy active", 0.0),
                         (6, "alpha^2", 1e-8), (7, "tr-region shape", EIGEN_SUM_REL),
                         (8, "tr-region volume", EIGEN_SUM_REL), (10, "KL(in||old) shape", EIGEN_SUM_REL),
                         (11, "KL(in||old) volume", EIGEN_SUM_REL), (12, "KL(out||old) shape", EIGEN_SUM_REL),
                         (13, "KL(out||old) volume", EIGEN_SUM_REL)]:
        bd.per_matrix(f"state[{k}] {name}", (sc[:, k] - ref["scalars"][:, k].detach()).abs(), rel * scale[:, k])
    Hs = torch.maximum(ref["scalars"][:, 9].detach().abs(), torch.ones(1, dtype=F64))
    bd.per_matrix("state[9] entropy of the output", (sc[:, 9] - ref["scalars"][:, 9].detach()).abs(), 1e-8 * Hs)
    for name, got, r in (("proj_L", proj, ref["proj"]), ("out_L", out, ref["out"])):
        if got is None:
            continue
        r = r.detach()
        e = _amax(got.cpu().double() - r)
        bd.per_matrix(f"{name} (abs)", e, 1e-4)
        bd.per_matrix(f"{name} (of max)", e, FACTOR_OF_MAX * _amax(r))


def check_grad(bd, what, got, ref_grad, upstream, output, Lt):
    """2e-4 of max|grad| (the project's gradient tolerance), but never below 1e-5 of the gradient's scale without the
    constraint, max|upstream| max|output| / max|L~|: that is the relative residual the Jacobi stopping rule documents
    for f(N), and the level of the rounding noise where the gradient vanishes analytically (n = 1 with the KL step or
    the entropy control active: KL(out || old) = eps or H(out) = beta fixes the output's covariance)."""
    natural = _amax(upstream.double()) * _amax(output.detach()) / _amax(Lt.detach())
    tol = torch.maximum(2e-4 * _amax(ref_grad), 1e-5 * natural)
    e = _amax(got.cpu().double() - ref_grad)
    bd.per_matrix(what, e, tol)


def _ref(Lt, Lo, eps=EPS, beta=None, equality=False):
    Ltg = Lt.clone().requires_grad_(True)
    r = kl_reference(Ltg, Lo, eps, beta, equality)
    r["Lt"], r["Lo"] = Ltg, Lo
    return r


def _ref_grad(r, loss):
    (g,) = torch.autograd.grad(loss, r["Lt"], retain_graph=True)
    return torch.tril(g)


def _upstream(shape, seed):
    g = _gen(seed)
    G = torch.tril(torch.randn(shape, generator=g)).float()                   # factor path (fp32, lower)
    S = torch.randn(shape, generator=g, dtype=F64)
    return G, S + S.transpose(-1, -2)                                          # Sigma path (fp64, symmetric)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("n", NS)
def test_kl_cov_forward_backward_on_spectra(n, layout):
    """``ops.proj_kl_cov`` (cold): factor, state, scalars and the factor-path gradient on every spectrum."""
    labels, Lt, Lo = _layout_batch(layout, MAIN, n, seed=100 + n)
    ref = _ref(Lt, Lo)
    G, _ = _upstream(Lt.shape, 7 + n)
    bd = Bounds(labels)
    L = Lt.float().to(DEV).requires_grad_(True)
    state = ops.kl_state(len(labels), n, DEV)
    proj, info = ops.proj_kl_cov(L, Lo.float().to(DEV), EPS, state, False)
    (proj * G.to(DEV)).sum().backward()
    check_forward(bd, ref, state, n, proj=proj.detach(), info=info)
    check_grad(bd, "L.grad", L.grad, _ref_grad(ref, (ref["proj"] * G.double()).sum()), G, ref["proj"], Lt)
    bd.check()


@pytest.mark.gpu
@pytest.mark.parametrize("split,equality", [(False, False), (True, False), (False, True), (True, True)])
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("n", NS)
def test_kl_entropy_on_spectra(n, layout, split, equality):
    """``ops.proj_kl_entropy`` (fused entropy control, one or two launches): gradients through the output factor and,
    with ``return_sigma``, through Sigma_out (``tce_proj_kl_bwd_sigma``).  The entropy bound sits 0.3 nats above the
    projected entropy for every other matrix and 0.3 below for the rest."""
    labels, Lt, Lo = _layout_batch(layout, MAIN, n, seed=200 + n)
    B = len(labels)
    H = _ref(Lt, Lo)["scalars"][:, 9].detach()
    beta = H + torch.where(torch.arange(B) % 2 == 0, 0.3, -0.3).to(F64)
    ref = _ref(Lt, Lo, EPS, beta, equality)
    G, S = _upstream(Lt.shape, 9 + n)
    bd = Bounds(labels)
    Ld, Lod, betad = Lt.float().to(DEV), Lo.float().to(DEV), beta.to(DEV)
    L = Ld.clone().requires_grad_(True)
    state = ops.kl_state(B, n, DEV)
    out, proj, info = ops.proj_kl_entropy(L, Lod, EPS, state, False, betad, equality, split)
    (out * G.to(DEV)).sum().backward()
    check_forward(bd, ref, state, n, proj=proj, out=out.detach(), info=info)
    check_grad(bd, "L.grad (factor path)", L.grad, _ref_grad(ref, (ref["out"] * G.double()).sum()), G, ref["out"],
               Lt)
    L2 = Ld.clone().requires_grad_(True)
    state2 = ops.kl_state(B, n, DEV)
    res = ops.proj_kl_entropy(L2, Lod, EPS, state2, False, betad, equality, split, return_sigma=True)
    (res[3] * S.to(DEV)).sum().backward()                      # d loss / d Sigma_out, Sigma_out = alpha^2 Sigma0
    sig_out = ref["alpha"][:, None, None] ** 2 * ref["sigma"]
    check_grad(bd, "L.grad (Sigma path)", L2.grad, _ref_grad(ref, (sig_out * S).sum()), S, sig_out, Lt)
    bd.check()


@pytest.mark.gpu
@pytest.mark.parametrize("side", ["barely_active", "barely_inactive"])
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("n", NS)
def test_kl_cov_at_the_bound(n, layout, side):
    """eps = kl0 / (1 + 1e-6) (active, eta ~ 5e-7: below the search grid's first point 2^-10) and kl0 (1 + 1e-6)
    (inactive).  eps is a scalar per launch, so a batch above the SM count is one matrix repeated."""
    label = "near_one"
    Lt1, Lo1 = make_pair(lambda n_, g: torch.exp(0.06 * torch.randn(n_, generator=g, dtype=F64)), n, 300 + n)
    reps = 1 if layout == "one_cta_per_matrix" else _sms() + 5
    Lt, Lo = Lt1.expand(reps, n, n).contiguous(), Lo1.expand(reps, n, n).contiguous()
    kl0 = _ref(Lt1[None], Lo1[None])["kl0"].item()
    eps = kl0 / (1.0 + 1e-6) if side == "barely_active" else kl0 * (1.0 + 1e-6)
    ref = _ref(Lt, Lo, eps)
    assert bool(ref["active"].all()) == (side == "barely_active")
    G, _ = _upstream(Lt.shape, 11 + n)
    bd = Bounds([label] * reps)
    L = Lt.float().to(DEV).requires_grad_(True)
    state = ops.kl_state(reps, n, DEV)
    proj, info = ops.proj_kl_cov(L, Lo.float().to(DEV), eps, state, False)
    (proj * G.to(DEV)).sum().backward()
    # eta ~ 5e-7 moves by (error of KL(0)) / |KL'(0)|: a relative error of 1e-10 in the kernel's kl0 (the eigenvalues of
    # an fp64 Jacobi sweep on W = L~^-1 L_old) is 1e-4 of eta here.  What eta is for -- the constraint, Sigma_proj, the
    # factor -- is held to the usual bounds, and the dual solve to 1e-6 on the kernel's own eigenvalues.
    check_forward(bd, ref, state, n, proj=proj.detach(), info=info, eps=eps, eta_vs_reference=False)
    check_grad(bd, "L.grad", L.grad, _ref_grad(ref, (ref["proj"] * G.double()).sum()), G, ref["proj"], Lt)
    bd.check()


def _vec_from_factor(Lt, min_std):
    """The covariance vector that the policy head maps back to L~: softplus^-1(L~_ii - min_std), then the strictly
    lower entries row by row."""
    n = Lt.shape[-1]
    d = torch.diagonal(Lt) - min_std
    v_diag = d + torch.log(-torch.expm1(-d))                                   # softplus^-1, stable
    r, c = torch.tril_indices(n, n, -1)
    return torch.cat([v_diag, Lt[r, c]])


# Measured misses of the gradient bound, left failing on purpose: with the trust-region term folded in, the gradient
# on the 3 x 1e-6-clustered spectrum is off by 2.0e-4, 2.5e-4 and 2.4e-4 of max|grad| at n = 32, 63, 64, i.e. ~1e-4
# of the gradient's unconstrained scale, ten times the Jacobi residual.  Not fixed here: any change to the backward
# changes the shared-covariance epoch's results.  A likely cause is that the term's closed form (csrc/tce_proj.cu,
# proj_kl_cov_bwd_sigma_kernel: Sigma_out^-1 L~ = L~^-T U~ diag(1 / (alpha^2 lam^2 D)) U~^T) takes the columns of U~
# as exactly orthogonal.  Strict: a kernel that meets the bound turns these into failures, and the entries go.
VEC_GRAD_MISSES = {(32, "clustered_3x1e-6"), (63, "clustered_3x1e-6"), (64, "clustered_3x1e-6")}


def _vec_cases():
    for n in NS:
        for label in MAIN:
            marks = [pytest.mark.xfail(strict=True, reason="measured gradient miss (VEC_GRAD_MISSES)")] \
                if (n, label) in VEC_GRAD_MISSES else []
            yield pytest.param(n, label, marks=marks, id=f"{n}-{label}")


@pytest.mark.gpu
@pytest.mark.parametrize("n,label", list(_vec_cases()))
def test_fused_head_shared_vector_path_on_spectra(n, label):
    """The shared-covariance epoch's chain (rl/fast_epoch.py): ``tce_proj_kl_entropy_fwd_sigma_vec`` (policy head
    fused in, B = 1, ldb_vec = 0) -> ``tce_proj_kl_bwd_prep`` -> ``tce_proj_kl_bwd_sigma_k_vec`` (gradient w.r.t. the
    vector, with the trust-region term tr_coeff KL_cov(N(L~ L~^T) || N(Sigma_out detached)) folded in as the epoch does
    when the trust-region loss has a covariance part)."""
    p = ops._p
    min_std, tr_coeff = 1e-4, 1.0
    k = MAIN.index(label)
    Lt, Lo = make_pair(label, n, 400 + 31 * k + n)
    vec = _vec_from_factor(Lt, min_std).float().to(DEV)
    H = _ref(Lt[None], Lo[None])["scalars"][:, 9].detach()
    beta = H + (0.3 if k % 2 == 0 else -0.3)
    L_new = torch.empty(1, n, n, device=DEV)
    scratch = torch.empty(2, n, n, device=DEV)
    info = torch.empty(1, device=DEV, dtype=torch.int32)
    state = ops.kl_state(1, n, DEV)
    Lod = Lo.float().to(DEV)[None].contiguous()
    s = torch.cuda.current_stream().cuda_stream
    _lib.call("tce_proj_kl_entropy_fwd_sigma_vec", p(vec), 0, float(min_std), p(L_new), p(Lod), EPS,
              p(beta.to(DEV)), 0, 0, p(scratch[0]), p(scratch[1]), p(state), p(info), 0, 1, n, s)
    _lib.call("tce_proj_kl_bwd_prep", p(state), 1, n, s)
    _, S = _upstream((1, n, n), 13 + k)
    g_S = S.to(DEV).contiguous()
    gvec = torch.full_like(vec, float("nan"))
    _lib.call("tce_proj_kl_bwd_sigma_k_vec", p(L_new), p(vec), 0, p(g_S), p(state), 1, tr_coeff, p(gvec), 1, n,
              s)
    torch.cuda.synchronize()
    Lb = L_new.cpu().double()
    bd = Bounds([label])
    # the factor the head built: L~ up to the fp32 softplus
    bd.per_matrix("L_built", _amax(Lb - Lt[None]), 4e-7 * _amax(Lt[None]))
    ref = _ref(Lb, Lo[None], EPS, beta, False)
    check_forward(bd, ref, state, n)             # (info: written by the Cholesky launch, which this chain skips)
    sig_out = ref["alpha"][:, None, None] ** 2 * ref["sigma"]
    C = ref["out"].detach()                                              # Sigma_out = C C^T, detached
    X = _tsolve(C, ref["Lt"])
    kl_tr = 0.5 * ((X * X).sum() - n + 2.0 * _logdiag(C).sum() - 2.0 * _logdiag(ref["Lt"]).sum())
    gL = _ref_grad(ref, (sig_out * S).sum() + tr_coeff * kl_tr)[0]
    r, c = torch.tril_indices(n, n, -1)
    sig = torch.sigmoid(vec.cpu().double()[:n])
    g_ref = torch.cat([torch.diagonal(gL) * sig, gL[r, c]])
    check_grad(bd, "vec.grad", gvec[None], g_ref[None], S, sig_out, Lb)
    bd.check()


# ---------------------------------------------------------------------------------------------------------------------
# warm starts that have work to do
# ---------------------------------------------------------------------------------------------------------------------
WARM_N = 63                      # the box-pushing policy's parameter count


def _warm_sequence(label, B, seed, steps=6):
    """L_k = L_0 + k Delta with Delta ~1e-3 |L_0| per entry (lower, random signs): rotates the eigen-basis instead of
    scaling it, as one Adam step of the covariance parameters does."""
    lab = [label] * B
    Lt0, Lo = make_batch(lab, WARM_N, seed)
    D = 1e-3 * torch.tril(torch.randn(Lt0.shape, generator=_gen(seed + 1), dtype=F64)) * Lt0.abs()
    return lab, Lo, [(Lt0 + k * D).float().double() for k in range(steps)]


def _layout_B(layout):
    return 1 if layout == "one_cta_per_matrix" else _sms() + 5


def _run_cov(Lt, Lo, state, warm, G):
    L = Lt.float().to(DEV).requires_grad_(True)
    proj, info = ops.proj_kl_cov(L, Lo.float().to(DEV), EPS, state, warm)
    (proj * G.to(DEV)).sum().backward()
    return proj.detach(), info, L.grad


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("label", ["clustered_2x1e-4", "clustered_3x1e-6", "wide_1e-3_1e3", "wide_1e-4_1e5"])
def test_warm_start_sequence_equals_cold_and_reference(label, layout):
    """Six calls of one update (warm = True: Jacobi starts from the previous basis, Newton from the previous eta): each
    equals a cold call on the same input and the reference, within the bounds of the cold tests."""
    B = _layout_B(layout)
    labels, Lo, seq = _warm_sequence(label, B, seed=500)
    state = ops.kl_state(B, WARM_N, DEV)
    G, _ = _upstream(Lo.shape, 17)
    fails = []
    for k, Lt in enumerate(seq):
        ref = _ref(Lt, Lo)
        g_ref = _ref_grad(ref, (ref["proj"] * G.double()).sum())
        for mode in ("warm", "cold"):
            st = state if mode == "warm" else ops.kl_state(B, WARM_N, DEV)
            proj, info, grad = _run_cov(Lt, Lo, st, mode == "warm", G)
            bd = Bounds([f"{lb} step {k} {mode}" for lb in labels])
            check_forward(bd, ref, st, WARM_N, proj=proj, info=info)
            check_grad(bd, "L.grad", grad, g_ref, G, ref["proj"], Lt)
            fails += bd.fails
            if mode == "warm":
                warm_proj = proj
            else:
                e = _amax(warm_proj.cpu().double() - proj.cpu().double())
                bd2 = Bounds([f"{lb} step {k}" for lb in labels])
                bd2.per_matrix("warm vs cold proj_L", e, FACTOR_OF_MAX * _amax(proj.cpu().double()))
                fails += bd2.fails
    assert not fails, f"{len(fails)} bound(s) missed:\n" + "\n".join(fails[:60])


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("jump", ["eta0_1e3_times_root", "eta0_1e-3_times_root", "previous_step_inactive"])
def test_warm_start_after_an_eta_jump(jump, layout):
    """The warm Newton solve starts from a previous eta 1e3x above or below the new root (it must leave the positive
    axis or run out of steps and fall back to the bracket), or after an inactive call whose eta must be ignored.  The
    warm Newton accepts only a converged root, so a stale eta0 can cost steps but not change the result: the inactive
    case checks the result after such a call, not that eta0 was skipped."""
    B = _layout_B(layout)
    labels, Lo, seq = _warm_sequence("clustered_2x1e-4", B, seed=600, steps=2)
    state = ops.kl_state(B, WARM_N, DEV)
    G, _ = _upstream(Lo.shape, 19)
    ref = _ref(seq[1], Lo)
    if jump == "previous_step_inactive":
        _run_cov((Lo * (1.0 + 1e-4)).float().double(), Lo, state, True, G)
        sc = ops.kl_state_scalars(state, B, WARM_N)
        assert bool((sc[:, 1] == 0).all())
        sc[:, 0] = 1e3 * ref["eta"].detach().to(DEV)                   # must be ignored: the step was inactive
    else:
        _run_cov(seq[0], Lo, state, True, G)
        sc = ops.kl_state_scalars(state, B, WARM_N)
        assert bool((sc[:, 1] != 0).all())
        ratio = 1e3 if jump == "eta0_1e3_times_root" else 1e-3
        sc[:, 0] = ratio * ref["eta"].detach().to(DEV)
    proj, info, grad = _run_cov(seq[1], Lo, state, True, G)
    bd = Bounds(labels)
    check_forward(bd, ref, state, WARM_N, proj=proj, info=info)
    check_grad(bd, "L.grad", grad, _ref_grad(ref, (ref["proj"] * G.double()).sum()), G, ref["proj"], seq[1])
    bd.check()


# ---------------------------------------------------------------------------------------------------------------------
# diagonal factors: the same eigenvalues through the closed-form kernel
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", NS)
def test_kl_diag_on_the_same_spectra(n):
    """``ops.proj_kl_diag`` on lam_i = (s_old,i / s_i)^2 from every spectrum: eta, output and gradient against the
    reference, and the dense kernel on the same diagonal factors finds the same eta."""
    g = _gen(700 + n)
    Lt, Lo = [], []
    for label in MAIN:
        so = 0.3 + 0.5 * torch.rand(n, generator=g, dtype=F64)
        spec = CASES[label]
        lam = torch.full((n,), 1.0 / spec ** 2, dtype=F64) if isinstance(spec, float) else spec(n, g)
        Lo.append(torch.diag(so).float().double())
        Lt.append(torch.diag(so / lam.sqrt()).float().double())
    Lt, Lo = torch.stack(Lt), torch.stack(Lo)
    ref = _ref(Lt, Lo)
    G, _ = _upstream(Lt.shape, 23 + n)
    G = torch.diag_embed(torch.diagonal(G, dim1=-2, dim2=-1))
    bd = Bounds(MAIN)
    L = Lt.float().to(DEV).requires_grad_(True)
    out, st, info = ops.proj_kl_diag(L, Lo.float().to(DEV), EPS, None, False)
    (out * G.to(DEV)).sum().backward()
    st = st.cpu()
    act = ref["active"]
    bd.per_matrix("info", info.cpu().abs().to(F64), 0.0)
    bd.per_matrix("active flag", (st[:, 1] - act.to(F64)).abs(), 0.0)
    eta_r = ref["eta"].detach()
    bd.per_matrix("eta (rel)", (st[:, 0] - eta_r).abs(), 1e-6 * eta_r, act)
    e = _amax(out.detach().cpu().double() - ref["proj"].detach())
    bd.per_matrix("out (abs)", e, 1e-4)
    bd.per_matrix("out (of max)", e, 2e-6 * _amax(ref["proj"].detach()))
    g_ref = torch.diag_embed(torch.diagonal(_ref_grad(ref, (ref["proj"] * G.double()).sum()), dim1=-2, dim2=-1))
    check_grad(bd, "L.grad", torch.diag_embed(torch.diagonal(L.grad, dim1=-2, dim2=-1)), g_ref, G,
               ref["proj"], Lt)
    state = ops.kl_state(len(MAIN), n, DEV)
    ops.proj_kl_cov(Lt.float().to(DEV), Lo.float().to(DEV), EPS, state, False)
    eta_dense = ops.kl_state_scalars(state, len(MAIN), n)[:, 0].cpu()
    bd.per_matrix("eta dense vs diagonal kernel (rel)", (eta_dense - st[:, 0]).abs(), 1e-6 * st[:, 0], act)
    bd.check()

"""Full-covariance projections and Gaussian statistics at 64 < n <= 128 (the workspace kernels) vs the CPU fp64 oracle.

Tolerances as in test_gpu_projection.py: projected parameters / KLs / losses <= 1e-4 absolute, gradients relative to
their scale.  Factors are drawn here (synthetic_inputs stops at Dp = 63).
"""
import copy

import pytest
import torch

from oracle import agent as oa
from oracle import policy as opol
from oracle import projection as oproj

pytestmark = pytest.mark.gpu
if torch.cuda.is_available():
    from tce_rl_b200 import _lib, ops
    from tce_rl_b200.rl import agent_factory, critic_factory, policy_factory, projection_factory
    from tce_rl_b200.rl.agent import _KL_KEYS

DEV = "cuda:0"
LAYERS = [("KLProjectionLayer", 0.05, 5e-4), ("FrobeniusProjectionLayer", 0.05, 5e-4),
          ("WassersteinProjectionLayer", 0.005, 2.5e-4)]
SIZES = [65, 70, 96, 112, 127, 128]


def f64(t):
    return t.detach().double().cpu()


def layer_kwargs(typ, mb, cb, Dp, schedule="linear", scale_prec=True):
    return dict(proj_type=typ, mean_bound=mb, cov_bound=cb, trust_region_coeff=1.0, scale_prec=scale_prec,
                entropy_schedule=schedule, action_dim=Dp, total_train_steps=7500, target_entropy=0.0,
                temperature=0.7, entropy_eq=False, entropy_first=False, do_regression=False)


class FakePolicy:
    """Duck-typed policy surface the GPU layers need."""
    def __init__(self, contextual):
        self.contextual_std, self.is_diag = contextual, False

    def entropy(self, p):
        return ops.gauss_stats(p[0], p[1], p[0], p[1])[:, 4]


def draw(B, n, contextual, seed=0):
    """fp32 (mean, L, mean_old, L_old); episode 0 lies inside the trust region (identity branch)."""
    g = torch.Generator().manual_seed(seed)
    Bf = B if contextual else 1
    Lo = torch.tril(torch.randn(Bf, n, n, generator=g) * 0.3 / n ** 0.5, -1) \
        + torch.diag_embed(0.5 + torch.rand(Bf, n, generator=g))
    L = Lo + torch.tril(torch.randn(Bf, n, n, generator=g) * 0.02 / n ** 0.5, -1) \
        + torch.diag_embed(Lo.diagonal(dim1=-2, dim2=-1) * 0.05 * torch.randn(Bf, n, generator=g))
    mo = torch.randn(B, n, generator=g) * 0.1
    m = mo + 0.05 * torch.randn(B, n, generator=g)
    m[0] = mo[0] + 1e-4
    if contextual:
        L[0] = Lo[0] * (1 + 1e-5)
    else:
        L, Lo = L.expand(B, n, n).contiguous(), Lo.expand(B, n, n).contiguous()
    return m.float(), L.float(), mo.float(), Lo.float()


def spectrum_factors(n, kind, seed=0):
    """(L, L_old) whose generalised eigenvalues are clustered, wide or extreme (as test_gpu_kl_spectra.py)."""
    g = torch.Generator().manual_seed(seed)
    Q, _ = torch.linalg.qr(torch.randn(n, n, generator=g, dtype=torch.float64))
    if kind == "clustered":
        lam = torch.cat([torch.full((n // 2,), 1.0), torch.full((n - n // 2,), 1.3)]) \
            + 1e-4 * torch.arange(n, dtype=torch.float64) / n
    elif kind == "wide":
        lam = torch.logspace(-1, 1, n, dtype=torch.float64)
    else:
        lam = torch.logspace(-3, 3, n, dtype=torch.float64)
    Lo = torch.linalg.cholesky(torch.eye(n, dtype=torch.float64) + 0.1 * torch.ones(n, n, dtype=torch.float64))
    # Sigma = Lo Q diag(1 / lam) Q^T Lo^T: eigenvalues of Sigma_o relative to Sigma are lam
    S = Lo @ Q @ torch.diag(1.0 / lam) @ Q.T @ Lo.T
    L = torch.linalg.cholesky(0.5 * (S + S.T))
    return L.float(), Lo.float()


@pytest.mark.parametrize("typ,mb,cb", LAYERS)
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("contextual", [True, False])
def test_layer_forward_backward(typ, mb, cb, n, contextual):
    """Every projection layer forward, trust-region loss and backward, active and inactive episodes."""
    B = 6
    m, L, mo, Lo = draw(B, n, contextual, seed=n)
    d = lambda t: t.double()
    opolicy = opol.BlackBoxPolicy(n, contextual=contextual, min_std=1e-4)
    olayer = oproj.projection_factory(typ, dtype=torch.float64, **layer_kwargs(typ, mb, cb, n))
    olayer.initial_entropy = opolicy.entropy([d(mo), d(Lo)]).mean()
    m64, L64 = d(m).requires_grad_(True), d(L).requires_grad_(True)
    pm, pL = olayer(opolicy, (m64, L64), (d(mo), d(Lo)), 100)
    g = torch.Generator().manual_seed(1)
    wm = torch.randn(B, n, generator=g, dtype=torch.float64)
    wL = torch.tril(torch.randn(B, n, n, generator=g, dtype=torch.float64))
    tr = olayer.get_trust_region_loss(opolicy, (m64, L64), (pm, pL), set_variance=False)
    gm, gL = torch.autograd.grad((pm * wm).sum() + (pL * wL).sum() + tr, [m64, L64])

    layer = projection_factory(typ, device=DEV, dtype="float32", **layer_kwargs(typ, mb, cb, n))
    layer.initial_entropy = olayer.initial_entropy.float().to(DEV)
    pol = FakePolicy(contextual)
    mg, Lg = m.to(DEV).requires_grad_(True), L.to(DEV).requires_grad_(True)
    pmg, pLg = layer(pol, (mg, Lg), (mo.to(DEV), Lo.to(DEV)), 100)
    assert (f64(pmg) - pm.detach()).abs().max() <= 1e-4
    assert (f64(pLg) - pL.detach()).abs().max() <= 1e-4
    trg = layer.get_trust_region_loss(pol, (mg, Lg), (pmg, pLg), set_variance=False)
    assert abs(trg.item() - tr.item()) <= 1e-4 * max(1.0, abs(tr.item()))
    ((pmg * wm.float().to(DEV)).sum() + (pLg * wL.float().to(DEV)).sum() + trg).backward()
    assert (f64(mg.grad) - gm).abs().max() <= 2e-4 * max(1.0, gm.abs().max().item())
    gL_t, gL_g = torch.tril(gL), f64(Lg.grad)
    if not contextual:
        gL_t, gL_g = gL_t.sum(0), gL_g.sum(0)
    assert (gL_g - gL_t).abs().max() <= 2e-4 * max(1.0, gL_t.abs().max().item())
    mp0, cp0 = olayer.trust_region_value(opolicy, (d(m), d(L)), (d(mo), d(Lo)))
    assert (mp0 > mb).any() and (mp0 <= mb).any()
    if contextual and typ != "WassersteinProjectionLayer":
        assert (cp0 > cb).any() and (cp0 <= cb).any()


def kl_cov(L, Lo, state, warm):
    """Covariance of the GPU KL projection (fp64 on the CPU) and the factor it came from."""
    P = ops.proj_kl_cov(L, Lo, 5e-4, state, warm)[0]
    return P, f64(P) @ f64(P).mT


@pytest.mark.parametrize("n", [65, 128])
@pytest.mark.parametrize("B", [1, 149, 300])
def test_kl_projection_batches(n, B):
    """Per-episode KL covariance projection forward and backward: one matrix, and batches that are not a multiple of
    a launch of as many CTAs as SMs."""
    m, L, mo, Lo = draw(B, n, True, seed=7 + B)
    L64 = L.double().requires_grad_(True)
    ref, active = oproj.kl_cov_projection(L64, Lo.double(), 5e-4)
    assert active[1:].all() and not active[0]
    Lg = L.to(DEV).requires_grad_(True)
    P, cov = kl_cov(Lg, Lo.to(DEV), ops.kl_state(B, n, DEV), False)
    assert (cov - ref.detach()).abs().max() <= 1e-4 * max(1.0, ref.abs().max().item())
    w = torch.randn(B, n, n, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    (gref,) = torch.autograd.grad((ref * w).sum(), [L64])
    (((P @ P.mT) * w.float().to(DEV)).sum()).backward()
    assert (f64(Lg.grad) - torch.tril(gref)).abs().max() <= 2e-3 * max(1.0, gref.abs().max().item())


@pytest.mark.parametrize("kind", ["clustered", "wide", "extreme"])
def test_kl_hard_spectra_and_warm_start(kind):
    """n = 128: clustered, wide and extreme generalised spectra; a warm start from the state of the same L_old (the
    fingerprint matches) and one from another L_old (it does not) match the oracle as the cold start does."""
    n = 128
    L, Lo = spectrum_factors(n, kind)
    state = ops.kl_state(1, n, DEV)
    for LL, LO, warm, reused in ((L, Lo, False, False), (L * 1.001, Lo, True, True), (L, Lo * 1.01, True, False)):
        ref = oproj.kl_cov_projection(LL.double()[None], LO.double()[None], 5e-4)[0]
        fp_before = ops.kl_state_scalars(state, 1, n)[0, 3].item()
        with torch.no_grad():
            cov = kl_cov(LL.to(DEV)[None], LO.to(DEV)[None], state, warm)[1]
        # the forward starts from the saved basis exactly when the fingerprint of L_old it saved matches this one's
        assert (ops.kl_state_scalars(state, 1, n)[0, 3].item() == fp_before) == reused
        assert (cov - ref).abs().max() <= 1e-4 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("n", SIZES)
def test_gauss_stats_tri_inverse_cov_distance(n):
    B = 5
    m, L, mo, Lo = draw(B, n, True, seed=3 * n)
    d = lambda t: t.double()
    S, So = d(L) @ d(L).mT, d(Lo) @ d(Lo).mT
    Soi = torch.cholesky_inverse(d(Lo))
    diff = d(m) - d(mo)
    ref = torch.stack([torch.einsum("bi,bij,bj->b", diff, Soi, diff), (Soi @ S).diagonal(dim1=-2, dim2=-1).sum(-1),
                       torch.logdet(S), torch.logdet(So),
                       0.5 * n * (1 + 1.8378770664093453) + d(L).diagonal(dim1=-2, dim2=-1).log().sum(-1)], 1)
    mg, Lg = m.to(DEV).requires_grad_(True), L.to(DEV).requires_grad_(True)
    out = ops.gauss_stats(mg, Lg, mo.to(DEV), Lo.to(DEV))
    assert (f64(out) - ref).abs().max() <= 1e-4 * max(1.0, ref.abs().max().item())
    w = torch.randn(B, 5, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    m64, L64 = d(m).requires_grad_(True), d(L).requires_grad_(True)
    S64 = L64 @ L64.mT
    r64 = torch.stack([torch.einsum("bi,bij,bj->b", m64 - d(mo), Soi, m64 - d(mo)),
                       (Soi @ S64).diagonal(dim1=-2, dim2=-1).sum(-1), torch.logdet(S64), torch.logdet(So),
                       0.5 * n * (1 + 1.8378770664093453) + L64.diagonal(dim1=-2, dim2=-1).log().sum(-1)], 1)
    gm, gL = torch.autograd.grad((r64 * w).sum(), [m64, L64])
    (out * w.to(DEV)).sum().backward()
    assert (f64(mg.grad) - gm).abs().max() <= 2e-4 * max(1.0, gm.abs().max().item())
    assert (f64(Lg.grad) - torch.tril(gL)).abs().max() <= 2e-4 * max(1.0, gL.abs().max().item())
    inv = f64(ops.tri_inverse(Lo.to(DEV)))
    assert (inv - torch.linalg.inv(d(Lo))).abs().max() <= 1e-8 * max(1.0, inv.abs().max().item())
    opolicy = opol.BlackBoxPolicy(n, contextual=True, min_std=1e-4)
    for kind in (0, 1):
        for sp in (False, True) if kind == 1 else (False,):
            if kind == 0:
                rv = oproj.gaussian_frobenius(opolicy, (d(m), d(L)), (d(mo), d(Lo)))[1]
            else:
                rv = oproj.gaussian_wasserstein_commutative(opolicy, (d(m), d(L)), (d(mo), d(Lo)), scale_prec=sp)[1]
            val = f64(ops.cov_distance(kind, L.to(DEV), Lo.to(DEV), sp))
            assert (val - rv).abs().max() <= 1e-4 * max(1.0, rv.abs().max().item())


def test_workspace_sizes_and_refusals():
    """The *_ws twins size their workspace by the SM count, not by B; the plain entry points still refuse n > 64."""
    lib = _lib.load()
    assert lib.tce_proj_work_bytes(4, 64) == 0 and lib.tce_proj_work_bytes(4, 129) == 0
    one = lib.tce_proj_work_bytes(1, 128)
    assert one == 8 * 6 * 128 * 129
    assert lib.tce_proj_work_bytes(10 ** 6, 128) == lib.tce_proj_work_bytes(10 ** 4, 128)
    L = torch.eye(70, device=DEV).expand(2, 70, 70).contiguous()
    out = torch.empty(2, 70, 70, device=DEV, dtype=torch.float64)
    st = torch.cuda.current_stream().cuda_stream
    assert lib.tce_tri_inverse(L.data_ptr(), 70 * 70, out.data_ptr(), 2, 70, st) == -2
    assert lib.tce_tri_inverse_ws(L.data_ptr(), 70 * 70, out.data_ptr(), 2, 70, None, st) == -2


def test_empty_batch():
    """B = 0 at n > 64: every op of the family returns empty results without a launch."""
    n = 100
    z = torch.empty(0, n, device=DEV)
    zL = torch.empty(0, n, n, device=DEV)
    assert ops.gauss_stats(z, zL, z, zL).shape == (0, 5)
    assert ops.tri_inverse(zL).shape == (0, n, n)
    assert ops.gauss_stats_bwd(torch.empty(0, 5, device=DEV, dtype=torch.float64), z, zL, z, zL, True)[1].shape == (0, n, n)
    for kind in (0, 1):
        assert ops.cov_distance(kind, zL, zL, True).shape == (0,)
    assert ops.proj_frob_cov(zL, zL, 5e-4)[0].shape == (0, n, n)
    assert ops.proj_w2_cov(zL, zL, 2.5e-4, True)[0].shape == (0, n, n)
    P = ops.proj_kl_cov_fwd(zL, zL, 5e-4, ops.kl_state(0, n, DEV), False)[0]
    assert P.shape == (0, n, n)
    assert ops.proj_kl_cov_bwd(zL, zL, P, ops.kl_state(0, n, DEV)).shape == (0, n, n)


# ---- the BBRL agent (BlackBoxAgent) with a full-covariance policy above 64 parameters -------------------------------
BB_PROJ = dict(mean_bound=0.05, trust_region_coeff=10.0, scale_prec=True, entropy_schedule="linear",
               total_train_steps=100, target_entropy=0.0, temperature=0.7, entropy_eq=False, entropy_first=False,
               do_regression=False)


def bbrl_build(Dp, typ, cb, contextual, B=24, obs_dim=9, **agent_kw):
    torch.manual_seed(0)
    var_args = dict(std_only=False, contextual=contextual)
    if contextual:
        var_args.update(avg_neuron=32, num_hidden=1, shape=0.0)
    policy = policy_factory("BlackBoxPolicy", dim_in=obs_dim, dim_out=Dp,
                            mean_net_args=dict(avg_neuron=32, num_hidden=2, shape=0.0), variance_net_args=var_args,
                            init_method="orthogonal", out_layer_gain=0.01, act_func_hidden="leaky_relu",
                            act_func_last=None, dtype="float32", device=DEV, min_std=1e-4)
    critic = critic_factory("ValueFunction", dim_in=obs_dim, dim_out=1, hidden=dict(avg_neuron=32, num_hidden=2, shape=0.0),
                            init_method="orthogonal", out_layer_gain=1, act_func_hidden="leaky_relu",
                            act_func_last=None, dtype="float32", device=DEV)
    layer = projection_factory(typ, device=DEV, dtype="float32", action_dim=Dp, proj_type=typ, cov_bound=cb, **BB_PROJ)
    kw = dict(lr_policy=3e-4, lr_critic=1e-3, wd_policy=5e-5, wd_critic=5e-5, epochs_policy=2, epochs_critic=1,
              num_minibatchs=1, norm_advantages=True, set_variance=False, balance_check=10)
    kw.update(agent_kw)
    agent = agent_factory("BlackBoxAgent", policy=policy, critic=critic, sampler=None, projection=layer, dtype="float32",
                          device=DEV, **kw)
    g = torch.Generator().manual_seed(6)
    obs = torch.randn(B, obs_dim, generator=g).to(DEV)
    with torch.no_grad():
        mean_old, L_old = policy.policy(obs)
        mean_old = (mean_old + 0.05 * torch.randn(B, Dp, generator=g).to(DEV)).contiguous()
        Bf = B if contextual else 1
        L_old = 1.03 * L_old[:Bf] + 0.01 * torch.tril(torch.randn(Bf, Dp, Dp, generator=g), -1).to(DEV)
        L_old = L_old.expand(B, -1, -1).contiguous()
        actions = policy.sample(False, mean_old, L_old, eps=torch.randn(B, Dp, generator=g).to(DEV))
        lp_old = policy.log_prob(actions, mean_old, L_old)
        for p in policy.parameters:
            p.add_(0.02 * torch.randn(p.shape, generator=g).to(DEV))
    dataset = dict(segment_state=obs, segment_action=actions, segment_log_prob=lp_old, segment_params_mean=mean_old,
                   segment_params_L=L_old, segment_reward=torch.randn(B, generator=g).to(DEV),
                   segment_value=torch.randn(B, generator=g).to(DEV))
    return agent, dataset


@pytest.mark.parametrize("typ,mb,cb", LAYERS)
@pytest.mark.parametrize("Dp", [70, 128])
@pytest.mark.parametrize("contextual", [False, True])
def test_bbrl_epoch_matches_oracle(typ, mb, cb, Dp, contextual):
    """One BlackBoxAgent policy epoch: loss terms, the 12 logging KLs and every parameter gradient."""
    agent, dataset = bbrl_build(Dp, typ, cb, contextual)
    policy, layer = agent.policy, agent.projection
    dataset = agent.process_dataset(dataset)
    odata = {k: f64(v) for k, v in dataset.items()}
    layer.initial_entropy = policy.entropy([dataset["segment_params_mean"], dataset["segment_params_L"]]).mean()
    params0 = [p.detach().clone() for p in policy.parameters]
    metrics = agent.policy_epoch(dataset, None, None).cpu()
    grads = [p.grad.detach().double().cpu() for p in policy.parameters]
    mean_net = copy.deepcopy(policy.mean_net).cpu().double()
    n_mean = len(list(mean_net.parameters()))
    with torch.no_grad():
        for p, p0 in zip(mean_net.parameters(), params0):
            p.copy_(p0.double().cpu())
    if contextual:
        var_net = copy.deepcopy(policy.variance_net).cpu().double()
        with torch.no_grad():
            for p, p0 in zip(var_net.parameters(), params0[n_mean:]):
                p.copy_(p0.double().cpu())
        opolicy = opol.BlackBoxPolicy(Dp, mean_net=mean_net, variance_net=var_net, contextual=True, min_std=1e-4)
        wrt = list(mean_net.parameters()) + list(var_net.parameters())
    else:
        cov_vec = params0[-1].double().cpu().requires_grad_(True)
        opolicy = opol.BlackBoxPolicy(Dp, mean_net=mean_net, cov_vector=cov_vec, contextual=False, min_std=1e-4)
        wrt = list(mean_net.parameters()) + [cov_vec]
    olayer = oproj.projection_factory(typ, dtype=torch.float64, action_dim=Dp, proj_type=typ, cov_bound=cb, **BB_PROJ)
    olayer.initial_entropy = f64(layer.initial_entropy)
    loss, parts = oa.policy_epoch_bbrl(opolicy, olayer, odata, 0, set_variance=False, with_metrics=True)
    ograds = torch.autograd.grad(loss, wrt)
    assert abs(metrics[0].item() - parts["surrogate_loss"].item()) <= 1e-4
    assert abs(metrics[2].item() - parts["trust_region_loss"].item()) <= 1e-4 * max(1.0, abs(parts["trust_region_loss"].item()))
    assert abs(metrics[4].item() - parts["entropy"].item()) <= 1e-4 * max(1.0, abs(parts["entropy"].item()))
    for i, key in enumerate(_KL_KEYS):
        ref = parts["kl"][key].item()
        assert abs(metrics[7 + i].item() - ref) <= 1e-4 * max(1.0, abs(ref)), key
    for g, og in zip(grads, ograds):
        assert (g - og).abs().max() <= 1e-3 * max(1e-3, og.abs().max().item())


@pytest.mark.parametrize("typ,mb,cb", LAYERS)
def test_bbrl_update_policy_eager_and_graph(typ, mb, cb):
    """update_policy at Dp = 112, eager and CUDA-graph, from the same start: the same parameters come out."""
    out = []
    for use_graph in (False, True):
        agent, dataset = bbrl_build(112, typ, cb, False, use_cuda_graph=use_graph)
        agent.num_iterations = 2                           # no balance check: graph replay when requested
        dataset = agent.process_dataset(dataset)
        p0 = [p.detach().clone() for p in agent.policy.parameters]
        res = agent.update_policy(dataset)
        assert (agent._graph is not None) == use_graph          # the epochs were replayed from a captured graph
        assert res["policy_loss_mean"] == res["policy_loss_mean"]
        assert any((p - q).abs().max() > 0 for p, q in zip(agent.policy.parameters, p0))
        out.append([p.detach().clone() for p in agent.policy.parameters])
    for a, b in zip(*out):
        assert (a - b).abs().max() <= 1e-5 * max(1.0, a.abs().max().item())


@pytest.mark.parametrize("n", [65, 128])
def test_waves_match_single_matrix_calls(n):
    """A batch of 149 matrices runs as two launches (at most as many CTAs as SMs); every op gives each matrix exactly what a
    call on that matrix alone gives (same kernel, same arithmetic: only the slice and the batch offset differ)."""
    B = 149
    m, L, mo, Lo = draw(B, n, True, seed=11)
    m, L, mo, Lo = m.to(DEV), L.to(DEV), mo.to(DEV), Lo.to(DEV)
    G = torch.tril(torch.randn(B, n, n, generator=torch.Generator().manual_seed(5))).to(DEV)
    g5 = torch.randn(B, 5, generator=torch.Generator().manual_seed(6), dtype=torch.float64).to(DEV)
    gv = torch.randn(B, generator=torch.Generator().manual_seed(7), dtype=torch.float64).to(DEV)

    def run(sl):
        out = {"stats": ops.gauss_stats(m[sl], L[sl], mo[sl], Lo[sl]), "inv": ops.tri_inverse(Lo[sl])}
        out["stats_g"] = ops.gauss_stats_bwd(g5[sl], m[sl], L[sl], mo[sl], Lo[sl], True)
        for kind, sp in ((0, False), (1, False), (1, True)):
            out[f"dist{kind}{sp}"] = ops.cov_distance(kind, L[sl], Lo[sl], sp)
            out[f"dist{kind}{sp}_g"] = ops.cov_distance_bwd(gv[sl], kind, L[sl], Lo[sl], sp)
        Pf, scf = ops.proj_frob_cov(L[sl], Lo[sl], 5e-4)[:2]
        out["frob"], out["frob_g"] = Pf, ops.proj_frob_cov_bwd(G[sl], L[sl], Lo[sl], Pf, scf, 5e-4)
        out["w2"] = ops.proj_w2_cov(L[sl], Lo[sl], 2.5e-4, True)[0]
        out["w2_g"] = ops.proj_w2_cov_bwd(G[sl], L[sl], Lo[sl], 2.5e-4, True)
        state = ops.kl_state(L[sl].shape[0], n, DEV)
        Pk = ops.proj_kl_cov_fwd(L[sl], Lo[sl], 5e-4, state, False)[0]
        out["kl"], out["kl_g"] = Pk, ops.proj_kl_cov_bwd(G[sl], L[sl], Pk, state)
        return out

    whole = run(slice(0, B))
    for b in (0, 1, 147, 148):                            # first and last matrix of each wave
        single = run(slice(b, b + 1))
        for k, v in single.items():
            for x, y in zip(v if isinstance(v, tuple) else (v,), whole[k] if isinstance(v, tuple) else (whole[k],)):
                assert torch.equal(x[0], y[b]), (k, b)


@pytest.mark.parametrize("n", [70, 128])
def test_fused_head_chain_above_64(n):
    """The shared-covariance chain with the policy head fused in, above n = 64: the factor built from the covariance
    vector, the state's Sigma_proj against the oracle, and the covariance-space backward with K = L~^-T U~ from
    tce_proj_kl_bwd_prep (w.r.t. the vector and w.r.t. the factor) against the oracle's autograd and against the
    backward without K."""
    p, min_std = ops._p, 1e-4
    g = torch.Generator().manual_seed(n)
    nv = n + n * (n - 1) // 2
    vec = torch.cat([0.6 + 0.1 * torch.randn(n, generator=g, dtype=torch.float64),
                     0.03 / n ** 0.5 * torch.randn(nv - n, generator=g, dtype=torch.float64)])
    vec64 = vec.clone().requires_grad_(True)
    r, c = torch.tril_indices(n, n, -1)

    def head(v):                                          # abstract_policy.py:166-187
        Lh = torch.diag_embed(torch.nn.functional.softplus(v[:n]) + min_std)
        return Lh.index_put((r, c), v[n:])

    Lref = head(vec64)
    Lo = (head(vec.detach()) * 1.05).float()
    S_ref = oproj.kl_cov_projection(Lref[None], Lo.double()[None], 5e-4)[0][0]
    work = torch.empty(max(_lib.load().tce_proj_work_bytes(1, n) // 8, 1), device=DEV, dtype=torch.float64)
    vec_d, Lod = vec.float().to(DEV), Lo.to(DEV)[None].contiguous()
    L_new = torch.empty(1, n, n, device=DEV)
    out = torch.empty(2, n, n, device=DEV)
    info = torch.empty(1, device=DEV, dtype=torch.int32)
    state = ops.kl_state(1, n, DEV)
    s = torch.cuda.current_stream().cuda_stream
    _lib.call("tce_proj_kl_entropy_fwd_sigma_vec_ws", p(vec_d), 0, min_std, p(L_new), p(Lod), 5e-4, None, 0, 0,
              p(out[0]), p(out[1]), p(state), p(info), 0, 1, n, p(work), s)
    assert (f64(L_new[0]) - Lref.detach()).abs().max() <= 1e-6
    sig0 = f64(ops.kl_state_sigma(state, 1, n)[0][0])
    assert (sig0 - S_ref.detach()).abs().max() <= 1e-4 * max(1.0, S_ref.abs().max().item())
    gS = torch.randn(n, n, generator=g, dtype=torch.float64)
    gS = 0.5 * (gS + gS.T)
    (gvec_ref,) = torch.autograd.grad((S_ref * gS).sum(), [vec64])
    gS_d = gS.to(DEV)[None].contiguous()
    g_noK = torch.empty(1, n, n, device=DEV)
    _lib.call("tce_proj_kl_bwd_sigma_ws", p(L_new), p(gS_d), p(state), 1, 0.0, p(g_noK), 1, n, p(work), s)
    _lib.call("tce_proj_kl_bwd_prep_ws", p(state), 1, n, p(work), s)
    g_K = torch.empty(1, n, n, device=DEV)
    _lib.call("tce_proj_kl_bwd_sigma_k_ws", p(L_new), p(gS_d), p(state), 1, 0.0, p(g_K), 1, n, p(work), s)
    gvec = torch.full((nv,), float("nan"), device=DEV)
    _lib.call("tce_proj_kl_bwd_sigma_k_vec_ws", p(L_new), p(vec_d), 0, p(gS_d), p(state), 1, 0.0, p(gvec), 1, n,
              p(work), s)
    torch.cuda.synchronize()
    scale = max(1.0, gvec_ref.abs().max().item())
    assert (f64(gvec) - gvec_ref).abs().max() <= 2e-3 * scale
    assert (f64(g_K) - f64(g_noK)).abs().max() <= 1e-5 * max(1.0, f64(g_noK).abs().max().item())
    sig = torch.sigmoid(vec[:n])
    gL = f64(g_K[0])
    assert (torch.cat([gL.diagonal() * sig, gL[r, c]]) - f64(gvec)).abs().max() <= 1e-5 * scale

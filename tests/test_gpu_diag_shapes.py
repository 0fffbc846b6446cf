"""Diagonal-covariance (std_only) policies at every ProDMP shape the tables accept, past the 64 parameters of the
full-covariance path: the diagonal likelihood up to Dp = 128, the diagonal Gaussian scalars / Frobenius / W2 / distance
kernels, and the policy epochs of both agents, against the fp64 CPU oracle (and, at a compiled shape, against the dense
kernels each diagonal kernel replaces)."""
import copy

import pytest
import torch

from oracle import agent as oa
from oracle import policy as opol
from oracle import projection as oproj
from oracle import projection_diag as oproj_diag
from oracle import util as ou
from oracle.gen_golden import MP_CONFIGS, NUM_TIMES

pytestmark = pytest.mark.gpu
if torch.cuda.is_available():
    from tce_rl_b200 import _lib, ops
    from tce_rl_b200._lib import TceError
    from tce_rl_b200.rl import (TemporalCorrelatedAgent, agent_factory, critic_factory, policy_factory,
                                projection_factory)
    from tce_rl_b200.rl.agent import _KL_KEYS, SegmentTimeSampler

DEV = "cuda:0"
SHAPES = [(7, 10), (5, 13), (6, 16), (8, 16), (7, 9)]          # (num_dof, K1): Dp = 70, 65, 96, 128 and a compiled one
KL_KW = dict(proj_type="kl", mean_bound=0.05, cov_bound=5e-4, trust_region_coeff=1.0, scale_prec=True,
             total_train_steps=7500, target_entropy=0.0, temperature=0.7, entropy_eq=False, entropy_first=False,
             do_regression=False)
LAYERS = {"KLProjectionLayer": (0.05, 5e-4), "FrobeniusProjectionLayer": (0.05, 5e-4),
          "WassersteinProjectionLayer": (0.005, 2.5e-4)}
# entry points that hold n x n matrices (the full-covariance path): none may run in a std_only epoch
DENSE = {"tce_gauss_stats", "tce_gauss_stats_bwd", "tce_gauss_maha", "tce_gauss_maha_bwd_full", "tce_tri_inverse",
         "tce_gauss_maha_shared", "tce_proj_frob_cov_fwd", "tce_proj_frob_cov_bwd", "tce_proj_w2_cov_fwd",
         "tce_proj_w2_cov_bwd", "tce_cov_distance", "tce_proj_kl_cov_fwd", "tce_proj_kl_cov_bwd",
         "tce_proj_kl_entropy_fwd", "tce_proj_kl_entropy_bwd", "tce_chol_fwd", "tce_chol_bwd", "tce_seglik_gram",
         "tce_seglik_chol", "tce_seglik_bwd", "tce_seglik_fused", "tce_seglik_prepass"}


def f64(t):
    return t.detach().double().cpu()


def mp_cfg(D, K1):
    return dict(MP_CONFIGS["box"], num_dof=D, num_basis=K1 - 1), NUM_TIMES["box"]


def sigmas(B, n, seed, spread=0.1):
    g = torch.Generator().manual_seed(seed)
    s_old = torch.exp(0.3 * torch.randn(B, n, generator=g))
    return s_old * torch.exp(spread * torch.randn(B, n, generator=g)), s_old


# ---- likelihood ----------------------------------------------------------------------------------------------------
def lik_inputs(D, K1, B, P, ragged, seed=1234):
    cfg, T = mp_cfg(D, K1)
    Dp = D * K1
    g = torch.Generator().manual_seed(seed)
    mean = 0.5 * torch.randn(B, Dp, generator=g)
    s, _ = sigmas(B, Dp, seed + 1, spread=0.2)
    init_time = torch.rand(B, generator=g) * 0.3                                 # per episode
    init_pos, init_vel = torch.rand(B, D, generator=g) * 2 - 1, 0.1 * torch.randn(B, D, generator=g)
    eps = torch.randn(B, Dp, generator=g)
    times = ou.get_times(init_time.double(), T, cfg["dt"]).float()
    pairs = (torch.tensor([[0, 1], [0, 99], [5, 50], [98, 99], [10, 11], [11, 12], [40, 80]]) if ragged
             else ou.get_time_pairs(T, dict(num_select=P + 1, fixed_interval=True))[:P])
    return cfg, dict(mean=mean, s=s, init_time=init_time, init_pos=init_pos, init_vel=init_vel, eps=eps, times=times,
                     pairs=pairs)


@pytest.mark.parametrize("D,K1", SHAPES)
@pytest.mark.parametrize("B,P,ragged,layout", [(1024, 24, False, "dense"), (33, 25, False, "packed"),
                                               (1, 25, False, "shared"), (17, 7, True, "shared"),
                                               (64, 25, False, "shared")])
def test_diag_likelihood_matches_oracle(D, K1, B, P, ragged, layout):
    Dp = D * K1
    cfg, inp = lik_inputs(D, K1, B, P, ragged)
    if layout == "shared":
        inp["s"] = inp["s"][:1].expand(B, -1)
    L64 = torch.diag_embed(inp["s"].double())
    pol = opol.TemporalCorrelatedPolicy(Dp, mp=dict(type="prodmp", args=dict(cfg, dtype=torch.float64)),
                                        contextual=layout != "shared", std_only=True, min_std=1e-4)
    args64 = (inp["times"].double(), inp["init_time"].double(), inp["init_pos"].double(), inp["init_vel"].double())
    smp = pol.sample(False, inp["mean"].double(), L64, *args64, eps=inp["eps"].double()).float()
    mean64 = inp["mean"].double().requires_grad_(True)
    s64 = (inp["s"][:1] if layout == "shared" else inp["s"]).double().requires_grad_(True)
    lp = pol.log_prob(smp.double(), mean64, torch.diag_embed(s64).expand(B, -1, -1), *args64, pred_pairs=inp["pairs"])
    w = torch.linspace(0.5, 1.5, lp.numel(), dtype=torch.float64).reshape(lp.shape)
    gm, gs = torch.autograd.grad((lp * w).sum(), [mean64, s64])

    tabs = ops.Tables(**cfg)
    c = lambda t: t.to(DEV)
    args = (c(inp["times"]), c(inp["init_time"]), c(inp["init_pos"]), c(inp["init_vel"]), c(inp["pairs"]), tabs)
    s_dev = c(inp["s"][:1] if layout == "shared" else inp["s"]).requires_grad_(True)
    if layout == "dense":
        L = torch.diag_embed(s_dev)
    elif layout == "packed":                    # [B, n] vectors seen as [B, n, n] diagonals: inc = 1
        L = torch.as_strided(s_dev, (B, Dp, Dp), (Dp, 0, 1))
    else:                                       # ONE [1, n, n] factor for the batch
        L = torch.diag_embed(s_dev)
    mean_g = c(inp["mean"]).requires_grad_(True)
    got, info, _ = ops.seg_logprob_diag(c(smp), mean_g, L, *args, return_info=True)
    assert got.shape == (B, P) and int(info.abs().max()) == 0
    assert (f64(got) - lp.detach()).abs().max() <= 1e-4
    (got * c(w.float())).sum().backward()
    assert (f64(mean_g.grad) - gm).abs().max() <= 2e-4 * gm.abs().max()
    assert (f64(s_dev.grad) - gs).abs().max() <= 2e-4 * gs.abs().max()
    if (D, K1) == (7, 9) and layout == "dense":   # the dense staged kernels on the same diagonal factors
        dense = ops.seg_logprob_staged(c(smp), mean_g.detach(), torch.diag_embed(s_dev.detach()).contiguous(), *args)
        assert (dense - got).abs().max().item() <= 1e-4


@pytest.mark.parametrize("D,K1", [(7, 10), (8, 16)])
def test_diag_likelihood_empty_batch(D, K1):
    cfg, inp = lik_inputs(D, K1, 0, 24, False)
    tabs = ops.Tables(**cfg)
    c = lambda t: t.to(DEV)
    mean = c(inp["mean"]).requires_grad_(True)
    L = torch.zeros(0, D * K1, D * K1, device=DEV, requires_grad=True)
    lp = ops.seg_logprob_diag(torch.zeros(0, NUM_TIMES["box"], 2 * D, device=DEV), mean, L, c(inp["times"]),
                              c(inp["init_time"]), c(inp["init_pos"]), c(inp["init_vel"]), c(inp["pairs"]), tabs)
    assert lp.shape == (0, 24)
    lp.sum().backward()
    assert mean.grad.shape == (0, D * K1)


def test_full_covariance_policy_above_64_parameters_raises():
    D, K1 = 7, 10
    cfg, T = mp_cfg(D, K1)
    B, Dp = 4, D * K1
    tabs = ops.Tables(**cfg)
    assert not tabs.dense_likelihood
    z = lambda *s: torch.zeros(*s, device=DEV)
    pairs = ou.get_time_pairs(T, dict(num_select=26, fixed_interval=True))[:25].to(DEV)
    policy = tce_policy(cfg, Dp, contextual=True, std_only=False)
    mean, L = policy.policy(z(B, 10))
    with pytest.raises(TceError, match="unsupported"):
        policy.log_prob(z(B, T, 2 * D), mean, L, z(B, T), z(B), z(B, D), z(B, D), pred_pairs=pairs)


# ---- diagonal Gaussian kernels -------------------------------------------------------------------------------------
NS = [12, 63, 65, 128, 500]


def kernel_case(n, B, old, equal=False, seed=5):
    s, s_old = sigmas(B, n, seed)
    if equal:
        s = torch.full((B, n), 0.9)
    if old == "shared":
        s_old = s_old[:1]
    g = torch.Generator().manual_seed(seed + 2)
    mean, mean_o = torch.randn(B, n, generator=g), torch.randn(B, n, generator=g)
    return s, s_old, mean, mean_o


@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("old,equal", [("per_episode", False), ("shared", False), ("per_episode", True)])
def test_gauss_stats_and_maha_diag_match_oracle(n, old, equal):
    B = 37
    s, s_old, mean, mean_o = kernel_case(n, B, old, equal)
    L64, Lo64 = torch.diag_embed(s.double()).requires_grad_(True), torch.diag_embed(s_old.double())
    m64 = mean.double().requires_grad_(True)
    pol = opol.BlackBoxPolicy(n, std_only=True, contextual=True, min_std=1e-4)
    Lo64b = Lo64.expand(B, -1, -1)
    maha = pol.maha(m64, mean_o.double(), Lo64b)
    tr = oproj.batched_trace(pol.precision(Lo64b) @ pol.covariance(L64))
    ld, ldo = pol.log_determinant(L64), pol.log_determinant(Lo64b)
    ent = pol.entropy([m64, L64])
    ref = torch.stack([maha, tr, ld, ldo, ent], -1)
    w = torch.randn(B, 5, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    gm, gL = torch.autograd.grad((ref * w).sum(), [m64, L64])

    c = lambda t: t.to(DEV)
    mg, Lg = c(mean).requires_grad_(True), c(torch.diag_embed(s)).requires_grad_(True)
    st = ops.gauss_stats_diag(mg, Lg, c(mean_o), c(torch.diag_embed(s_old)))
    assert (f64(st) - ref.detach()).abs().max() <= 1e-4 * max(1.0, ref.abs().max().item())
    (st * c(w)).sum().backward()
    assert (f64(mg.grad) - gm).abs().max() <= 2e-4 * gm.abs().max()
    assert (f64(Lg.grad) - gL.diagonal(dim1=-2, dim2=-1).diag_embed()).abs().max() <= 2e-4 * gL.abs().max()
    # the Mahalanobis mode and zero means
    mg2 = c(mean).requires_grad_(True)
    mh = ops.gauss_maha_diag(mg2, c(mean_o), c(torch.diag_embed(s_old)))
    assert (f64(mh) - maha.detach()).abs().max() <= 1e-4 * max(1.0, maha.abs().max().item())
    (mh * c(w[:, 0])).sum().backward()
    assert (f64(mg2.grad) - gm).abs().max() <= 2e-4 * gm.abs().max()
    z = ops.gauss_stats_diag(None, c(torch.diag_embed(s)), None, c(torch.diag_embed(s_old)))
    assert float(z[:, 0].abs().max()) == 0.0 and torch.allclose(z[:, 1:], st[:, 1:].detach())
    if n <= 64:                                       # the dense kernels it replaces
        Lo_dense = c(torch.diag_embed(s_old.expand(B, -1)).contiguous())
        dense = ops.gauss_stats(c(mean), c(torch.diag_embed(s)), c(mean_o), Lo_dense)
        assert (dense - st).abs().max().item() <= 1e-6 * max(1.0, dense.abs().max().item())
        assert (ops.gauss_maha(c(mean), c(mean_o), Lo_dense) - mh).abs().max().item() <= 1e-6 * mh.abs().max().item()


def _proj_oracle(kind, L64, Lo64, eps, scale_prec):
    layer = oproj.FrobeniusProjectionLayer if kind == 0 else oproj.WassersteinProjectionLayer
    pol = opol.BlackBoxPolicy(L64.shape[-1], std_only=True, contextual=True, min_std=1e-4)
    mean = torch.zeros(L64.shape[0], L64.shape[-1], dtype=torch.float64)
    lay = layer(scale_prec=scale_prec, cpu=True, dtype=torch.float64)
    return lay._trust_region_projection(pol, (mean, L64), (mean, Lo64), 1.0, eps)[1]


@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("kind,scale_prec", [(0, False), (1, True), (1, False)])
@pytest.mark.parametrize("old,equal", [("per_episode", False), ("shared", False), ("per_episode", True)])
def test_frob_w2_projection_and_distance_diag_match_oracle(n, kind, scale_prec, old, equal):
    B = 9
    s, s_old, _, _ = kernel_case(n, B, old, equal, seed=n)
    s[0] = s_old[0] * (1 + 1e-5)                      # inside the trust region: identity branch
    eps = 1e-2 if kind == 0 else 2e-3
    Lo64 = torch.diag_embed(s_old.double()).expand(B, -1, -1)
    L64 = torch.diag_embed(s.double()).requires_grad_(True)
    proj = _proj_oracle(kind, L64, Lo64, eps, scale_prec)
    dist = oproj.gaussian_frobenius if kind == 0 else oproj.gaussian_wasserstein_commutative
    zeros = torch.zeros(B, n, dtype=torch.float64)
    polo = opol.BlackBoxPolicy(n, std_only=True, contextual=True, min_std=1e-4)
    cp = dist(polo, (zeros, L64), (zeros, Lo64), scale_prec if kind == 1 else False)[1]
    w = torch.randn(B, n, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    wd = torch.linspace(0.5, 1.5, B, dtype=torch.float64)
    gP, = torch.autograd.grad((proj.diagonal(dim1=-2, dim2=-1) * w).sum(), L64)
    gD, = torch.autograd.grad((cp * wd).sum(), L64)

    c = lambda t: t.to(DEV)
    Lg, Lo = c(torch.diag_embed(s)).requires_grad_(True), c(torch.diag_embed(s_old))
    if kind == 0:
        out, sc, info = ops.proj_frob_diag(Lg, Lo, eps)
        assert int(info.abs().max()) == 0
    else:
        out, sc = ops.proj_w2_diag(Lg, Lo, eps, scale_prec)
    assert sc[0, 1].item() == 0.0 and bool((sc[1:, 1] == 1.0).all())     # one identity, the rest projected
    assert (f64(out) - proj.detach()).abs().max() <= 1e-4 * max(1.0, proj.abs().max().item())
    (out.diagonal(dim1=-2, dim2=-1) * c(w.float())).sum().backward()
    assert (f64(Lg.grad).diagonal(dim1=-2, dim2=-1) - gP.diagonal(dim1=-2, dim2=-1)).abs().max() <= \
        1e-3 * gP.abs().max()
    Lg2 = c(torch.diag_embed(s)).requires_grad_(True)
    val = ops.cov_distance_diag(kind, Lg2, Lo, scale_prec)
    assert (f64(val) - cp.detach()).abs().max() <= 1e-4 * max(1.0, cp.abs().max().item())
    (val * c(wd)).sum().backward()
    assert (f64(Lg2.grad).diagonal(dim1=-2, dim2=-1) - gD.diagonal(dim1=-2, dim2=-1)).abs().max() <= \
        2e-4 * gD.abs().max()
    if n <= 64:                                       # the dense kernels they replace
        Lo_d = c(torch.diag_embed(s_old.expand(B, -1)).contiguous())
        dense = (ops.proj_frob_cov(c(torch.diag_embed(s)), Lo_d, eps)[0] if kind == 0 else
                 ops.proj_w2_cov(c(torch.diag_embed(s)), Lo_d, eps, scale_prec)[0])
        assert (dense - out).abs().max().item() <= 1e-5 * dense.abs().max().item()
        dd = ops.cov_distance(kind, c(torch.diag_embed(s)), Lo_d, scale_prec)
        assert (dd - val).abs().max().item() <= 1e-6 * max(1.0, dd.abs().max().item())


def test_diag_kernels_take_an_empty_batch():
    L = torch.zeros(0, 70, 70, device=DEV)
    assert ops.gauss_stats_diag(None, L, None, L).shape == (0, 5)
    assert ops.proj_frob_diag(L, L, 1e-3)[0].shape == (0, 70, 70)
    assert ops.proj_w2_diag(L, L, 1e-3, True)[0].shape == (0, 70, 70)
    assert ops.cov_distance_diag(1, L, L, True).shape == (0,)


# ---- policy epochs -------------------------------------------------------------------------------------------------
def tce_policy(cfg, Dp, contextual, std_only=True, obs_dim=10, seed=0):
    torch.manual_seed(seed)
    return policy_factory("TemporalCorrelatedPolicy", dim_in=obs_dim, dim_out=Dp,
                          mean_net_args=dict(avg_neuron=32, num_hidden=2, shape=0.0),
                          variance_net_args=dict(std_only=std_only, contextual=contextual, avg_neuron=32, num_hidden=2,
                                                 shape=0.0),
                          init_method="orthogonal", out_layer_gain=0.01, act_func_hidden="leaky_relu",
                          act_func_last=None, dtype="float32", device=DEV, min_std=1e-4,
                          mp=dict(type="prodmp", args=dict(cfg)))


def epoch_setup(D, K1, typ, contextual, B=24, obs_dim=10):
    cfg, T = mp_cfg(D, K1)
    Dp = D * K1
    mb, cb = LAYERS[typ]
    kw = dict(KL_KW, proj_type=typ, mean_bound=mb, cov_bound=cb, entropy_schedule="linear", action_dim=Dp)
    policy = tce_policy(cfg, Dp, contextual, obs_dim=obs_dim)
    with torch.no_grad():
        for p in policy.parameters:
            p.add_(0.02 * torch.randn_like(p))
    layer = projection_factory(typ, device=DEV, dtype="float32", **kw)
    sampler = SegmentTimeSampler(cfg["dt"], T, dict(num_select=25, fixed_interval=True), device=DEV)
    torch.manual_seed(2)
    pairs = sampler.get_time_pairs()
    agent = TemporalCorrelatedAgent(policy, None, sampler, layer, dtype="float32", device=DEV, lr_policy=1e-4,
                                    lr_critic=1e-3, wd_policy=5e-5, wd_critic=5e-5, discount_factor=1.0,
                                    epochs_policy=1, epochs_critic=1, norm_advantages=True,
                                    segment_advantage="value_subtraction", set_variance=False)
    c = lambda t: t.to(DEV)
    g = torch.Generator().manual_seed(4)
    obs = torch.randn(B, obs_dim + 2 * D, generator=g)
    init_time = torch.rand(B, generator=g) * 0.3
    init_pos, init_vel = torch.rand(B, D, generator=g) * 2 - 1, 0.1 * torch.randn(B, D, generator=g)
    times = sampler.get_times(c(init_time), T)
    with torch.no_grad():
        mean_old, L_old = policy.policy(c(obs)[..., :-2 * D])
        mean_old = mean_old + 0.05 * c(torch.randn(B, Dp, generator=g))
        L_old = L_old * torch.diag_embed(torch.exp(0.05 * c(torch.randn(B if contextual else 1, Dp, generator=g))))
        if not contextual:
            L_old = L_old[:1].expand(B, -1, -1).contiguous()
        smp = policy.sample(False, mean_old, L_old, times, c(init_time), c(init_pos), c(init_vel),
                            eps=c(torch.randn(B, Dp, generator=g)))
        lp_old = policy.log_prob(smp, mean_old, L_old, times, c(init_time), c(init_pos), c(init_vel), pred_pairs=pairs)
        rewards, values = torch.randn(B, T, generator=g), torch.randn(B, T + 1, generator=g)
        dones = torch.zeros(B, T, dtype=torch.bool)
        dones[:, -1] = True
        adv, _ = agent.get_advantage_return(c(rewards), c(values), c(dones), c(torch.zeros(B, T, dtype=torch.bool)))
        seg_adv = agent.get_segment_advantage(c(rewards), c(values), adv, pairs)
    dataset = dict(segment_state=c(obs), step_actions=smp, segment_log_prob_estimate=lp_old,
                   segment_params_mean=mean_old, segment_params_L=L_old, segment_advantage=seg_adv,
                   segment_init_time=c(init_time), segment_init_pos=c(init_pos), segment_init_vel=c(init_vel))
    layer.initial_entropy = policy.entropy([mean_old, L_old]).mean()
    return cfg, kw, policy, layer, agent, dataset, times, pairs


@pytest.mark.parametrize("D,K1", [(7, 10), (8, 16)])
@pytest.mark.parametrize("typ", list(LAYERS))
@pytest.mark.parametrize("contextual", [True, False])
def test_std_only_policy_epoch_matches_oracle(D, K1, typ, contextual):
    Dp = D * K1
    cfg, kw, policy, layer, agent, dataset, times, pairs = epoch_setup(D, K1, typ, contextual)
    params0 = [p.detach().clone() for p in policy.parameters]
    agent.ensure_flat_grads(agent.policy_net_params)          # as update_policy: one flat gradient + FlatAdam
    agent._use_flat_adam()
    launched = []
    call = _lib.call

    def recording_call(name, *args):
        launched.append(name)
        return call(name, *args)
    _lib.call = recording_call
    try:
        metrics = agent.policy_epoch(dataset, times, pairs).cpu()
    finally:
        _lib.call = call
    assert not DENSE & set(launched), sorted(DENSE & set(launched))
    assert agent._fast is None
    grads = [p.grad.detach().double().cpu() for p in policy.parameters]

    mean_net = copy.deepcopy(policy.mean_net).cpu().double()
    var_net = copy.deepcopy(policy.variance_net).cpu().double() if contextual else None
    with torch.no_grad():
        for p, p0 in zip(list(mean_net.parameters()) + (list(var_net.parameters()) if contextual else []), params0):
            p.copy_(p0.double().cpu())
    cov_vec = None if contextual else params0[-1].double().cpu().requires_grad_(True)
    opolicy = opol.TemporalCorrelatedPolicy(Dp, mp=dict(type="prodmp", args=dict(cfg, dtype=torch.float64)),
                                            mean_net=mean_net, variance_net=var_net, cov_vector=cov_vec,
                                            contextual=contextual, std_only=True, min_std=1e-4)
    olayer = oproj_diag.projection_factory(typ, dtype=torch.float64, **kw)
    olayer.initial_entropy = f64(layer.initial_entropy)
    odata = {k: (f64(v) if v.is_floating_point() else v.cpu()) for k, v in dataset.items()}
    loss, parts = oa.policy_epoch(opolicy, olayer, odata, f64(times), pairs.cpu(), 0, set_variance=False,
                                  with_metrics=True)
    oparams = list(mean_net.parameters()) + (list(var_net.parameters()) if contextual else [cov_vec])
    ograds = torch.autograd.grad(loss, oparams)
    assert abs(metrics[0].item() - parts["surrogate_loss"].item()) <= 1e-4
    assert abs(metrics[2].item() - parts["trust_region_loss"].item()) <= 1e-4
    assert abs(metrics[3].item() - loss.item()) <= 2e-4
    assert abs(metrics[4].item() - parts["entropy"].item()) <= 1e-4 * max(1.0, abs(parts["entropy"].item()))
    assert abs(metrics[5].item() - parts["imp_smp_ratio"].item()) <= 1e-4
    for i, key in enumerate(_KL_KEYS):
        assert abs(metrics[7 + i].item() - parts["kl"][key].item()) <= 1e-4, key
    for gr, og in zip(grads, ograds):
        assert (gr - og).abs().max() <= 1e-3 * max(1e-3, og.abs().max().item())


def build_update(typ, contextual, use_graph, D=7, K1=10, B=64, epochs=3):
    cfg, T = mp_cfg(D, K1)
    Dp, obs_dim = D * K1, 12
    mb, cb = LAYERS[typ]
    torch.manual_seed(0)
    policy = tce_policy(cfg, Dp, contextual, obs_dim=obs_dim)
    critic = critic_factory("ValueFunction", dim_in=obs_dim, dim_out=1, hidden=dict(avg_neuron=32, num_hidden=2, shape=0.0),
                            init_method="orthogonal", out_layer_gain=1, act_func_hidden="leaky_relu",
                            act_func_last=None, dtype="float32", device=DEV)
    proj = projection_factory(typ, **dict(KL_KW, mean_bound=mb, cov_bound=cb, entropy_schedule="linear",
                                          action_dim=Dp, total_train_steps=100), dtype="float32", device=DEV)
    sampler = SegmentTimeSampler(cfg["dt"], T, dict(num_select=25, fixed_interval=True), device=DEV)
    torch.manual_seed(1)
    pairs = sampler.get_time_pairs()
    agent = TemporalCorrelatedAgent(policy, critic, sampler, proj, dtype="float32", device=DEV, lr_policy=3e-4,
                                    lr_critic=1e-3, wd_policy=5e-5, wd_critic=5e-5, discount_factor=1.0,
                                    epochs_policy=epochs, epochs_critic=2, num_minibatchs=2, norm_advantages=True,
                                    segment_advantage="value_subtraction", set_variance=False, gae_scaling=0.95,
                                    use_cuda_graph=use_graph, schedule_lr_policy=True, schedule_lr_critic=True)
    c = lambda t: t.to(DEV)
    g = torch.Generator().manual_seed(5)
    obs = torch.randn(B, obs_dim + 2 * D, generator=g)
    step_states = torch.randn(B, T, obs_dim + 2 * D, generator=g)
    init_time = torch.zeros(B)
    init_pos, init_vel = torch.rand(B, D, generator=g) * 2 - 1, 0.1 * torch.randn(B, D, generator=g)
    dones = torch.zeros(B, T, dtype=torch.bool)
    dones[:, -1] = True
    with torch.no_grad():
        times = sampler.get_times(c(init_time), T)
        mean_old, L_old = policy.policy(c(obs)[..., :-2 * D])
        smp = policy.sample(False, mean_old, L_old, times, c(init_time), c(init_pos), c(init_vel),
                            eps=c(torch.randn(B, Dp, generator=g)))
        lp_old = policy.log_prob(smp, mean_old, L_old, times, c(init_time), c(init_pos), c(init_vel), pred_pairs=pairs)
    dataset = dict(segment_state=c(obs), step_actions=smp, segment_log_prob_estimate=lp_old,
                   segment_params_mean=mean_old.clone(), segment_params_L=L_old.clone(),
                   segment_init_time=c(init_time), segment_init_pos=c(init_pos), segment_init_vel=c(init_vel),
                   step_states=c(step_states), step_rewards=c(torch.randn(B, T, generator=g)),
                   step_values=c(torch.randn(B, T + 1, generator=g)), step_dones=c(dones),
                   step_time_limit_dones=c(torch.zeros(B, T, dtype=torch.bool)))
    return agent, dataset


@pytest.mark.parametrize("typ", list(LAYERS))
@pytest.mark.parametrize("contextual", [True, False])
def test_std_only_graph_captured_update_equals_eager(typ, contextual):
    outs, params = [], []
    for use_graph in (False, True):
        agent, dataset = build_update(typ, contextual, use_graph)
        assert agent.policy.is_diag and not agent.policy.mp.tables.dense_likelihood
        agent.num_iterations = 1
        dataset = agent.process_dataset(dataset)
        out = agent.update_policy(dataset)
        # surrogate / trust-region gradient norm: infinite when the first epoch projects nothing (a shared covariance
        # without the covariance term has a zero trust-region gradient then)
        out.pop("balance_ratio", None)
        assert all(torch.isfinite(torch.tensor(float(v))) for v in out.values())
        outs.append(out)
        params.append([p.detach().clone() for p in agent.policy.parameters])
    for k in outs[0]:
        assert abs(outs[0][k] - outs[1][k]) <= 1e-4 * max(1.0, abs(outs[0][k])), k
    for p, q in zip(*params):
        assert (p - q).abs().max().item() <= 1e-5


def test_std_only_bbrl_epoch_above_64_parameters_matches_oracle():
    B, Dp, obs_dim = 48, 70, 9
    torch.manual_seed(0)
    policy = policy_factory("BlackBoxPolicy", dim_in=obs_dim, dim_out=Dp,
                            mean_net_args=dict(avg_neuron=32, num_hidden=2, shape=0.0),
                            variance_net_args=dict(std_only=True, contextual=False), init_method="orthogonal",
                            out_layer_gain=0.01, act_func_hidden="leaky_relu", act_func_last=None, dtype="float32",
                            device=DEV, min_std=1e-4)
    kw = dict(KL_KW, trust_region_coeff=10.0, entropy_schedule="linear", total_train_steps=100, action_dim=Dp)
    layer = projection_factory("KLProjectionLayer", device=DEV, dtype="float32", **kw)
    critic = critic_factory("ValueFunction", dim_in=obs_dim, dim_out=1, hidden=dict(avg_neuron=32, num_hidden=2, shape=0.0),
                            init_method="orthogonal", out_layer_gain=1, act_func_hidden="leaky_relu",
                            act_func_last=None, dtype="float32", device=DEV)
    agent = agent_factory("BlackBoxAgent", policy=policy, critic=critic, sampler=None, projection=layer, dtype="float32",
                          device=DEV, lr_policy=3e-4, lr_critic=1e-3, wd_policy=5e-5, wd_critic=5e-5, epochs_policy=3,
                          epochs_critic=2, num_minibatchs=2, norm_advantages=True, set_variance=False)
    g = torch.Generator().manual_seed(6)
    obs = torch.randn(B, obs_dim, generator=g).to(DEV)
    with torch.no_grad():
        mean_old, L_old = policy.policy(obs)
        mean_old = (mean_old + 0.05 * torch.randn(B, Dp, generator=g).to(DEV)).contiguous()
        L_old = (L_old[:1] * torch.exp(0.03 * torch.randn(Dp, generator=g)).to(DEV)).expand(B, -1, -1).contiguous()
        actions = policy.sample(False, mean_old, L_old, eps=torch.randn(B, Dp, generator=g).to(DEV))
        lp_old = policy.log_prob(actions, mean_old, L_old)
        for p in policy.parameters:
            p.add_(0.02 * torch.randn(p.shape, generator=g).to(DEV))
    dataset = dict(segment_state=obs, segment_action=actions, segment_log_prob=lp_old, segment_params_mean=mean_old,
                   segment_params_L=L_old, segment_reward=torch.randn(B, generator=g).to(DEV),
                   segment_value=torch.randn(B, generator=g).to(DEV))
    dataset = agent.process_dataset(dataset)
    odata = {k: f64(v) for k, v in dataset.items()}
    layer.initial_entropy = policy.entropy([dataset["segment_params_mean"], dataset["segment_params_L"]]).mean()
    params0 = [p.detach().clone() for p in policy.parameters]
    metrics = agent.policy_epoch(dataset, None, None).cpu()
    grads = [p.grad.detach().double().cpu() for p in policy.parameters]
    mean_net = copy.deepcopy(policy.mean_net).cpu().double()
    with torch.no_grad():
        for p, p0 in zip(mean_net.parameters(), params0):
            p.copy_(p0.double().cpu())
    cov_vec = params0[-1].double().cpu().requires_grad_(True)
    opolicy = opol.BlackBoxPolicy(Dp, mean_net=mean_net, cov_vector=cov_vec, contextual=False, std_only=True,
                                  min_std=1e-4)
    olayer = oproj_diag.projection_factory("KLProjectionLayer", dtype=torch.float64, **kw)
    olayer.initial_entropy = f64(layer.initial_entropy)
    loss, parts = oa.policy_epoch_bbrl(opolicy, olayer, odata, 0, set_variance=False, with_metrics=True)
    ograds = torch.autograd.grad(loss, list(mean_net.parameters()) + [cov_vec])
    assert abs(metrics[0].item() - parts["surrogate_loss"].item()) <= 1e-4
    assert abs(metrics[2].item() - parts["trust_region_loss"].item()) <= 1e-4 * max(1.0, abs(parts["trust_region_loss"].item()))
    for i, key in enumerate(_KL_KEYS):
        assert abs(metrics[7 + i].item() - parts["kl"][key].item()) <= 1e-4, key
    for gr, og in zip(grads, ograds):
        assert (gr - og).abs().max() <= 1e-3 * max(1e-3, og.abs().max().item())

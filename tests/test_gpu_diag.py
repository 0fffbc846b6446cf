"""Diagonal-covariance (std_only) policies on the GPU: the diagonal policy head, the closed-form diagonal KL projection,
the block-diagonal segment likelihood and the policy epoch of both agents, against the CPU oracle (fp64) and against
the dense kernels on the same diagonal inputs."""
import copy
import os

import pytest
import torch

from oracle import agent as oa
from oracle import policy as opol
from oracle import projection_diag as oproj
from oracle import util as ou
from oracle.gen_golden import MP_CONFIGS, NUM_TIMES, synthetic_inputs

pytestmark = pytest.mark.gpu
if torch.cuda.is_available():
    from tce_rl_b200 import ops
    from tce_rl_b200.rl import (TemporalCorrelatedAgent, agent_factory, critic_factory, policy_factory,
                                projection_factory)
    from tce_rl_b200.rl.agent import _KL_KEYS, SegmentTimeSampler

DEV = "cuda:0"
KL_KW = dict(proj_type="kl", mean_bound=0.05, cov_bound=5e-4, trust_region_coeff=1.0, scale_prec=True,
             total_train_steps=7500, target_entropy=0.0, temperature=0.7, entropy_eq=False, entropy_first=False,
             do_regression=False)
LAYERS = {"KLProjectionLayer": (0.05, 5e-4), "FrobeniusProjectionLayer": (0.05, 5e-4),
          "WassersteinProjectionLayer": (0.005, 2.5e-4)}


def f64(t):
    return t.detach().double().cpu()


def dims(name):
    cfg = MP_CONFIGS[name]
    return cfg, cfg["num_dof"], cfg["num_basis"] + 1, cfg["num_dof"] * (cfg["num_basis"] + 1)


class DiagPolicy:
    """Duck-typed policy surface of a std_only policy for the projection layers."""
    is_diag = True

    def __init__(self, contextual):
        self.contextual_std = contextual

    def entropy(self, p):
        return ops.gauss_stats(p[0], p[1], p[0], p[1])[:, 4]


def diag_case(name, B, contextual, seed=3, spread=0.1):
    inp = synthetic_inputs(name, B, seed=seed, dtype=torch.float32)
    g = torch.Generator().manual_seed(seed + 1)
    Dp = inp["mean"].shape[-1]
    s_old = torch.exp(0.3 * torch.randn(B, Dp, generator=g))
    s = s_old * torch.exp(spread * torch.randn(B, Dp, generator=g))
    if not contextual:
        s, s_old = s[:1].expand(B, -1), s_old[:1].expand(B, -1)
    inp["L"], inp["L_old"] = torch.diag_embed(s).contiguous(), torch.diag_embed(s_old).contiguous()
    return inp


# ---- head --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("contextual,B", [(True, 1), (True, 300), (False, 64)])
def test_policy_head_diag_matches_oracle(contextual, B):
    n = 63
    g = torch.Generator().manual_seed(0)
    vec = torch.randn(B, n, generator=g) if contextual else torch.randn(n, generator=g)
    opolicy = opol.BlackBoxPolicy(n, std_only=True, contextual=contextual, min_std=1e-4)
    v64 = vec.double().requires_grad_(True)
    L_o = opolicy.vector_to_cholesky(v64 if contextual else v64.expand(B, -1))
    w = torch.randn(B, n, n, generator=g, dtype=torch.float64)
    gv, = torch.autograd.grad((L_o * w).sum(), v64)
    vg = vec.to(DEV).requires_grad_(True)
    L = ops.policy_head_diag(vg, B, n, 1e-4)
    assert L.shape == (B, n, n) and (f64(L) - L_o.detach()).abs().max() <= 1e-6
    assert float((L - torch.diag_embed(L.diagonal(dim1=-2, dim2=-1))).abs().max().detach()) == 0.0
    (L * w.float().to(DEV)).sum().backward()
    assert (f64(vg.grad) - gv).abs().max() <= 1e-5 * max(1.0, gv.abs().max().item())


# ---- KL projection -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("schedule", ["linear", None])
@pytest.mark.parametrize("name,contextual", [("box", True), ("box", False), ("metaworld", True),
                                              ("table_tennis", False)])
def test_kl_diag_projection_matches_oracle(name, contextual, schedule):
    B = 12
    _, _, _, Dp = dims(name)
    inp = diag_case(name, B, contextual)
    inp["mean"][0] = inp["mean_old"][0] + 1e-3
    if contextual:
        inp["L"][0] = inp["L_old"][0] * (1 + 1e-4)        # inside the trust region: identity branch
    d = lambda k: inp[k].double()
    kw = dict(KL_KW, entropy_schedule=schedule, action_dim=Dp)
    opolicy = opol.BlackBoxPolicy(Dp, std_only=True, contextual=contextual, min_std=1e-4)
    olayer = oproj.projection_factory("KLProjectionLayer", dtype=torch.float64, **kw)
    init_ent = opolicy.entropy([d("mean_old"), d("L_old")]).mean() + 0.5       # the entropy control is active
    olayer.initial_entropy = init_ent
    m64, L64 = d("mean").requires_grad_(True), d("L").requires_grad_(True)
    pm, pL = olayer(opolicy, (m64, L64), (d("mean_old"), d("L_old")), 100)
    g = torch.Generator().manual_seed(0)
    wm = torch.randn(B, Dp, generator=g, dtype=torch.float64)
    wL = torch.randn(B, Dp, Dp, generator=g, dtype=torch.float64)
    tr = olayer.get_trust_region_loss(opolicy, (m64, L64), (pm, pL), set_variance=False)
    gm, gL = torch.autograd.grad((pm * wm).sum() + (pL * wL).sum() + tr, [m64, L64])

    layer = projection_factory("KLProjectionLayer", device=DEV, dtype="float32", **kw)
    layer.initial_entropy = init_ent.float().to(DEV)
    pol = DiagPolicy(contextual)
    c = lambda k: inp[k].to(DEV)
    mg, Lg = c("mean").requires_grad_(True), c("L").requires_grad_(True)
    pmg, pLg = layer(pol, (mg, Lg), (c("mean_old"), c("L_old")), 100)
    assert (f64(pmg) - pm.detach()).abs().max() <= 1e-4
    assert (f64(pLg) - pL.detach()).abs().max() <= 1e-4
    assert float((pLg - torch.diag_embed(pLg.diagonal(dim1=-2, dim2=-1))).abs().max()) == 0.0
    trg = layer.get_trust_region_loss(pol, (mg, Lg), (pmg, pLg), set_variance=False)
    assert abs(trg.item() - tr.item()) <= 1e-4 * max(1.0, abs(tr.item()))
    ((pmg * wm.float().to(DEV)).sum() + (pLg * wL.float().to(DEV)).sum() + trg).backward()
    assert (f64(mg.grad) - gm).abs().max() <= 2e-4 * max(1.0, gm.abs().max().item())
    gL_t, gL_g = torch.diag_embed(gL.diagonal(dim1=-2, dim2=-1)), f64(Lg.grad)
    if not contextual:                                   # only the batch sum reaches the one shared factor
        gL_t, gL_g = gL_t.sum(0), gL_g.sum(0)
    assert (gL_g - gL_t).abs().max() <= 1e-3 * max(1.0, gL_t.abs().max().item())


def test_kl_diag_forward_equals_dense_kernel():
    B, n = 64, 63
    inp = diag_case("box", B, True, seed=9)
    L, Lo = inp["L"].to(DEV), inp["L_old"].to(DEV)
    dense = ops.proj_kl_cov(L, Lo, 5e-4, ops.kl_state(B, n, DEV), False)[0]
    diag, state, info = ops.proj_kl_diag(L, Lo, 5e-4, None, False)
    assert int(info.abs().max()) == 0 and bool((state[:, 1] == 1.0).all())
    assert (diag - dense).abs().max().item() <= 1e-5 * dense.abs().max().item()
    # strided layouts: packed [B, n] vectors (inc = 1) and one factor (B = 1) give the same numbers
    pk = lambda M: torch.as_strided(M.diagonal(dim1=-2, dim2=-1).contiguous(), (B, n, n), (n, 0, 1))
    packed = ops.proj_kl_diag(pk(L), pk(Lo), 5e-4, None, False)[0]
    assert torch.equal(packed, diag)
    one = ops.proj_kl_diag(L[:1], Lo[:1], 5e-4, None, False)[0]
    assert torch.equal(one[0], diag[0])


def test_kl_diag_equal_sigma_start_state_has_finite_oracle_gradients():
    """A fresh std_only policy: every sigma equal (the eigen-decomposition of the dense path has no gradient there)."""
    B, n = 4, 63
    L = torch.full((B, n), 0.9).diag_embed()
    Lo = torch.eye(n).expand(B, n, n).contiguous()
    L64 = L.double().requires_grad_(True)
    cov, act = oproj.kl_cov_projection_diag(L64, Lo.double(), 5e-4)
    assert act.all()
    w = torch.linspace(0.5, 1.5, n, dtype=torch.float64)
    out = cov.diagonal(dim1=-2, dim2=-1).sqrt()
    gL, = torch.autograd.grad((out * w).sum(), L64)
    Lg = L.to(DEV).requires_grad_(True)
    o, _, _ = ops.proj_kl_diag(Lg, Lo.to(DEV), 5e-4, None, False)
    assert (f64(o.diagonal(dim1=-2, dim2=-1)) - out.detach()).abs().max() <= 1e-6
    (o.diagonal(dim1=-2, dim2=-1) * w.float().to(DEV)).sum().backward()
    assert torch.isfinite(Lg.grad).all()
    assert (f64(Lg.grad) - gL).abs().max() <= 2e-4 * gL.abs().max().item()


# ---- likelihood ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,B,P,ragged", [("box", 1024, 24, False), ("box", 1024, 25, False),
                                             ("metaworld", 4096, 24, False), ("box", 33, 7, True),
                                             ("table_tennis", 48, 24, False)])
def test_diag_likelihood_matches_oracle_and_dense(name, B, P, ragged):
    cfg, D, K1, Dp = dims(name)
    T = NUM_TIMES[name]
    inp = diag_case(name, B, True, seed=1234, spread=0.2)
    inp["init_time"] = (torch.rand(B, generator=torch.Generator().manual_seed(7)) * 0.3).float()   # per episode
    times = ou.get_times(inp["init_time"].double(), T, cfg["dt"]).float()
    torch.manual_seed(0)
    pairs = (torch.tensor([[0, 1], [0, 99], [5, 50], [98, 99], [10, 11], [11, 12], [40, 80]]) if ragged
             else ou.get_time_pairs(T, dict(num_select=P + 1, fixed_interval=True))[:P])
    assert pairs.shape[0] == P
    pol = opol.TemporalCorrelatedPolicy(Dp, mp=dict(type="prodmp", args=dict(cfg, dtype=torch.float64)),
                                        contextual=True, std_only=True, min_std=1e-4)
    d = lambda k: inp[k].double()
    args64 = (times.double(), d("init_time"), d("init_pos"), d("init_vel"))
    smp = pol.sample(False, d("mean"), d("L"), *args64, eps=d("eps")).float()
    mean64, L64 = d("mean").requires_grad_(True), d("L").requires_grad_(True)
    lp = pol.log_prob(smp.double(), mean64, L64, *args64, pred_pairs=pairs)
    w = torch.linspace(0.5, 1.5, lp.numel(), dtype=torch.float64).reshape(lp.shape)
    gm, gL = torch.autograd.grad((lp * w).sum(), [mean64, L64])
    gL = gL.diagonal(dim1=-2, dim2=-1)

    tabs = ops.Tables(**cfg)
    c = lambda t: t.to(DEV)
    args = (c(times), c(inp["init_time"]), c(inp["init_pos"]), c(inp["init_vel"]), c(pairs), tabs)
    mean_g, L_g = c(inp["mean"]).requires_grad_(True), c(inp["L"]).requires_grad_(True)
    got, info, _ = ops.seg_logprob_diag(c(smp), mean_g, L_g, *args, return_info=True)
    assert got.shape == (B, P) and int(info.abs().max()) == 0
    assert (f64(got) - lp.detach()).abs().max() <= 1e-4
    (got * c(w.float())).sum().backward()
    assert (f64(mean_g.grad) - gm).abs().max() <= 2e-4 * gm.abs().max()
    gd = f64(L_g.grad)
    assert (gd.diagonal(dim1=-2, dim2=-1) - gL).abs().max() <= 2e-4 * gL.abs().max()
    assert float((gd - torch.diag_embed(gd.diagonal(dim1=-2, dim2=-1))).abs().max()) == 0.0
    # the dense staged kernels on the same dense diagonal factors
    mean_s, L_s = c(inp["mean"]).requires_grad_(True), c(inp["L"]).requires_grad_(True)
    dense = ops.seg_logprob_staged(c(smp), mean_s, L_s, *args)
    assert (dense - got).abs().max().item() <= 1e-4
    (dense * c(w.float())).sum().backward()
    assert (mean_s.grad - mean_g.grad).abs().max().item() <= 2e-4 * mean_s.grad.abs().max().item()
    dd = L_s.grad.diagonal(dim1=-2, dim2=-1)
    assert (dd - L_g.grad.diagonal(dim1=-2, dim2=-1)).abs().max().item() <= 2e-4 * dd.abs().max().item()
    # deterministic: a second run gives the same bits
    again = ops.seg_logprob_diag(c(smp), mean_g.detach(), L_g.detach(), *args)
    assert torch.equal(again, got.detach())


# ---- policy epochs -------------------------------------------------------------------------------------------------
def tce_policy(name, contextual, obs_dim=10, seed=0):
    cfg = MP_CONFIGS[name]
    torch.manual_seed(seed)
    return policy_factory("TemporalCorrelatedPolicy", dim_in=obs_dim, dim_out=dims(name)[3],
                          mean_net_args=dict(avg_neuron=32, num_hidden=2, shape=0.0),
                          variance_net_args=dict(std_only=True, contextual=contextual, avg_neuron=32, num_hidden=2,
                                                 shape=0.0),
                          init_method="orthogonal", out_layer_gain=0.01, act_func_hidden="leaky_relu",
                          act_func_last=None, dtype="float32", device=DEV, min_std=1e-4,
                          mp=dict(type="prodmp", args=dict(cfg)))


@pytest.mark.parametrize("name,typ,contextual", [("box", "KLProjectionLayer", True), ("box", "KLProjectionLayer", False),
                                                 ("metaworld", "KLProjectionLayer", True),
                                                 ("table_tennis", "WassersteinProjectionLayer", True),
                                                 ("box", "WassersteinProjectionLayer", False),
                                                 ("box", "FrobeniusProjectionLayer", True),
                                                 ("table_tennis", "FrobeniusProjectionLayer", False)])
def test_std_only_policy_epoch_matches_oracle(name, typ, contextual):
    B, obs_dim = 24, 10
    cfg, D, K1, Dp = dims(name)
    T = NUM_TIMES[name]
    mb, cb = LAYERS[typ]
    kw = dict(KL_KW, proj_type=typ, mean_bound=mb, cov_bound=cb, entropy_schedule="linear", action_dim=Dp)
    inp = synthetic_inputs(name, B, seed=21, dtype=torch.float32)
    policy = tce_policy(name, contextual, obs_dim)
    assert policy.is_diag and policy.variance_net is not None
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
    obs = torch.randn(B, obs_dim + 2 * D)
    times = sampler.get_times(c(inp["init_time"]), T)
    with torch.no_grad():
        mean_old, L_old = policy.policy(c(obs)[..., :-2 * D])
        mean_old = mean_old + 0.05 * c(torch.randn(B, Dp))
        L_old = L_old * torch.diag_embed(torch.exp(0.05 * c(torch.randn(B if contextual else 1, Dp))))
        if not contextual:
            L_old = L_old[:1].expand(B, -1, -1).contiguous()
        smp = policy.sample(False, mean_old, L_old, times, c(inp["init_time"]), c(inp["init_pos"]),
                            c(inp["init_vel"]), eps=c(inp["eps"]))
        lp_old = policy.log_prob(smp, mean_old, L_old, times, c(inp["init_time"]), c(inp["init_pos"]),
                                 c(inp["init_vel"]), pred_pairs=pairs)
        adv, _ = agent.get_advantage_return(c(inp["rewards"]), c(inp["values"]), c(inp["dones"]),
                                            c(inp["time_limit_dones"]))
        seg_adv = agent.get_segment_advantage(c(inp["rewards"]), c(inp["values"]), adv, pairs)
    dataset = dict(segment_state=c(obs), step_actions=smp, segment_log_prob_estimate=lp_old,
                   segment_params_mean=mean_old, segment_params_L=L_old, segment_advantage=seg_adv,
                   segment_init_time=c(inp["init_time"]), segment_init_pos=c(inp["init_pos"]),
                   segment_init_vel=c(inp["init_vel"]))
    layer.initial_entropy = policy.entropy([mean_old, L_old]).mean()
    params0 = [p.detach().clone() for p in policy.parameters]
    metrics = agent.policy_epoch(dataset, times, pairs).cpu()
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
    olayer = oproj.projection_factory(typ, dtype=torch.float64, **kw)
    olayer.initial_entropy = f64(layer.initial_entropy)
    odata = {k: (f64(v) if v.is_floating_point() else v.cpu()) for k, v in dataset.items()}
    loss, parts = oa.policy_epoch(opolicy, olayer, odata, f64(times), pairs.cpu(), 0, set_variance=False,
                                  with_metrics=True)
    oparams = list(mean_net.parameters()) + (list(var_net.parameters()) if contextual else [cov_vec])
    ograds = torch.autograd.grad(loss, oparams)
    assert abs(metrics[0].item() - parts["surrogate_loss"].item()) <= 1e-4
    assert abs(metrics[2].item() - parts["trust_region_loss"].item()) <= 1e-4
    assert abs(metrics[3].item() - loss.item()) <= 2e-4
    assert abs(metrics[4].item() - parts["entropy"].item()) <= 1e-4
    assert abs(metrics[5].item() - parts["imp_smp_ratio"].item()) <= 1e-4
    for i, key in enumerate(_KL_KEYS):
        assert abs(metrics[7 + i].item() - parts["kl"][key].item()) <= 1e-4, key
    for g, og in zip(grads, ograds):
        assert (g - og).abs().max() <= 1e-3 * max(1e-3, og.abs().max().item())


def test_std_only_bbrl_epoch_matches_oracle():
    B, Dp, obs_dim = 48, 63, 9
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
    inp = synthetic_inputs("box", B, seed=4, dtype=torch.float32)
    g = torch.Generator().manual_seed(6)
    obs = torch.randn(B, obs_dim, generator=g).to(DEV)
    with torch.no_grad():
        mean_old, L_old = policy.policy(obs)
        mean_old = (mean_old + 0.05 * torch.randn(B, Dp, generator=g).to(DEV)).contiguous()
        L_old = (L_old[:1] * torch.exp(0.03 * torch.randn(Dp, generator=g)).to(DEV)).expand(B, -1, -1).contiguous()
        actions = policy.sample(False, mean_old, L_old, eps=inp["eps"].to(DEV))
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
    assert cov_vec.shape == (Dp,)
    opolicy = opol.BlackBoxPolicy(Dp, mean_net=mean_net, cov_vector=cov_vec, contextual=False, std_only=True,
                                  min_std=1e-4)
    olayer = oproj.projection_factory("KLProjectionLayer", dtype=torch.float64, **kw)
    olayer.initial_entropy = f64(layer.initial_entropy)
    loss, parts = oa.policy_epoch_bbrl(opolicy, olayer, odata, 0, set_variance=False, with_metrics=True)
    ograds = torch.autograd.grad(loss, list(mean_net.parameters()) + [cov_vec])
    assert abs(metrics[0].item() - parts["surrogate_loss"].item()) <= 1e-4
    assert abs(metrics[2].item() - parts["trust_region_loss"].item()) <= 1e-4 * max(1.0, abs(parts["trust_region_loss"].item()))
    for i, key in enumerate(_KL_KEYS):
        assert abs(metrics[7 + i].item() - parts["kl"][key].item()) <= 1e-4, key
    for gr, og in zip(grads, ograds):
        assert (gr - og).abs().max() <= 1e-3 * max(1e-3, og.abs().max().item())


def agent_with_data(use_graph, B=64, name="box"):
    """test_gpu_agent.build (agent, sampler and data of the shipped agent test) with a contextual std_only policy."""
    import test_gpu_agent
    orig = test_gpu_agent.policy_factory

    def std_only_factory(typ, **kw):
        kw["variance_net_args"] = dict(std_only=True, contextual=True, avg_neuron=32, num_hidden=2, shape=0.0)
        return orig(typ, **kw)
    test_gpu_agent.policy_factory = std_only_factory
    try:
        return test_gpu_agent.build(name=name, B=B, use_graph=use_graph, epochs=3)
    finally:
        test_gpu_agent.policy_factory = orig


def test_std_only_graph_captured_update_equals_eager():
    outs, params = [], []
    for use_graph in (False, True):
        agent, dataset = agent_with_data(use_graph)
        assert agent.policy.is_diag and agent.policy.contextual_cov
        agent.num_iterations = 1
        dataset = agent.process_dataset(dataset)
        out = agent.update_policy(dataset)
        assert all(torch.isfinite(torch.tensor(float(v))) for v in out.values())
        outs.append(out)
        params.append([p.detach().clone() for p in agent.policy.parameters])
    for k in outs[0]:
        assert abs(outs[0][k] - outs[1][k]) <= 1e-4 * max(1.0, abs(outs[0][k])), k
    for p, q in zip(*params):
        assert (p - q).abs().max().item() <= 1e-5


@pytest.mark.parametrize("contextual", [True, False])
def test_std_only_checkpoint_round_trip(tmp_path, contextual):
    policy = tce_policy("box", contextual, seed=0)
    with torch.no_grad():
        for p in policy.parameters:
            p.add_(0.1 * torch.randn_like(p))
    policy.save_weights(str(tmp_path), 3)
    files = set(os.listdir(tmp_path))
    var = "TemporalCorrelatedPolicy_variance_mlp_weights_3" if contextual else \
        "TemporalCorrelatedPolicy_variance_variable_weights_3"
    assert {"TemporalCorrelatedPolicy_mean_mlp_weights_3", var} <= files, files
    other = tce_policy("box", contextual, seed=5)
    other.load_weights(str(tmp_path), 3)
    for p, q in zip(policy.parameters, other.parameters):
        assert torch.equal(p, q)
    obs = torch.randn(7, 10, device=DEV)
    (m1, L1), (m2, L2) = policy.policy(obs), other.policy(obs)
    assert torch.equal(m1, m2) and torch.equal(L1, L2)
    if not contextual:                                   # set_variance path: factor -> vector -> factor
        vec = policy.variance_net.variable.detach().clone()
        policy.set_cov_variable(L1[0])
        assert policy.variance_net.variable.shape == (63,)
        assert (policy.variance_net.variable - vec).abs().max().item() <= 1e-5

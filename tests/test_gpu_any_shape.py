"""ProDMP shapes without specialised kernels (any 1 <= num_dof <= 8, 2 <= K1 <= 16, Dp <= 64 other than the five shipped
pairs): trajectory synthesis, the segment likelihood on the staged kernels for every covariance input of
``ops_seglik.seglik`` and the policy epoch, against the fp64 CPU oracle.  The MP configs are built here (the box and
metaworld task settings with other num_dof / num_basis) so that the shipped parametrisations stay as they are."""
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
    from tce_rl_b200 import ops, ops_seglik
    from tce_rl_b200._lib import TceError
    from tce_rl_b200.rl import TemporalCorrelatedAgent, policy_factory, projection_factory
    from tce_rl_b200.rl.agent import _KL_KEYS, SegmentTimeSampler

DEV = "cuda:0"
SHAPES = [(1, 2), (5, 7), (6, 6), (3, 13), (8, 8), (4, 16)]          # (num_dof, K1)
TASK = {(1, 2): "box", (5, 7): "metaworld", (6, 6): "box", (3, 13): "metaworld", (8, 8): "box", (4, 16): "box"}


def f64(t):
    return t.detach().double().cpu()


def mp_cfg(D, K1):
    task = TASK.get((D, K1), "box")
    return dict(MP_CONFIGS[task], num_dof=D, num_basis=K1 - 1), NUM_TIMES[task]


def inputs(D, K1, B, seed=1234):
    """synthetic_inputs of oracle.gen_golden for any shape (float32)."""
    Dp = D * K1
    g = torch.Generator().manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    mean = 0.5 * rn(B, Dp)
    L = torch.tril(0.05 * rn(B, Dp, Dp), -1) + torch.diag_embed(torch.nn.functional.softplus(rn(B, Dp)) + 1e-4)
    out = dict(mean=mean, L=L, init_time=torch.rand(B, generator=g, dtype=torch.float64) * 0.3,
               init_pos=torch.rand(B, D, generator=g, dtype=torch.float64) * 2 - 1, init_vel=0.1 * rn(B, D),
               eps=rn(B, Dp))
    return {k: v.float() for k, v in out.items()}


def test_shipped_shapes_are_the_compiled_ones():
    for name, cfg in MP_CONFIGS.items():
        assert ops.Tables(**cfg).compiled, name
    for D, K1 in SHAPES:
        cfg, _ = mp_cfg(D, K1)
        assert not ops.Tables(**cfg).compiled


# ---- trajectory ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K1", list(range(2, 17)))
def test_trajectory_matches_oracle(K1):
    """Every K1 of the trajectory kernels' dispatch (2..16), the five compiled shapes' 3, 4 and 9 included: forward on
    per-episode and on one common time grid, and the backward."""
    D = 4
    cfg, T = mp_cfg(D, K1)
    B = 64                                              # >= 64: a common time grid takes the uniform kernels
    inp = inputs(D, K1, B, seed=K1)
    tabs = ops.Tables(**cfg)
    omp = ou_mp(cfg)
    c = lambda t: t.to(DEV)
    for uniform in (False, True):
        init_time = inp["init_time"][:1].expand(B).contiguous() if uniform else inp["init_time"]
        times = ou.get_times(init_time.double(), T, cfg["dt"]).float()
        params = c(inp["mean"]).requires_grad_(True)
        traj = ops.prodmp_traj(params, c(times), c(init_time), c(inp["init_pos"]), c(inp["init_vel"]), tabs.handle, D)
        omp.update_inputs(times.double(), inp["mean"].double(), None, init_time.double(), inp["init_pos"].double(),
                          inp["init_vel"].double())
        pos, vel = omp.get_traj_pos(), omp.get_traj_vel()
        ref = torch.cat([pos, vel], -1)
        assert traj.shape == ref.shape
        assert (f64(traj) - ref).abs().max() <= 1e-5 * ref.abs().max()
        w = torch.linspace(-1, 1, ref.numel(), dtype=torch.float64).reshape(ref.shape)
        p64 = inp["mean"].double().requires_grad_(True)
        omp.update_inputs(times.double(), p64, None, init_time.double(), inp["init_pos"].double(),
                          inp["init_vel"].double())
        g_ref, = torch.autograd.grad((torch.cat([omp.get_traj_pos(), omp.get_traj_vel()], -1) * w).sum(), p64)
        (traj * c(w.float())).sum().backward()
        assert (f64(params.grad) - g_ref).abs().max() <= 1e-5 * g_ref.abs().max()


def ou_mp(cfg):
    from oracle.prodmp import get_mp
    return get_mp(type="prodmp", args=dict(cfg, dtype=torch.float64))


# ---- likelihood ----------------------------------------------------------------------------------------------------
def lik_case(D, K1, B, P, ragged, seed=5):
    cfg, T = mp_cfg(D, K1)
    Dp = D * K1
    inp = inputs(D, K1, B, seed=seed)
    times = ou.get_times(inp["init_time"].double(), T, cfg["dt"]).float()
    torch.manual_seed(seed)
    if ragged:
        pairs = torch.tensor([[0, 1], [0, T - 1], [5, 50], [T - 2, T - 1], [10, 11], [11, 12], [40, 80]])[:P]
    else:
        pairs = ou.get_time_pairs(T, dict(num_select=P + 1, fixed_interval=True))[:P]
    pol = opol.TemporalCorrelatedPolicy(Dp, mp=dict(type="prodmp", args=dict(cfg, dtype=torch.float64)), contextual=True)
    d = lambda k: inp[k].double()
    args64 = (times.double(), d("init_time"), d("init_pos"), d("init_vel"))
    smp = pol.sample(False, d("mean"), d("L"), *args64, eps=d("eps")).float()
    return cfg, inp, times, pairs, pol, smp, args64


def run_seglik(tabs, smp, mean, L, sigma, times, inp, pairs, mode, grad_logp=None, logp_old=None, adv=None,
               want_L=False, want_S=False):
    c = lambda t: t.to(DEV)
    return ops_seglik.seglik(c(smp), mean, L, None if sigma is None else sigma[0], None if sigma is None else sigma[1],
                             c(times), c(inp["init_time"]), c(inp["init_pos"]), c(inp["init_vel"]), c(pairs),
                             tabs.handle, 1e-4, mode, grad_logp, logp_old, adv, ops_seglik.pairs_chained(c(pairs)),
                             False, want_L, want_S)


@pytest.mark.parametrize("D,K1", SHAPES)
@pytest.mark.parametrize("cov", ["episode", "shared_L", "shared_sigma"])
@pytest.mark.parametrize("B,P,ragged", [(37, 25, False), (1, 1, False), (1024, 25, False), (37, 7, True)])
def test_likelihood_matches_oracle(D, K1, cov, B, P, ragged):
    Dp = D * K1
    cfg, inp, times, pairs, pol, smp, args64 = lik_case(D, K1, B, P, ragged)
    tabs = ops.Tables(**cfg)
    c = lambda t: t.to(DEV)
    mean64 = inp["mean"].double().requires_grad_(True)
    if cov == "episode":
        L64 = inp["L"].double().requires_grad_(True)
        Lo, wrt = L64, L64
    elif cov == "shared_L":
        L64 = inp["L"][:1].double().requires_grad_(True)
        Lo, wrt = L64.expand(B, -1, -1), L64
    else:
        S = inp["L"][0].double() @ inp["L"][0].double().T
        S64 = S.clone().requires_grad_(True)
        Lo = torch.linalg.cholesky(0.5 * (S64 + S64.T)).expand(B, -1, -1)
        wrt = S64
    lp, _, _, reg = pol.log_prob(smp.double(), mean64, Lo, *args64, pred_pairs=pairs, return_parts=True)
    w = torch.linspace(0.5, 1.5, lp.numel(), dtype=torch.float64).reshape(lp.shape)
    g_mean_ref, g_cov_ref = torch.autograd.grad((lp * w).sum(), [mean64, wrt])
    # a factor's free entries are its lower triangle: the kernels return tril(d lp / d L)
    free = (lambda g: g) if cov == "shared_sigma" else torch.tril
    g_cov_ref = free(g_cov_ref)
    lp_old = (lp.detach() + 0.1 * torch.randn(lp.shape, generator=torch.Generator().manual_seed(1), dtype=torch.float64))
    adv = torch.randn(lp.shape, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    mean64b = inp["mean"].double().requires_grad_(True)
    wrt_b = wrt.detach().clone().requires_grad_(True)
    Lo_b = (wrt_b if cov == "episode" else wrt_b.expand(B, -1, -1)) if cov != "shared_sigma" else \
        torch.linalg.cholesky(0.5 * (wrt_b + wrt_b.T)).expand(B, -1, -1)
    lp_b = pol.log_prob(smp.double(), mean64b, Lo_b, *args64, pred_pairs=pairs)
    loss_ref, parts = oa.surrogate_loss(adv, lp_b, lp_old)
    gs_mean_ref, gs_cov_ref = torch.autograd.grad(loss_ref, [mean64b, wrt_b])
    gs_cov_ref = free(gs_cov_ref)

    mean = c(inp["mean"])
    if cov == "episode":
        L, sigma = c(inp["L"]), None
    elif cov == "shared_L":
        L, sigma = c(inp["L"][:1]), None
    else:
        L = None
        sigma = (c(S / 2.0), torch.full((1,), 2.0, device=DEV, dtype=torch.float64))   # Sigma = 2 * (S / 2)
    want_L, want_S = cov != "shared_sigma", cov == "shared_sigma"
    logp, info, acc, _, _, _ = run_seglik(tabs, smp, mean, L, sigma, times, inp, pairs, 0)
    assert logp.shape == (B, P) and int(info.abs().max()) == 0
    assert (f64(logp) - lp.detach()).abs().max() <= 1e-4
    # grad mode 1
    _, _, acc1, g_mean, g_L, g_S = run_seglik(tabs, smp, mean, L, sigma, times, inp, pairs, 1,
                                              grad_logp=c(w.float()), want_L=want_L, want_S=want_S)
    assert torch.equal(acc1[0], acc[0])
    assert (f64(g_mean) - g_mean_ref).abs().max() <= 2e-4 * g_mean_ref.abs().max()
    g_cov = f64(g_S) if want_S else f64(g_L).reshape(g_cov_ref.shape)
    assert (g_cov - g_cov_ref).abs().max() <= 2e-4 * g_cov_ref.abs().max()
    # grad mode 2: the fused surrogate
    _, _, acc2, g_mean2, g_L2, g_S2 = run_seglik(tabs, smp, mean, L, sigma, times, inp, pairs, 2,
                                                 logp_old=c(lp_old.float()), adv=c(adv.float()), want_L=want_L,
                                                 want_S=want_S)
    assert abs(acc2[1].item() - loss_ref.item()) <= 1e-4 * max(1.0, abs(loss_ref.item()))
    assert abs(acc2[2].item() - parts["imp_smp_ratio"].item()) <= 1e-4
    assert (f64(g_mean2) - gs_mean_ref).abs().max() <= 2e-4 * gs_mean_ref.abs().max()
    g_cov2 = f64(g_S2) if want_S else f64(g_L2).reshape(gs_cov_ref.shape)
    assert (g_cov2 - gs_cov_ref).abs().max() <= 2e-4 * gs_cov_ref.abs().max()
    # the regulariser: 1e-4 x the batch-global max of the un-regularised diagonal of C
    assert abs(1e-4 * acc[0].item() - reg) <= 1e-6 * reg


@pytest.mark.parametrize("D,K1", SHAPES)
def test_likelihood_empty_batch(D, K1):
    cfg, T = mp_cfg(D, K1)
    Dp = D * K1
    tabs = ops.Tables(**cfg)
    z = lambda *s: torch.zeros(*s, device=DEV)
    pairs = ou.get_time_pairs(T, dict(num_select=26, fixed_interval=True))[:25].to(DEV)
    for L, sigma, want_L, want_S in [(z(0, Dp, Dp), None, True, False), (z(1, Dp, Dp), None, True, False),
                                     (None, torch.eye(Dp, device=DEV, dtype=torch.float64), False, True)]:
        logp, info, acc, g_mean, g_L, g_S = ops_seglik.seglik(
            z(0, T, 2 * D), z(0, Dp), L, sigma, None, z(0, T), z(0), z(0, D), z(0, D), pairs, tabs.handle, 1e-4, 1,
            z(0, 25), None, None, True, False, want_L, want_S)
        assert logp.shape == (0, 25) and g_mean.shape == (0, Dp)
        if want_S:
            assert g_S.shape == (Dp, Dp) and float(g_S.abs().max()) == 0.0


@pytest.mark.parametrize("D,K1", [(6, 6), (4, 16), (8, 8)])
def test_cross_paths_on_new_shapes(D, K1):
    B, P = 64, 25
    Dp = D * K1
    cfg, inp, times, pairs, pol, smp, args64 = lik_case(D, K1, B, P, False, seed=9)
    tabs = ops.Tables(**cfg)
    c = lambda t: t.to(DEV)
    mean = c(inp["mean"])
    L1 = c(inp["L"][:1])
    w = c(torch.linspace(0.5, 1.5, B * P).reshape(B, P))
    # per-episode L with all rows equal == the shared L == the shared Sigma
    lp_e, _, _, gm_e, gL_e, _ = run_seglik(tabs, smp, mean, L1.expand(B, -1, -1).contiguous(), None, times, inp, pairs,
                                           1, grad_logp=w, want_L=True)
    lp_s, _, _, gm_s, gL_s, gS_s = run_seglik(tabs, smp, mean, L1, None, times, inp, pairs, 1, grad_logp=w,
                                              want_L=True, want_S=False)
    S = (L1[0].double() @ L1[0].double().T).contiguous()
    lp_S, _, _, gm_S, _, gS = run_seglik(tabs, smp, mean, None, (S, None), times, inp, pairs, 1, grad_logp=w,
                                         want_S=True)
    assert (lp_e - lp_s).abs().max().item() <= 1e-4 and (lp_S - lp_s).abs().max().item() <= 1e-4
    assert (gm_e - gm_s).abs().max().item() <= 2e-4 * gm_s.abs().max().item()
    assert (gm_S - gm_s).abs().max().item() <= 2e-4 * gm_s.abs().max().item()
    gsum = gL_e.double().sum(0)
    assert (gL_s[0].double() - gsum).abs().max().item() <= 2e-4 * gsum.abs().max().item()
    via_S = 2 * torch.tril(gS @ L1[0].double())
    assert (via_S - gsum).abs().max().item() <= 2e-4 * gsum.abs().max().item()
    # a shared-Sigma backward run twice gives the same bits
    _, _, _, gm_S2, _, gS2 = run_seglik(tabs, smp, mean, None, (S, None), times, inp, pairs, 1, grad_logp=w,
                                        want_S=True)
    assert torch.equal(gS2, gS) and torch.equal(gm_S2, gm_S)
    # the diagonal likelihood == the dense likelihood on diagonal factors
    s = c(torch.exp(0.3 * torch.randn(B, Dp, generator=torch.Generator().manual_seed(3))))
    Ld = torch.diag_embed(s).contiguous()
    args = (c(times), c(inp["init_time"]), c(inp["init_pos"]), c(inp["init_vel"]), c(pairs), tabs)
    mg, Lg = mean.clone().requires_grad_(True), Ld.clone().requires_grad_(True)
    lp_d = ops.seg_logprob_diag(c(smp), mg, Lg, *args)
    (lp_d * w).sum().backward()
    md, Ldd = mean.clone().requires_grad_(True), Ld.clone().requires_grad_(True)
    lp_dense = ops.seg_logprob_staged(c(smp), md, Ldd, *args)
    (lp_dense * w).sum().backward()
    assert (lp_d - lp_dense).abs().max().item() <= 1e-4
    assert (mg.grad - md.grad).abs().max().item() <= 2e-4 * md.grad.abs().max().item()
    dd = Ldd.grad.diagonal(dim1=-2, dim2=-1)
    assert (Lg.grad.diagonal(dim1=-2, dim2=-1) - dd).abs().max().item() <= 2e-4 * dd.abs().max().item()
    # the public entry points: seg_logprob (shared L -> seglik), seg_surrogate_staged, get_traj_pos_cov
    lp_pub = ops.seg_logprob(c(smp), mean, L1.expand(B, -1, -1), *args)
    assert (lp_pub - lp_s).abs().max().item() <= 1e-4
    loss, ratio, lp_sur = ops.seg_surrogate_staged(c(smp), mean, L1.expand(B, -1, -1).contiguous(), *args[:5],
                                                   lp_s.detach(), w, tabs)
    assert abs(ratio.item() - 1.0) <= 1e-5 and (lp_sur - lp_s).abs().max().item() <= 1e-4
    from tce_rl_b200 import mp as tmp
    tp = times[:, pairs]                                                   # [B, P, 2]
    ex = lambda t: t.unsqueeze(1).expand(B, P, *t.shape[1:])
    Le = inp["L"][:1].expand(B, -1, -1)
    C = tmp.ProDMP(tabs).get_traj_pos_cov(c(tp), c(ex(Le)), c(ex(inp["init_time"])), c(ex(inp["init_pos"])),
                                          c(ex(inp["init_vel"])))
    Cref = pol.mp.get_traj_pos_cov(tp.double(), ex(Le).double(), ex(inp["init_time"]).double(),
                                   ex(inp["init_pos"]).double(), ex(inp["init_vel"]).double())
    assert C.shape == Cref.shape and (f64(C) - Cref).abs().max() <= 1e-5 * Cref.abs().max()


def test_outside_the_supported_set_still_raises():
    D, K1 = 8, 9                                        # Dp = 72 > 64
    cfg = dict(MP_CONFIGS["box"], num_dof=D, num_basis=K1 - 1)
    tabs = ops.Tables(**cfg)
    assert not tabs.compiled
    B, P, T, Dp = 4, 25, NUM_TIMES["box"], D * K1
    z = lambda *s: torch.zeros(*s, device=DEV)
    pairs = ou.get_time_pairs(T, dict(num_select=26, fixed_interval=True))[:25].to(DEV)
    eye = torch.eye(Dp, device=DEV).expand(B, -1, -1).contiguous()
    for L in (eye, eye[:1]):
        with pytest.raises(TceError, match="unsupported"):
            ops_seglik.seglik(z(B, T, 2 * D), z(B, Dp), L, None, None, z(B, T), z(B), z(B, D), z(B, D), pairs,
                              tabs.handle, 1e-4, 0, None, None, None, True, False, False)


# ---- policy epochs -------------------------------------------------------------------------------------------------
KL_KW = dict(proj_type="kl", mean_bound=0.05, cov_bound=5e-4, trust_region_coeff=1.0, scale_prec=True,
             total_train_steps=7500, target_entropy=0.0, temperature=0.7, entropy_eq=False, entropy_first=False,
             do_regression=False)
LAYERS = {"KLProjectionLayer": (0.05, 5e-4), "FrobeniusProjectionLayer": (0.05, 5e-4),
          "WassersteinProjectionLayer": (0.005, 2.5e-4)}


def tce_policy(cfg, Dp, contextual, std_only, obs_dim=10, seed=0):
    torch.manual_seed(seed)
    return policy_factory("TemporalCorrelatedPolicy", dim_in=obs_dim, dim_out=Dp,
                          mean_net_args=dict(avg_neuron=32, num_hidden=2, shape=0.0),
                          variance_net_args=dict(std_only=std_only, contextual=contextual, avg_neuron=32, num_hidden=2,
                                                 shape=0.0),
                          init_method="orthogonal", out_layer_gain=0.01, act_func_hidden="leaky_relu",
                          act_func_last=None, dtype="float32", device=DEV, min_std=1e-4,
                          mp=dict(type="prodmp", args=dict(cfg)))


@pytest.mark.parametrize("D,K1", [(6, 6), (8, 8)])
@pytest.mark.parametrize("typ,contextual,std_only", [("KLProjectionLayer", False, False),
                                                     ("KLProjectionLayer", True, False),
                                                     ("WassersteinProjectionLayer", False, False),
                                                     ("FrobeniusProjectionLayer", False, False),
                                                     ("KLProjectionLayer", True, True)])
def test_policy_epoch_matches_oracle(D, K1, typ, contextual, std_only):
    B, obs_dim = 24, 10
    cfg, T = mp_cfg(D, K1)
    Dp = D * K1
    mb, cb = LAYERS[typ]
    kw = dict(KL_KW, proj_type=typ, mean_bound=mb, cov_bound=cb, entropy_schedule="linear", action_dim=Dp)
    inp = inputs(D, K1, B, seed=21)
    policy = tce_policy(cfg, Dp, contextual, std_only, obs_dim)
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
    init_time = torch.zeros(B)
    times = sampler.get_times(c(init_time), T)
    with torch.no_grad():
        mean_old, L_old = policy.policy(c(obs)[..., :-2 * D])
        mean_old = mean_old + 0.05 * c(torch.randn(B, Dp, generator=g))
        L_old = L_old * torch.diag_embed(torch.exp(0.05 * c(torch.randn(B if contextual else 1, Dp, generator=g))))
        if not contextual:
            L_old = L_old[:1].expand(B, -1, -1).contiguous()
        smp = policy.sample(False, mean_old, L_old, times, c(init_time), c(inp["init_pos"]), c(inp["init_vel"]),
                            eps=c(inp["eps"]))
        lp_old = policy.log_prob(smp, mean_old, L_old, times, c(init_time), c(inp["init_pos"]), c(inp["init_vel"]),
                                 pred_pairs=pairs)
        rewards, values = torch.randn(B, T, generator=g), torch.randn(B, T + 1, generator=g)
        dones = torch.zeros(B, T, dtype=torch.bool)
        dones[:, -1] = True
        adv, _ = agent.get_advantage_return(c(rewards), c(values), c(dones), c(torch.zeros(B, T, dtype=torch.bool)))
        seg_adv = agent.get_segment_advantage(c(rewards), c(values), adv, pairs)
    dataset = dict(segment_state=c(obs), step_actions=smp, segment_log_prob_estimate=lp_old,
                   segment_params_mean=mean_old, segment_params_L=L_old, segment_advantage=seg_adv,
                   segment_init_time=c(init_time), segment_init_pos=c(inp["init_pos"]),
                   segment_init_vel=c(inp["init_vel"]))
    layer.initial_entropy = policy.entropy([mean_old, L_old]).mean()
    params0 = [p.detach().clone() for p in policy.parameters]
    agent.ensure_flat_grads(agent.policy_net_params)          # as update_policy: one flat gradient + FlatAdam
    agent._use_flat_adam()
    metrics = agent.policy_epoch(dataset, times, pairs).cpu()
    grads = [p.grad.detach().double().cpu() for p in policy.parameters]
    # the hand-scheduled shared-covariance KL epoch serves the new shapes through the staged likelihood
    assert (agent._fast is not None) == (typ == "KLProjectionLayer" and not contextual and not std_only)

    mean_net = copy.deepcopy(policy.mean_net).cpu().double()
    var_net = copy.deepcopy(policy.variance_net).cpu().double() if contextual else None
    with torch.no_grad():
        for p, p0 in zip(list(mean_net.parameters()) + (list(var_net.parameters()) if contextual else []), params0):
            p.copy_(p0.double().cpu())
    cov_vec = None if contextual else params0[-1].double().cpu().requires_grad_(True)
    opolicy = opol.TemporalCorrelatedPolicy(Dp, mp=dict(type="prodmp", args=dict(cfg, dtype=torch.float64)),
                                            mean_net=mean_net, variance_net=var_net, cov_vector=cov_vec,
                                            contextual=contextual, std_only=std_only, min_std=1e-4)
    olayer = (oproj_diag if std_only else oproj).projection_factory(typ, dtype=torch.float64, **kw)
    olayer.initial_entropy = f64(layer.initial_entropy)
    odata = {k: (f64(v) if v.is_floating_point() else v.cpu()) for k, v in dataset.items()}
    loss, parts = oa.policy_epoch(opolicy, olayer, odata, f64(times), pairs.cpu(), 0, set_variance=False,
                                  with_metrics=True)
    oparams = list(mean_net.parameters()) + (list(var_net.parameters()) if contextual else [cov_vec])
    ograds = torch.autograd.grad(loss, oparams)
    assert abs(metrics[0].item() - parts["surrogate_loss"].item()) <= 1e-4
    assert abs(metrics[2].item() - parts["trust_region_loss"].item()) <= 1e-4
    assert abs(metrics[3].item() - loss.item()) <= 2e-4
    assert abs(metrics[5].item() - parts["imp_smp_ratio"].item()) <= 1e-4
    for i, key in enumerate(_KL_KEYS):
        assert abs(metrics[7 + i].item() - parts["kl"][key].item()) <= 1e-4, key
    for gr, og in zip(grads, ograds):
        assert (gr - og).abs().max() <= 1e-3 * max(1e-3, og.abs().max().item())


def test_graph_captured_update_equals_eager_on_a_new_shape():
    import test_gpu_agent
    from oracle import gen_golden
    name = "_any_shape_6x6"
    gen_golden.MP_CONFIGS[name], gen_golden.NUM_TIMES[name] = mp_cfg(6, 6)
    try:
        outs, params = [], []
        for use_graph in (False, True):
            agent, dataset = test_gpu_agent.build(name=name, B=64, use_graph=use_graph, epochs=3)
            assert not agent.policy.mp.tables.compiled
            agent.num_iterations = 1
            dataset = agent.process_dataset(dataset)
            out = agent.update_policy(dataset)
            assert all(torch.isfinite(torch.tensor(float(v))) for v in out.values())
            outs.append(out)
            params.append([p.detach().clone() for p in agent.policy.parameters])
    finally:
        del gen_golden.MP_CONFIGS[name], gen_golden.NUM_TIMES[name]
    for k in outs[0]:
        assert abs(outs[0][k] - outs[1][k]) <= 1e-4 * max(1.0, abs(outs[0][k])), k
    for p, q in zip(*params):
        assert (p - q).abs().max().item() <= 1e-5

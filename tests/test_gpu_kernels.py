"""Parity of the CUDA kernels (through the C ABI / torch custom ops) against the CPU oracle.

Tolerances (BASELINE.json north_star): index sampling bit exact, trajectories <= 1e-5 relative,
log-probs / KLs / projected parameters <= 1e-4 absolute.  Inputs are fp32 tensors; the oracle evaluates
the same fp32 values in fp64.
"""
import math

import pytest
import torch

from oracle import agent as oa
from oracle import policy as opol
from oracle import util as ou
from oracle.gen_golden import MP_CONFIGS, NUM_TIMES, synthetic_inputs

pytestmark = pytest.mark.gpu

CUDA = torch.cuda.is_available()
if CUDA:
    from tce_rl_b200 import ops

DEV = "cuda:0"


def f64(t):
    return t.detach().double().cpu()


def make_oracle_policy(name, **kw):
    cfg = MP_CONFIGS[name]
    Dp = cfg["num_dof"] * (cfg["num_basis"] + 1)
    return opol.TemporalCorrelatedPolicy(Dp, mp=dict(type="prodmp", args=dict(cfg, dtype=torch.float64)),
                                         contextual=True, min_std=1e-4, **kw)


def setup_case(name, B, seed=1234, init_time_spread=0.0, P_select=25):
    cfg = MP_CONFIGS[name]
    T = NUM_TIMES[name]
    inp = synthetic_inputs(name, B, seed=seed, dtype=torch.float32)
    if init_time_spread:
        inp["init_time"] = (torch.rand(B, generator=torch.Generator().manual_seed(seed)) * init_time_spread).float()
    times = ou.get_times(inp["init_time"].double() + cfg.get("delay", 0.0) * 0, T, cfg["dt"]).float()
    torch.manual_seed(0)
    pairs = ou.get_time_pairs(T, dict(num_select=P_select, fixed_interval=True))
    return cfg, T, inp, times, pairs


@pytest.mark.parametrize("name", list(MP_CONFIGS))
def test_tables_match_oracle(name, golden):
    tabs = ops.Tables(**MP_CONFIGS[name])
    got = tabs.export()
    want = golden("oracle_path.pt")[name]["tables"]
    for k in ("y1", "y2", "dy1", "dy2", "pos_basis", "vel_basis", "scale"):
        scale = want[k].abs().max()
        assert (got[k] - want[k]).abs().max() <= 1e-11 * scale, k


@pytest.mark.parametrize("name", list(MP_CONFIGS))
@pytest.mark.parametrize("B", [1, 5, 300])
def test_trajectory_parity(name, B):
    cfg, T, inp, times, _ = setup_case(name, B, init_time_spread=0.2 if B == 5 else 0.0)
    pol = make_oracle_policy(name)
    d = lambda k: inp[k].double()
    theta = d("mean") + torch.einsum('bij,bj->bi', d("L"), d("eps"))
    want = pol.sample(False, theta, d("L"), times.double(), d("init_time"), d("init_pos"), d("init_vel"), use_mean=True)
    tabs = ops.Tables(**cfg)
    c = lambda t: t.float().to(DEV)
    got = ops.prodmp_traj(c(theta), c(times), c(inp["init_time"]), c(inp["init_pos"]), c(inp["init_vel"]),
                          tabs.handle, cfg["num_dof"])
    # theta is rounded to fp32 for the kernel: compare against the oracle on the rounded parameters
    want = pol.sample(False, theta.float().double(), d("L"), times.double(), d("init_time"), d("init_pos"),
                      d("init_vel"), use_mean=True)
    D = cfg["num_dof"]
    for sl in (slice(0, D), slice(D, 2 * D)):
        scale = want[..., sl].abs().max()
        assert (f64(got)[..., sl] - want[..., sl]).abs().max() <= 1e-5 * scale


@pytest.mark.parametrize("name", list(MP_CONFIGS))
def test_uniform_grid_trajectory_path_equals_general_kernel(name):
    """One time grid for the whole batch: basis rows evaluated once + per-episode matrix product
    (tce_prodmp_traj_fwd_uniform) against the general kernel and the oracle; a batch with per-episode start times must
    not take it."""
    B = 200
    cfg, T, inp, times, _ = setup_case(name, B)
    tabs = ops.Tables(**cfg)
    c = lambda t: t.to(DEV)
    args = (c(inp["mean"]), c(times), c(inp["init_time"]), c(inp["init_pos"]), c(inp["init_vel"]), tabs.handle, cfg["num_dof"])
    n0 = _lib_launch_count("tce_prodmp_traj_fwd_uniform")
    fast = ops.prodmp_traj(*args)
    assert _lib_launch_count("tce_prodmp_traj_fwd_uniform") == n0 + 1
    ops.UNIFORM_TRAJ = False
    try:
        general = ops.prodmp_traj(*args)
    finally:
        ops.UNIFORM_TRAJ = True
    scale = general.abs().max().item()
    assert (fast - general).abs().max().item() <= 2e-6 * scale
    pol = make_oracle_policy(name)
    want = pol.sample(False, inp["mean"].double(), inp["L"].double(), times.double(), inp["init_time"].double(),
                      inp["init_pos"].double(), inp["init_vel"].double(), use_mean=True)
    assert (f64(fast) - want).abs().max() <= 1e-5 * want.abs().max()
    cfg, T, inp2, times2, _ = setup_case(name, B, init_time_spread=0.2)
    n1 = _lib_launch_count("tce_prodmp_traj_fwd_uniform")
    ops.prodmp_traj(c(inp2["mean"]), c(times2), c(inp2["init_time"]), c(inp2["init_pos"]), c(inp2["init_vel"]), tabs.handle,
                    cfg["num_dof"])
    assert _lib_launch_count("tce_prodmp_traj_fwd_uniform") == n1


_COUNTS = {}


def _lib_launch_count(name):
    """Launches of one ABI entry so far (a counting wrapper installed on first use)."""
    from tce_rl_b200 import _lib
    if "installed" not in _COUNTS:
        orig = _lib.call

        def counting(n, *a):
            _COUNTS[n] = _COUNTS.get(n, 0) + 1
            return orig(n, *a)
        _lib.call = counting
        _COUNTS["installed"] = True
    return _COUNTS.get(name, 0)


def test_rsample_injected_and_philox():
    B, n = 257, 63
    inp = synthetic_inputs("box", B, dtype=torch.float32)
    c = lambda t: t.to(DEV)
    got = ops.mvn_rsample(c(inp["mean"]), c(inp["L"]), c(inp["eps"]), 0, 0)
    want = inp["mean"].double() + torch.einsum('bij,bj->bi', inp["L"].double(), inp["eps"].double())
    assert (f64(got) - want).abs().max() < 1e-5
    # shared (stride-0) covariance
    Ls = c(inp["L"][:1]).expand(B, n, n)
    got = ops.mvn_rsample(c(inp["mean"]), Ls, c(inp["eps"]), 0, 0)
    want = inp["mean"].double() + torch.einsum('ij,bj->bi', inp["L"][0].double(), inp["eps"].double())
    assert (f64(got) - want).abs().max() < 1e-5
    # in-kernel Philox draws: standard normal moments, reproducible, offset changes the stream
    Bbig = 4096
    mean0 = torch.zeros(Bbig, n, device=DEV)
    eye = torch.eye(n, device=DEV).expand(Bbig, n, n)
    z1 = ops.mvn_rsample(mean0, eye, None, 42, 0)
    z2 = ops.mvn_rsample(mean0, eye, None, 42, 0)
    z3 = ops.mvn_rsample(mean0, eye, None, 42, 1)
    assert torch.equal(z1, z2) and not torch.equal(z1, z3)
    assert abs(z1.mean().item()) < 0.01 and abs(z1.std().item() - 1) < 0.01
    assert abs((z1 ** 4).mean().item() - 3) < 0.1


@pytest.mark.parametrize("name,B", [("box", 64), ("box", 1), ("metaworld", 48), ("table_tennis", 48)])
def test_segment_logprob_parity(name, B):
    cfg, T, inp, times, pairs = setup_case(name, B)
    pol = make_oracle_policy(name)
    d = lambda k: inp[k].double()
    args64 = (times.double(), d("init_time"), d("init_pos"), d("init_vel"))
    smp = pol.sample(False, d("mean"), d("L"), *args64, eps=d("eps")).float()
    mean64, L64 = d("mean").requires_grad_(True), d("L").requires_grad_(True)
    lp, _, _, reg = pol.log_prob(smp.double(), mean64, L64, *args64, pred_pairs=pairs, return_parts=True)
    w = torch.linspace(0.5, 1.5, lp.numel(), dtype=torch.float64).reshape(lp.shape)
    gm, gL = torch.autograd.grad((lp * w).sum(), [mean64, L64])

    tabs = ops.Tables(**cfg)
    c = lambda t: t.to(DEV)
    mean_g, L_g = c(inp["mean"]).requires_grad_(True), c(inp["L"]).requires_grad_(True)
    got, info, diag_max = ops.seg_logprob(c(smp), mean_g, L_g, c(times), c(inp["init_time"]), c(inp["init_pos"]),
                                          c(inp["init_vel"]), c(pairs), tabs, return_info=True)
    assert int(info.abs().max()) == 0
    assert abs(diag_max.item() * 1e-4 - reg) <= 1e-6 * reg      # Sigma = L L^T is accumulated in fp32
    assert (f64(got) - lp.detach()).abs().max() <= 1e-4
    (got * c(w.float())).sum().backward()
    assert (f64(mean_g.grad) - gm).abs().max() <= 2e-4 * gm.abs().max()
    gL_t = torch.tril(gL)
    assert (f64(L_g.grad) - gL_t).abs().max() <= 2e-4 * gL_t.abs().max()
    assert float(L_g.grad.triu(1).abs().max()) == 0.0


def test_segment_logprob_shared_cov_and_ragged_pairs():
    """Stride-0 (non-contextual) covariance, per-episode init times, irregular / repeated time pairs."""
    name, B = "box", 33
    cfg, T, inp, times, _ = setup_case(name, B, init_time_spread=0.3)
    pairs = torch.tensor([[0, 1], [0, 99], [5, 50], [98, 99], [10, 11], [11, 12], [40, 80]])
    pol = make_oracle_policy(name)
    d = lambda k: inp[k].double()
    L1 = d("L")[:1]
    args64 = (times.double(), d("init_time"), d("init_pos"), d("init_vel"))
    smp = pol.sample(False, d("mean"), L1.expand(B, -1, -1), *args64, eps=d("eps")).float()
    L64 = L1.clone().requires_grad_(True)
    lp = pol.log_prob(smp.double(), d("mean"), L64.expand(B, -1, -1), *args64, pred_pairs=pairs)
    gL, = torch.autograd.grad(lp.sum(), L64)
    tabs = ops.Tables(**cfg)
    c = lambda t: t.to(DEV)
    L_g = c(inp["L"][:1]).requires_grad_(True)
    got = ops.seg_logprob(c(smp), c(inp["mean"]), L_g.expand(B, -1, -1), c(times), c(inp["init_time"]),
                          c(inp["init_pos"]), c(inp["init_vel"]), c(pairs), tabs)
    assert (f64(got) - lp.detach()).abs().max() <= 1e-4
    got.sum().backward()
    gL_t = torch.tril(gL)
    assert (f64(L_g.grad) - gL_t).abs().max() <= 2e-4 * gL_t.abs().max()


@pytest.mark.parametrize("B,T,gamma", [(6, 100, 1.0), (33, 37, 0.99), (2, 500, 0.97), (1, 1, 0.9)])
def test_gae_and_segment_advantage(B, T, gamma):
    g = torch.Generator().manual_seed(5)
    rewards, values = torch.randn(B, T, generator=g), torch.randn(B, T + 1, generator=g)
    dones = torch.zeros(B, T, dtype=torch.bool)
    dones[:, -1] = True
    if T > 4:
        dones[0, T // 2] = True
    tl = torch.zeros(B, T, dtype=torch.bool)
    if B > 1 and T > 4:
        tl[1, T // 3] = True
    c = lambda t: t.to(DEV)
    for use_gae in (True, False):
        adv_w, ret_w = oa.get_advantage_return(rewards.double(), values.double(), dones, tl, gamma, 0.95, use_gae)
        adv, ret = ops.gae(c(rewards), c(values), c(dones), c(tl), gamma, 0.95, use_gae)
        scale = max(1.0, ret_w.abs().max().item())
        assert (f64(adv) - adv_w).abs().max() <= 2e-6 * scale and (f64(ret) - ret_w).abs().max() <= 2e-6 * scale
    if T < 8:
        return
    torch.manual_seed(1)
    pairs = ou.get_time_pairs(T, dict(num_select=min(25, T // 3), fixed_interval=True))
    adv_w, _ = oa.get_advantage_return(rewards.double(), values.double(), dones, tl, gamma, 0.95, True)
    adv = c(adv_w.float())
    for mode_i, mode in enumerate(("accumulate", "value_subtraction")):
        for norm in (False, True):
            adv_in = adv_w.float().double()
            if mode == "accumulate" and norm:
                continue        # double normalisation is exercised through the agent class
            want = oa.get_segment_advantage(rewards.double(), values.double(), adv_in, pairs, gamma, mode, norm)
            got = ops.segment_advantage(mode_i, c(rewards), c(values), adv, c(pairs), gamma, norm)
            assert (f64(got) - want).abs().max() <= 1e-5 * max(1.0, want.abs().max().item())


@pytest.mark.parametrize("n,B", [(63, 17), (28, 5), (6, 3), (128, 2)])
def test_cholesky_fwd_bwd(n, B):
    g = torch.Generator().manual_seed(n)
    M = torch.randn(B, n, n, generator=g, dtype=torch.float64) / math.sqrt(n)
    A = (M @ M.transpose(-1, -2) + 0.5 * torch.eye(n, dtype=torch.float64)).float()
    A64 = A.double().requires_grad_(True)
    L64 = torch.linalg.cholesky(A64)
    Wt = torch.tril(torch.randn(B, n, n, generator=g, dtype=torch.float64))
    gA, = torch.autograd.grad((L64 * Wt).sum(), A64)
    A_g = A.to(DEV).requires_grad_(True)
    if n > 96:
        L_g, info = ops.chol_fwd(A_g.detach())
        assert (f64(L_g) - L64.detach()).abs().max() < 1e-5 and int(info.max()) == 0
        return
    L_g = ops.cholesky(A_g)
    assert (f64(L_g) - L64.detach()).abs().max() < 1e-5
    (L_g * Wt.float().to(DEV)).sum().backward()
    gA_sym = 0.5 * (gA + gA.transpose(-1, -2))
    assert (f64(A_g.grad) - gA_sym).abs().max() <= 1e-4 * gA_sym.abs().max()
    # non positive definite input is reported, not raised (LAPACK-style info)
    bad = A.clone()
    bad[0, 2, 2] = -1.0
    _, info = ops.chol_fwd(bad.to(DEV))
    assert int(info[0]) == 3 and int(info[1:].abs().max() if B > 1 else 0) == 0


def test_policy_head_and_gauss_stats():
    n, B = 63, 40
    pol = opol.BlackBoxPolicy(n, contextual=False, min_std=1e-4, dtype=torch.float64)
    g = torch.Generator().manual_seed(0)
    vec = (pol.cov_vector + 0.1 * torch.randn(pol.cov_vector.shape, generator=g, dtype=torch.float64)).float()
    vec64 = vec.double().requires_grad_(True)
    L64 = pol.vector_to_cholesky(ou.add_expand_dim(vec64, [0], [B]))
    W = torch.randn(B, n, n, generator=g, dtype=torch.float64)
    gv, = torch.autograd.grad((L64 * W).sum(), vec64)
    vec_g = vec.to(DEV).requires_grad_(True)
    L_g = ops.policy_head(vec_g, B, n, 1e-4)
    assert (f64(L_g) - L64.detach()).abs().max() < 1e-6
    (L_g * W.float().to(DEV)).sum().backward()
    assert (f64(vec_g.grad) - gv).abs().max() <= 1e-5 * gv.abs().max()
    # contextual layout [B, nvec]
    vecB = (vec[None] + 0.05 * torch.randn(B, vec.numel(), generator=g)).float()
    LB = pol.vector_to_cholesky(vecB.double())
    assert (f64(ops.policy_head(vecB.to(DEV), B, n, 1e-4)) - LB).abs().max() < 1e-6
    # Gaussian scalars
    inp = synthetic_inputs("box", B, dtype=torch.float32)
    d = lambda k: inp[k].double()
    c = lambda k: inp[k].to(DEV)
    st = f64(ops.gauss_stats(c("mean"), c("L"), c("mean_old"), c("L_old")))
    assert (st[:, 0] - pol.maha(d("mean"), d("mean_old"), d("L_old"))).abs().max() < 1e-9
    tr = (pol.precision(d("L_old")) @ pol.covariance(d("L"))).diagonal(dim1=-2, dim2=-1).sum(-1)
    assert (st[:, 1] - tr).abs().max() < 1e-8
    assert (st[:, 2] - pol.log_determinant(d("L"))).abs().max() < 1e-10
    assert (st[:, 3] - pol.log_determinant(d("L_old"))).abs().max() < 1e-10
    assert (st[:, 4] - pol.entropy([d("mean"), d("L")])).abs().max() < 1e-10


def test_empty_batch_is_a_no_op():
    """B = 0 (an empty shard of a data-parallel split): every entry point returns an empty result, no launch error."""
    name = "box"
    cfg, T, inp, times, pairs = setup_case(name, 4)
    tabs = ops.Tables(**cfg)
    c = lambda t: t.to(DEV)[:0].contiguous()
    D, P = cfg["num_dof"], pairs.shape[0]
    traj = ops.prodmp_traj(c(inp["mean"]), c(times), c(inp["init_time"]), c(inp["init_pos"]), c(inp["init_vel"]),
                           tabs.handle, D)
    assert traj.shape == (0, T, 2 * D)
    lp = ops.seg_logprob(traj, c(inp["mean"]), c(inp["L"]), c(times), c(inp["init_time"]), c(inp["init_pos"]),
                         c(inp["init_vel"]), pairs.to(DEV), tabs)
    assert lp.shape == (0, P)
    adv, ret = ops.gae(c(inp["rewards"]), c(inp["values"]), c(inp["dones"]), c(inp["time_limit_dones"]), 1.0, 0.95, True)
    assert adv.shape[0] == 0 and ret.shape[0] == 0
    z = ops.mvn_rsample(c(inp["mean"]), c(inp["L"]), c(inp["eps"]), 0, 0)
    assert z.shape[0] == 0
    torch.cuda.synchronize()


def test_surrogate_single_factor_path_equals_broadcast_path():
    """seg_surrogate on a stride-0 broadcast factor that carries its [1, n, n] origin (gradient = one GEMV batch
    sum) == the same call on a materialised [B, n, n] factor followed by the batch sum."""
    name, B = "box", 40
    cfg, T, inp, times, pairs = setup_case(name, B)
    tabs = ops.Tables(**cfg)
    c = lambda t: t.to(DEV)
    smp = ops.prodmp_traj(c(inp["mean"]) + 0.01, c(times), c(inp["init_time"]), c(inp["init_pos"]), c(inp["init_vel"]),
                          tabs.handle, cfg["num_dof"])
    P = pairs.shape[0]
    lp_old = torch.zeros(B, P, device=DEV) - 30.0
    adv = torch.linspace(-1, 1, B * P, device=DEV).reshape(B, P)
    res = []
    for mode in ("first", "dense"):
        L1 = c(inp["L"][:1]).requires_grad_(True)
        mean = c(inp["mean"]).requires_grad_(True)
        if mode == "first":
            L = L1.expand(B, -1, -1)
            L._tce_first = L1
        else:
            L = L1.expand(B, -1, -1).contiguous()
        loss, ratio, lp = ops.seg_surrogate(smp, mean, L, c(times), c(inp["init_time"]), c(inp["init_pos"]),
                                            c(inp["init_vel"]), c(pairs), lp_old, adv, tabs)
        loss.backward()
        res.append((loss.detach(), lp, mean.grad, L1.grad))
    (l0, lp0, gm0, gL0), (l1, lp1, gm1, gL1) = res
    # shared factor -> uniform-grid kernels, materialised factors -> per-episode fused kernel: two algorithms
    assert (lp0 - lp1).abs().max() <= 2e-5 and abs(l0.item() - l1.item()) <= 1e-6
    assert (gm0 - gm1).abs().max() <= 2e-5 * gm1.abs().max()
    assert gL0.shape == gL1.shape == (1,) + tuple(inp["L"].shape[1:])
    assert (gL0 - gL1).abs().max() <= 1e-4 * gL1.abs().max()


def test_staged_ops_refuse_one_factor_for_many_episodes():
    """The staged likelihood ops read L[b] for every episode b: a contiguous [1, n, n] factor with B > 1 is refused
    (shared factors go through the fused kernels).  The factor is the first matrix of a [B, n, n] buffer, so a missing
    check would read valid memory and fail the assertion rather than read out of bounds."""
    from tce_rl_b200._lib import TceError
    name, B = "box", 8
    cfg, T, inp, times, pairs = setup_case(name, B)
    tabs = ops.Tables(**cfg)
    c = lambda t: t.to(DEV)
    Dp, P = inp["mean"].shape[-1], pairs.shape[0]
    full = c(inp["L"])
    one = full[:1]
    assert one.is_contiguous() and one.shape == (1, Dp, Dp)
    smp = ops.prodmp_traj(c(inp["mean"]), c(times), c(inp["init_time"]), c(inp["init_pos"]), c(inp["init_vel"]),
                          tabs.handle, cfg["num_dof"])
    args = (c(times), c(inp["init_time"]), c(inp["init_pos"]), c(inp["init_vel"]), c(pairs))
    lp_old, adv = torch.zeros(B, P, device=DEV), torch.ones(B, P, device=DEV)
    _, work, diag_max, _ = ops.seglik_fwd(smp, c(inp["mean"]), full, *args, tabs.handle, 1e-4)
    _, _, adj, _ = ops.seglik_surrogate_fwd(smp, c(inp["mean"]), full, *args, lp_old, adv, tabs.handle, 1e-4)
    with pytest.raises(TceError, match=r"\[B, n, n\]"):
        ops.seglik_fwd(smp, c(inp["mean"]), one, *args, tabs.handle, 1e-4)
    with pytest.raises(TceError, match=r"\[B, n, n\]"):
        ops.seglik_surrogate_fwd(smp, c(inp["mean"]), one, *args, lp_old, adv, tabs.handle, 1e-4)
    with pytest.raises(TceError, match=r"\[B, n, n\]"):
        ops.seglik_bwd(torch.ones(B, P, device=DEV), work, diag_max, one, c(times), c(inp["init_time"]), c(pairs),
                       tabs.handle, 1e-4, Dp)
    with pytest.raises(TceError, match=r"\[B, n, n\]"):
        ops.seglik_surrogate_bwd(torch.ones(1, device=DEV), adj, one, c(times), c(inp["init_time"]), c(pairs),
                                 tabs.handle, Dp)
    # a stride-0 expand of the same matrix is one factor per episode and still accepted
    lp, _, _, _ = ops.seglik_fwd(smp, c(inp["mean"]), one.expand(B, -1, -1), *args, tabs.handle, 1e-4)
    assert torch.isfinite(lp).all()


@pytest.mark.parametrize("n,B", [(63, 200), (63, 203), (63, 9), (63, 3), (28, 37), (6, 64), (64, 16), (100, 12)])
def test_gauss_maha_values_and_gradients(n, B):
    """tce_gauss_maha / tce_gauss_maha_bwd_full (black_box_policy.py:183-224 ``maha``) against fp64 torch: value and the
    gradients w.r.t. both means and the factor -- through the warp-per-episode kernel (n <= 64, B >= 8), the
    CTA-per-episode kernel (few episodes, n > 64) and a broadcast factor [1, n, n]."""
    g = torch.Generator().manual_seed(n * 1000 + B)
    mean, mean_o = torch.randn(B, n, generator=g), torch.randn(B, n, generator=g)
    L = torch.tril(0.1 * torch.randn(B, n, n, generator=g), -1) + torch.diag_embed(0.5 + torch.rand(B, n, generator=g))
    w = torch.rand(B, generator=g, dtype=torch.float64)
    for shared in (False, True):
        Lc = L[:1].clone() if shared else L
        m64, o64, L64 = (t.double().requires_grad_(True) for t in (mean, mean_o, Lc))
        d = (m64 - o64)[..., None]
        z = torch.linalg.solve_triangular(L64.expand(B, n, n), d, upper=False)
        want = z.square().sum((1, 2))
        gm, go, gL = torch.autograd.grad((want * w).sum(), [m64, o64, L64])
        md, od, Ld = (t.to(DEV).requires_grad_(True) for t in (mean, mean_o, Lc))
        got = ops.gauss_maha(md, od, Ld)
        assert (got.cpu() - want.detach()).abs().max() <= 1e-5 * want.abs().max()
        g_m, g_o, g_L = torch.autograd.grad((got * w.to(DEV)).sum(), [md, od, Ld])
        assert (g_m.cpu().double() - gm).abs().max() <= 2e-5 * gm.abs().max()
        assert (g_o.cpu().double() - go).abs().max() <= 2e-5 * go.abs().max()
        assert (g_L.cpu().double() - torch.tril(gL)).abs().max() <= 5e-5 * gL.abs().max()
        assert torch.triu(g_L, 1).abs().max().item() == 0.0


@pytest.mark.parametrize("n,B", [(63, 2051), (63, 35), (24, 1203), (9, 64)])
def test_bulk_copy_kernels_large_batches(n, B):
    """The bulk-asynchronous-copy kernels (per-episode factors fetched / written as one contiguous block per group of
    four episodes: rsample and maha for odd n, the policy head for every n) with several groups per CTA and a tail of
    B % 4 episodes that runs through the row-wise kernels -- against fp64 torch."""
    g = torch.Generator().manual_seed(7 * n + B)
    mean, mean_o, eps = (torch.randn(B, n, generator=g) for _ in range(3))
    nvec = n + n * (n - 1) // 2
    vec = 0.3 * torch.randn(B, nvec, generator=g)
    # policy head (abstract_policy.py:166-187): softplus(diagonal) + min_std, strict lower triangle row by row
    L = ops.policy_head(vec.to(DEV), B, n, 1e-4)
    want = torch.zeros(B, n, n, dtype=torch.float64)
    r, c = torch.tril_indices(n, n, -1)
    want[:, r, c] = vec[:, n:].double()
    want += torch.diag_embed(torch.nn.functional.softplus(vec[:, :n].double()) + 1e-4)
    assert (f64(L) - want).abs().max() < 1e-6
    assert torch.triu(L, 1).abs().max().item() == 0.0
    # rsample with injected noise and with Philox draws (the tail must continue the same counter sequence)
    got = ops.mvn_rsample(mean.to(DEV), L, eps.to(DEV), 0, 0)
    ref = mean.double() + torch.einsum('bij,bj->bi', want, eps.double())
    assert (f64(got) - ref).abs().max() < 2e-5
    z = ops.mvn_rsample(torch.zeros(B, n, device=DEV), torch.eye(n, device=DEV).repeat(B, 1, 1), None, 11, 3)
    z_rows = ops.mvn_rsample(torch.zeros(B, n, device=DEV), torch.eye(n, device=DEV).expand(B, n, n), None, 11, 3)
    assert torch.equal(z, z_rows)                       # stride-0 factors run through the row-wise kernel
    # Mahalanobis term, value and gradients
    md, od, Ld = (t.to(DEV).requires_grad_(True) for t in (mean, mean_o, L.detach()))
    w = torch.rand(B, generator=g, dtype=torch.float64)
    maha = ops.gauss_maha(md, od, Ld)
    m64, L64 = mean.double().requires_grad_(True), want.clone().requires_grad_(True)
    zz = torch.linalg.solve_triangular(L64, (m64 - mean_o.double())[..., None], upper=False)
    mref = zz.square().sum((1, 2))
    assert (maha.cpu() - mref.detach()).abs().max() <= 1e-5 * mref.abs().max()
    gm, gL = torch.autograd.grad((mref * w).sum(), [m64, L64])
    g_m, g_o, g_L = torch.autograd.grad((maha * w.to(DEV)).sum(), [md, od, Ld])
    assert (g_m.cpu().double() - gm).abs().max() <= 2e-5 * gm.abs().max()
    assert (g_o.cpu().double() + gm).abs().max() <= 2e-5 * gm.abs().max()
    assert (g_L.cpu().double() - torch.tril(gL)).abs().max() <= 5e-5 * gL.abs().max()

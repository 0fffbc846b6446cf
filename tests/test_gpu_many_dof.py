"""ProDMP policies with 9 to 16 degrees of freedom (two 7-DoF arms, 16-joint hands): tables, trajectories, the dense
likelihood on the staged kernels (the per-segment factorisation runs one warp per segment above 8 DoF), the diagonal
likelihood, policy epochs and CUDA-graph updates, against the fp64 CPU oracle and against the 8-DoF kernels on
duplicated DoF."""
import pytest
import torch

from oracle import util as ou
from oracle.gen_golden import MP_CONFIGS, NUM_TIMES

pytestmark = pytest.mark.gpu
if torch.cuda.is_available():
    import test_gpu_any_shape as tas
    import test_gpu_diag_shapes as tds
    from test_gpu_kernels import _lib_launch_count
    from tce_rl_b200 import ops, ops_seglik
    from tce_rl_b200._lib import TceError

DEV = "cuda:0"
DENSE = [(9, 7), (10, 6), (12, 5), (14, 4), (16, 4), (16, 2)]


def f64(t):
    return t.detach().double().cpu()


def cfg_of(D, K1, task="box"):
    return dict(MP_CONFIGS[task], num_dof=D, num_basis=K1 - 1)


# ---- tables --------------------------------------------------------------------------------------------------------
def test_tables_do_not_depend_on_num_dof():
    ref = ops.Tables(**cfg_of(7, 5)).export()
    for D in (9, 14, 16):
        tabs = ops.Tables(**cfg_of(D, 5))
        assert not tabs.compiled and tabs.dense_likelihood == (D * 5 <= 64)
        got = tabs.export()
        for k in ref:
            assert torch.equal(got[k], ref[k]), (D, k)
    for D, K1 in [(17, 2), (9, 15), (16, 9)]:
        with pytest.raises(TceError, match="unsupported"):
            ops.Tables(**cfg_of(D, K1))
    assert not ops.Tables(**cfg_of(16, 8)).dense_likelihood        # 128 parameters: diagonal likelihood only


# ---- trajectories --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D,K1", [(9, 7), (9, 14), (14, 4), (14, 9), (16, 2), (16, 8)])
@pytest.mark.parametrize("T", [1, 31, 33])
def test_trajectory_matches_oracle(D, K1, T):
    cfg = cfg_of(D, K1, "metaworld" if K1 == 9 else "box")
    B = 64                                              # >= 64: a common time grid takes the uniform kernels
    inp = tas.inputs(D, K1, B, seed=D * 17 + K1)
    tabs = ops.Tables(**cfg)
    omp = tas.ou_mp(cfg)
    c = lambda t: t.to(DEV)
    for uniform in (False, True):
        init_time = inp["init_time"][:1].expand(B).contiguous() if uniform else inp["init_time"]
        times = ou.get_times(init_time.double(), T, cfg["dt"]).float()
        params = c(inp["mean"]).requires_grad_(True)
        ip, iv = c(inp["init_pos"]).requires_grad_(True), c(inp["init_vel"]).requires_grad_(True)
        n0 = _lib_launch_count("tce_prodmp_traj_fwd_uniform")
        traj = ops.prodmp_traj(params, c(times), c(init_time), ip, iv, tabs.handle, D)
        assert _lib_launch_count("tce_prodmp_traj_fwd_uniform") == n0 + int(uniform)
        p64 = inp["mean"].double().requires_grad_(True)
        ip64, iv64 = inp["init_pos"].double().requires_grad_(True), inp["init_vel"].double().requires_grad_(True)
        omp.update_inputs(times.double(), p64, None, init_time.double(), ip64, iv64)
        ref = torch.cat([omp.get_traj_pos(), omp.get_traj_vel()], -1)
        assert traj.shape == ref.shape == (B, T, 2 * D)
        assert (f64(traj) - ref).abs().max() <= 1e-5 * ref.abs().max()
        w = torch.linspace(-1, 1, ref.numel(), dtype=torch.float64).reshape(ref.shape)
        refs = torch.autograd.grad((ref * w).sum(), [p64, ip64, iv64])
        (traj * c(w.float())).sum().backward()
        for got, want in zip((params.grad, ip.grad, iv.grad), refs):
            assert (f64(got) - want).abs().max() <= 1e-5 * want.abs().max()


# ---- dense likelihood ----------------------------------------------------------------------------------------------
def _staged_routes():
    return {k: _lib_launch_count(k) for k in ("tce_seglik_gram", "tce_seglik_gram_sigma", "tce_seglik_chol",
                                              "tce_seglik_fused", "tce_seglik_uniform_main")}


@pytest.mark.parametrize("D,K1", DENSE)
@pytest.mark.parametrize("cov", ["episode", "shared_L", "shared_sigma"])
@pytest.mark.parametrize("B,P,ragged", [(33, 25, False), (1, 1, False), (33, 7, True), (1024, 25, False),
                                        (2, 128, False)])
def test_likelihood_matches_oracle(D, K1, cov, B, P, ragged, monkeypatch):
    if B == 1024 and (D, K1) not in [(9, 7), (16, 4)]:
        pytest.skip("B = 1024 on the first and the widest shape only")
    if P == 128:                                        # 129 chained time points: the metaworld horizon (500 steps)
        monkeypatch.setitem(tas.TASK, (D, K1), "metaworld")
    before = _staged_routes()
    tas.test_likelihood_matches_oracle(D, K1, cov, B, P, ragged)
    after = _staged_routes()
    gram = "tce_seglik_gram_sigma" if cov == "shared_sigma" else "tce_seglik_gram"
    assert after[gram] - before[gram] == 3 and after["tce_seglik_chol"] - before["tce_seglik_chol"] == 3
    assert after["tce_seglik_fused"] == before["tce_seglik_fused"]
    assert after["tce_seglik_uniform_main"] == before["tce_seglik_uniform_main"]


@pytest.mark.parametrize("D,K1", [(9, 7), (16, 4)])
@pytest.mark.parametrize("cov", ["episode", "shared_L"])
def test_one_hot_upstream_on_first_and_last_segment(D, K1, cov):
    """A lost or misplaced adjoint of a single segment shows: the upstream gradient is 1 on one segment only."""
    B, P = 5, 25
    cfg, inp, times, pairs, pol, smp, args64 = tas.lik_case(D, K1, B, P, False, seed=11)
    tabs = ops.Tables(**cfg)
    c = lambda t: t.to(DEV)
    L = c(inp["L"]) if cov == "episode" else c(inp["L"][:1])
    for b, p in [(0, 0), (B - 1, P - 1)]:
        w = torch.zeros(B, P, dtype=torch.float64)
        w[b, p] = 1.0
        mean64 = inp["mean"].double().requires_grad_(True)
        L64 = (inp["L"] if cov == "episode" else inp["L"][:1]).double().requires_grad_(True)
        lp = pol.log_prob(smp.double(), mean64, L64.expand(B, -1, -1), *args64, pred_pairs=pairs)
        gm_ref, gL_ref = torch.autograd.grad((lp * w).sum(), [mean64, L64])
        gL_ref = torch.tril(gL_ref)
        _, _, _, gm, gL, _ = tas.run_seglik(tabs, smp, c(inp["mean"]), L, None, times, inp, pairs, 1,
                                            grad_logp=c(w.float()), want_L=True)
        assert (f64(gm) - gm_ref).abs().max() <= 2e-4 * gm_ref.abs().max()
        assert (f64(gL).reshape(gL_ref.shape) - gL_ref).abs().max() <= 2e-4 * gL_ref.abs().max()
        assert float(torch.triu(gL, 1).abs().max()) == 0.0


def _duplicate(inp, smp, D):
    """The 2D-DoF case whose DoF D..2D-1 copy DoF 0..D-1: same means, block-diagonal factors, same trajectories."""
    out = dict(inp)
    out["mean"] = torch.cat([inp["mean"], inp["mean"]], -1)
    out["L"] = torch.stack([torch.block_diag(Lb, Lb) for Lb in inp["L"]])
    out["init_pos"] = torch.cat([inp["init_pos"], inp["init_pos"]], -1)
    out["init_vel"] = torch.cat([inp["init_vel"], inp["init_vel"]], -1)
    pos, vel = smp[..., :D], smp[..., D:]
    return out, torch.cat([pos, pos, vel, vel], -1)


@pytest.mark.parametrize("D,K1", [(8, 4), (5, 6)])
def test_duplicated_dof_match_the_shipped_kernel(D, K1):
    B, P = 40, 25
    cfg, inp, times, pairs, pol, smp, _ = tas.lik_case(D, K1, B, P, False, seed=3)
    inp2, smp2 = _duplicate(inp, smp, D)
    tabs, tabs2 = ops.Tables(**cfg), ops.Tables(**dict(cfg, num_dof=2 * D))
    c = lambda t: t.to(DEV)
    w = c(torch.linspace(0.5, 1.5, B * P).reshape(B, P))
    lp1, info1, acc1, gm1, gL1, _ = tas.run_seglik(tabs, smp, c(inp["mean"]), c(inp["L"]), None, times, inp, pairs, 1,
                                                   grad_logp=w, want_L=True)
    lp2, info2, acc2, gm2, gL2, _ = tas.run_seglik(tabs2, smp2, c(inp2["mean"]), c(inp2["L"]), None, times, inp2,
                                                   pairs, 1, grad_logp=w, want_L=True)
    l0, _, _, _, _, _ = tas.run_seglik(tabs2, smp2, c(inp2["mean"]), c(inp2["L"]), None, times, inp2, pairs, 0)
    assert torch.equal(l0, lp2)                         # grad mode 0 and 1 give the same log-probs
    assert int(info1.abs().max()) == 0 and int(info2.abs().max()) == 0
    assert torch.equal(acc1[0], acc2[0])                # the same regulariser seed
    assert (lp2.double() - 2 * lp1.double()).abs().max().item() <= 1e-4
    Dp = D * K1
    scale = gm1.abs().max().item()
    for h in (0, 1):
        assert (gm2[:, h * Dp:(h + 1) * Dp] - gm1).abs().max().item() <= 1e-4 * scale
    scale = gL1.abs().max().item()
    for h in (0, 1):
        blk = gL2[:, h * Dp:(h + 1) * Dp, h * Dp:(h + 1) * Dp]
        assert (blk - gL1).abs().max().item() <= 1e-4 * scale


@pytest.mark.parametrize("D,K1,d", [(9, 7, 8), (16, 4, 9), (16, 4, 15)])
def test_first_non_positive_pivot(D, K1, d):
    B, P = 3, 25
    cfg, inp, times, pairs, pol, smp, _ = tas.lik_case(D, K1, B, P, False, seed=7)
    L = inp["L"].clone()
    L[:, d * K1:(d + 1) * K1, :] = 0.0                  # DoF d has no variance: rows (2d, 2d + 1) of C vanish
    tabs = ops.Tables(**cfg)
    c = lambda t: t.to(DEV)
    _, info, _ = ops.seg_logprob_staged(c(smp), c(inp["mean"]), c(L), c(times), c(inp["init_time"]),
                                        c(inp["init_pos"]), c(inp["init_vel"]), c(pairs), tabs, reg_rel=0.0,
                                        return_info=True)
    assert torch.equal(info.cpu(), torch.full((B, P), 2 * d + 1, dtype=torch.int32))


def _gram_smem(D, K1, P):
    """Shared memory of the gram kernel (gram_smem, csrc/tce_seglik.cu): it bounds P for every layout."""
    Dp = D * K1
    NR, NR4 = (Dp + 1) & ~1, (Dp + 3) & ~3
    return 8 * (NR * (NR + 1) + 2 * P * K1 + 4 * P + 5 + 2 * K1 + 1) + 4 * NR4 * (NR4 + 1) + 16


def test_segment_count_bound():
    D, K1 = 16, 4
    Pmax = max(P for P in range(1, 4097) if _gram_smem(D, K1, P) <= 200 * 1024)
    assert Pmax == 1612
    cfg = cfg_of(D, K1)
    tabs = ops.Tables(**cfg)
    T, B, Dp = 50, 1, D * K1
    inp = tas.inputs(D, K1, B, seed=2)
    times = ou.get_times(inp["init_time"].double(), T, cfg["dt"]).float()
    c = lambda t: t.to(DEV)
    smp = c(torch.zeros(B, T, 2 * D))
    for P in (Pmax, Pmax + 1):
        pairs = torch.tensor([[3, 9]]).expand(P, 2).contiguous()
        mean, L = c(inp["mean"]).requires_grad_(True), c(inp["L"]).requires_grad_(True)
        args = (c(times), c(inp["init_time"]), c(inp["init_pos"]), c(inp["init_vel"]), c(pairs), tabs)
        if P == Pmax:
            lp = ops.seg_logprob_staged(smp, mean, L, *args)
            lp.sum().backward()
            assert torch.isfinite(lp).all() and torch.isfinite(L.grad).all()
        else:
            n0 = _lib_launch_count("tce_seglik_chol")
            with pytest.raises(TceError, match="unsupported"):
                ops.seg_logprob_staged(smp, mean, L, *args)
            assert _lib_launch_count("tce_seglik_chol") == n0


@pytest.mark.parametrize("D,K1", [(9, 8), (16, 5)])
def test_full_covariance_above_64_parameters_still_raises(D, K1):
    tabs = ops.Tables(**cfg_of(D, K1))
    assert not tabs.compiled and not tabs.dense_likelihood
    B, P, T, Dp = 4, 25, NUM_TIMES["box"], D * K1
    z = lambda *s: torch.zeros(*s, device=DEV)
    pairs = ou.get_time_pairs(T, dict(num_select=26, fixed_interval=True))[:25].to(DEV)
    eye = torch.eye(Dp, device=DEV).expand(B, -1, -1).contiguous()
    for L in (eye, eye[:1]):
        with pytest.raises(TceError, match="unsupported"):
            ops_seglik.seglik(z(B, T, 2 * D), z(B, Dp), L, None, None, z(B, T), z(B), z(B, D), z(B, D), pairs,
                              tabs.handle, 1e-4, 0, None, None, None, True, False, False)


@pytest.mark.parametrize("D,K1", [(14, 4), (16, 4)])
def test_cross_paths_and_traj_pos_cov(D, K1):
    """Per-episode, shared-L and shared-Sigma layouts agree, the diagonal likelihood equals the dense one on diagonal
    factors, and the public entry points and mp.ProDMP.get_traj_pos_cov match the oracle."""
    tas.test_cross_paths_on_new_shapes(D, K1)


# ---- diagonal likelihood -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D,K1", [(16, 8), (12, 10), (9, 14)])
@pytest.mark.parametrize("B,P,ragged,layout", [(1024, 24, False, "dense"), (33, 25, False, "packed"),
                                               (17, 7, True, "shared"), (64, 25, False, "shared")])
def test_diag_likelihood_matches_oracle(D, K1, B, P, ragged, layout):
    n0 = _lib_launch_count("tce_seglik_diag_fwd")
    tds.test_diag_likelihood_matches_oracle(D, K1, B, P, ragged, layout)
    assert _lib_launch_count("tce_seglik_diag_fwd") == n0 + 1


# ---- policy epochs -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D,K1,typ,contextual,std_only", [
    (14, 4, "KLProjectionLayer", False, False),       # the hand-scheduled shared-covariance KL epoch
    (14, 4, "KLProjectionLayer", True, False),
    (14, 4, "WassersteinProjectionLayer", False, False),
    (14, 4, "FrobeniusProjectionLayer", False, False),
    (16, 8, "KLProjectionLayer", False, True),
    (16, 8, "KLProjectionLayer", True, True)])
def test_policy_epoch_matches_oracle(D, K1, typ, contextual, std_only):
    tas.test_policy_epoch_matches_oracle(D, K1, typ, contextual, std_only)


def test_graph_captured_update_equals_eager():
    import test_gpu_agent
    from oracle import gen_golden
    name = "_many_dof_14x4"
    gen_golden.MP_CONFIGS[name], gen_golden.NUM_TIMES[name] = cfg_of(14, 4), NUM_TIMES["box"]
    try:
        outs, params = [], []
        for use_graph in (False, True):
            agent, dataset = test_gpu_agent.build(name=name, B=64, use_graph=use_graph, epochs=3)
            assert agent.policy.num_dof == 14 and not agent.policy.mp.tables.compiled
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

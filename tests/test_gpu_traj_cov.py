"""mp.ProDMP.get_traj_pos_cov / get_traj_pos_std on any time grid (tce::traj_pos_cov, tce::traj_pos_std) against the
fp64 CPU oracle: values, gradients w.r.t. params_L, every shape the tables accept up to 128 parameters, per-episode,
common and pair grids, per-episode, shared and batched factors, determinism of the shared-factor gradient, the
empty batch, the previous pair-only computation, and eager against CUDA-graph calls."""
import pytest
import torch

from oracle import util as ou
from oracle.gen_golden import MP_CONFIGS

pytestmark = pytest.mark.gpu
if torch.cuda.is_available():
    import test_gpu_any_shape as tas
    from tce_rl_b200 import _lib, mp as gmp, ops

DEV = "cuda:0"
SHAPES = [(7, 9), (3, 4), (1, 2), (9, 7), (16, 4), (14, 9), (16, 8)]


def f64(t):
    return t.detach().double().cpu()


def cfg_of(D, K1):
    return dict(MP_CONFIGS["box"], num_dof=D, num_basis=K1 - 1)


def close(got, want, rel):
    return (f64(got) - want).abs().max().item() <= rel * want.abs().max().item()


def case(D, K1, B, T, seed, common=False):
    inp = tas.inputs(D, K1, B, seed=seed)
    init_time = inp["init_time"][:1].expand(B).contiguous() if common else inp["init_time"]
    times = ou.get_times(init_time.double(), T, cfg_of(D, K1)["dt"]).float()
    return times, inp["L"], init_time


def pos_std(cov, D):
    """mp_pytorch's get_traj_pos_std restated on the oracle's covariance: sqrt of its diagonal (rows DoF-major) as
    [*a, T, D]."""
    diag = torch.diagonal(cov, dim1=-2, dim2=-1)
    return torch.sqrt(diag).reshape(*diag.shape[:-1], D, -1).transpose(-1, -2)


def oracle(cfg, times, L64, init_time, w_cov=None, w_std=None, reg=1e-4):
    """(cov, std, d(sum w_cov cov + sum w_std std) / d L64) of the fp64 oracle; L64 may be an expand of a leaf."""
    omp = tas.ou_mp(cfg)
    cov = omp.get_traj_pos_cov(times.double(), L64, init_time.double(), reg=reg)
    std = pos_std(cov, cfg["num_dof"])
    grad = None
    if w_cov is not None:
        leaf = L64 if L64.is_leaf else L64._base
        grad, = torch.autograd.grad((cov * w_cov).sum() + (std * w_std).sum(), leaf)
    return cov.detach(), std.detach(), grad


def run(tabs, times, L, init_time, w_cov=None, w_std=None, reg=1e-4):
    mp = gmp.ProDMP(tabs)
    cov = mp.get_traj_pos_cov(times.to(DEV), L, init_time.to(DEV), reg=reg)
    std = mp.get_traj_pos_std(reg=reg)
    grad = None
    if w_cov is not None:
        leaf = L if L.is_leaf else L._base
        grad, = torch.autograd.grad((cov * w_cov.to(DEV)).sum() + (std * w_std.to(DEV)).sum(), leaf)
    return cov, std, grad


def weights(cov_shape, std_shape, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(cov_shape, generator=g, dtype=torch.float64), torch.randn(std_shape, generator=g,
                                                                                 dtype=torch.float64)


def check_consistent(cov, std, D, T):
    diag = torch.diagonal(f64(cov), dim1=-2, dim2=-1)                              # DoF-major
    s2 = (f64(std) ** 2).transpose(-1, -2).reshape(diag.shape)
    assert (s2 - diag).abs().max().item() <= 1e-5 * diag.abs().max().item()
    torch.linalg.cholesky(f64(cov))                                                 # SPD with the regulariser


@pytest.mark.parametrize("D,K1", SHAPES)
@pytest.mark.parametrize("T", [1, 2, 31, 33, 100])
def test_per_episode_grids_and_factors_match_oracle(D, K1, T):
    B = 5 if D * T > 400 else 9
    times, L, init_time = case(D, K1, B, T, seed=D * 31 + K1 + T)
    tabs = ops.Tables(**cfg_of(D, K1))
    wc, ws = weights((B, D * T, D * T), (B, T, D), seed=T)
    cov_w, std_w, g_w = oracle(cfg_of(D, K1), times, L.double().requires_grad_(True), init_time, wc, ws)
    cov, std, g = run(tabs, times, L.to(DEV).requires_grad_(True), init_time, wc, ws)
    assert cov.shape == cov_w.shape and std.shape == std_w.shape == (B, T, D)
    assert close(cov, cov_w, 1e-5) and close(std, std_w, 1e-5)
    assert close(g, torch.tril(g_w), 2e-4)
    assert torch.equal(torch.triu(g, 1), torch.zeros_like(g))
    check_consistent(cov, std, D, T)
    flat = gmp.ProDMP(tabs).get_traj_pos_std(times.to(DEV), L.to(DEV), init_time.to(DEV), flat_shape=True)
    assert torch.equal(flat, std.transpose(-1, -2).reshape(B, D * T))


@pytest.mark.parametrize("D,K1", [(7, 9), (3, 4), (16, 8)])
@pytest.mark.parametrize("B", [1, 33])
def test_common_grid_shared_and_batched_factors(D, K1, B):
    T = 33
    Dp = D * K1
    cfg = cfg_of(D, K1)
    tabs = ops.Tables(**cfg)
    times, L, init_time = case(D, K1, B, T, seed=7 * D + B, common=True)
    wc, ws = weights((B, D * T, D * T), (B, T, D), seed=B)
    # one factor broadcast over the batch (stride 0): read once, gradient summed over the batch in a fixed order
    L1 = L[0]
    cov_w, std_w, g_w = oracle(cfg, times, L1.double().requires_grad_(True).expand(B, Dp, Dp), init_time, wc, ws)
    Lg = L1.to(DEV).requires_grad_(True)
    cov, std, g = run(tabs, times, Lg.expand(B, Dp, Dp), init_time, wc, ws)
    assert close(cov, cov_w, 1e-5) and close(std, std_w, 1e-5) and close(g, torch.tril(g_w), 2e-4)
    _, _, g2 = run(tabs, times, Lg.expand(B, Dp, Dp), init_time, wc, ws)
    assert torch.equal(g, g2)
    check_consistent(cov, std, D, T)
    # [*a]-batched factors and grids: [3, B, ...]
    times3 = torch.stack([times, times + 0.01, times + 0.02])
    it3 = torch.stack([init_time, init_time + 0.01, init_time + 0.02])
    L3 = torch.stack([L, 0.5 * L, 2.0 * L])
    wc3, ws3 = weights((3, B, D * T, D * T), (3, B, T, D), seed=B + 1)
    cov_w, std_w, g_w = oracle(cfg, times3, L3.double().requires_grad_(True), it3, wc3, ws3)
    cov, std, g = run(tabs, times3, L3.to(DEV).requires_grad_(True), it3, wc3, ws3)
    assert cov.shape == (3, B, D * T, D * T) and std.shape == (3, B, T, D)
    assert close(cov, cov_w, 1e-5) and close(std, std_w, 1e-5) and close(g, torch.tril(g_w), 2e-4)


def _gram_pair_cov(tabs, times2, L3, init_time, reg):
    """The pair-only computation mp.ProDMP.get_traj_pos_cov ran before it took any grid: the gram stage of the staged
    likelihood on zero trajectories, mirrored and regularised on the host."""
    n, D, Dp = times2.shape[0], tabs.num_dof, tabs.dim_params
    dev = times2.device
    zeros, zpos = torch.zeros(n, Dp, device=dev), torch.zeros(n, D, device=dev)
    pairs = torch.tensor([[0, 1]], device=dev, dtype=torch.int64)
    smp = torch.zeros(n, 2, 2 * D, device=dev)
    work = ops._work(tabs.handle, n, 1, dev)
    dmax = torch.zeros(1, device=dev, dtype=torch.float64)
    Lc, ldb = ops._batched_matrix(L3)
    _lib.call("tce_seglik_gram", tabs.handle, smp.data_ptr(), zeros.data_ptr(), Lc.data_ptr(), ldb,
              times2.contiguous().data_ptr(), init_time.data_ptr(), zpos.data_ptr(), zpos.data_ptr(), pairs.data_ptr(),
              work.data_ptr(), dmax.data_ptr(), n, 2, 1, ops._stream())
    N = 2 * D
    tri = work[:n * N * (N + 1) // 2].reshape(n, N * (N + 1) // 2)
    r, c = torch.tril_indices(N, N, device=dev)
    cov = torch.zeros(n, N, N, device=dev, dtype=torch.float64)
    cov[:, r, c] = tri
    cov[:, c, r] = tri
    return (cov + torch.eye(N, device=dev, dtype=torch.float64) * (dmax * reg)).float()


@pytest.mark.parametrize("D,K1", [(7, 9), (3, 4), (9, 7)])
def test_pair_grids_as_tce_passes_them(D, K1):
    B, T, Dp = 33, 100, D * K1
    cfg = cfg_of(D, K1)
    tabs = ops.Tables(**cfg)
    times, L, init_time = case(D, K1, B, T, seed=D + K1)
    torch.manual_seed(0)
    pairs = ou.get_time_pairs(T, dict(num_select=25, fixed_interval=True))
    P = pairs.shape[0]
    tp = times[:, pairs]                                                          # [B, P, 2]
    ex = lambda t: t.unsqueeze(1).expand(B, P, *t.shape[1:])
    wc, ws = weights((B, P, 2 * D, 2 * D), (B, P, 2, D), seed=P)
    cov_w, std_w, g_w = oracle(cfg, tp, ex(L.double().requires_grad_(True)), ex(init_time), wc, ws)
    Lg = L.to(DEV).requires_grad_(True)
    cov, std, g = run(tabs, tp, ex(Lg), ex(init_time), wc, ws)
    assert cov.shape == (B, P, 2 * D, 2 * D)
    assert close(cov, cov_w, 1e-5) and close(std, std_w, 1e-5) and close(g, torch.tril(g_w), 2e-4)
    check_consistent(cov, std, D, 2)
    # the previous pair-only computation (fp32 L L^T in its gram stage)
    old = _gram_pair_cov(tabs, tp.reshape(B * P, 2).to(DEV), ex(L).reshape(B * P, Dp, Dp).to(DEV).contiguous(),
                         ex(init_time).reshape(-1).to(DEV).contiguous(), 1e-4)
    assert close(cov.reshape(B * P, 2 * D, 2 * D), f64(old), 3e-5)
    # one-hot upstream gradients on entries of off-diagonal DoF blocks (and their mirror images)
    L64 = ex(L.double().requires_grad_(True))
    cov_o = tas.ou_mp(cfg).get_traj_pos_cov(tp.double(), L64, ex(init_time).double())
    for (b, p, i, j) in [(0, 0, 0, 2 * D - 1), (B - 1, P - 1, 2 * D - 2, 1), (5, 7, 2, 3)]:
        want, = torch.autograd.grad(cov_o[b, p, i, j], L64._base, retain_graph=True)
        Lg.grad = None
        cov = gmp.ProDMP(tabs).get_traj_pos_cov(tp.to(DEV), ex(Lg), ex(init_time).to(DEV))
        cov[b, p, i, j].backward()
        assert close(Lg.grad, torch.tril(want), 2e-4), (b, p, i, j)


def _ref_diag(cfg, times, L, init_time):
    """diag(F F^T) [B, D, T] in fp64 without the D T x D T matrices."""
    omp = tas.ou_mp(cfg)
    omp.update_inputs(times.double(), None, L.double(), init_time.double())
    Hp = omp._terms()[4]                                                          # [B, T, K1]
    D, K1 = cfg["num_dof"], cfg["num_basis"] + 1
    F = torch.einsum('btk,bdkj->bdtj', Hp, L.double().reshape(L.shape[0], D, K1, -1))
    return (F ** 2).sum(-1)


@pytest.mark.parametrize("D,K1,T,shared", [(3, 4, 31, False), (7, 9, 100, False), (16, 8, 100, True)])
def test_large_batch(D, K1, T, shared):
    B, Dp = 1024, D * K1
    cfg = cfg_of(D, K1)
    tabs = ops.Tables(**cfg)
    times, L, init_time = case(D, K1, B, T, seed=11)
    if shared:
        L = L[:1].expand(B, Dp, Dp)
    Lg = (L[0] if shared else L).to(DEV).requires_grad_(True)
    Lin = Lg.expand(B, Dp, Dp) if shared else Lg
    mp = gmp.ProDMP(tabs)
    cov = mp.get_traj_pos_cov(times.to(DEV), Lin, init_time.to(DEV))
    std = mp.get_traj_pos_std()
    r = 1e-4 * _ref_diag(cfg, times, L, init_time).max().item()
    for b in (0, B // 2, B - 1):
        omp = tas.ou_mp(cfg)
        want = omp.get_traj_pos_cov(times[b:b + 1].double(), L[b:b + 1].double(), init_time[b:b + 1].double(),
                                    reg_override=r)
        assert close(cov[b:b + 1], want, 1e-5), b
        assert close(std[b:b + 1], torch.sqrt(torch.diagonal(want, dim1=-2, dim2=-1)).reshape(1, D, T)
                     .transpose(-1, -2), 1e-5), b
    w = torch.randn(cov.shape, device=DEV, generator=torch.Generator(DEV).manual_seed(1))
    g1, = torch.autograd.grad((cov * w).sum(), Lg, retain_graph=True)
    g2, = torch.autograd.grad((cov * w).sum(), Lg)
    assert torch.equal(g1, g2)
    if shared:
        # the batch-summed gradient of the shared factor == the sum of the per-episode gradients
        Le = Lg.detach().expand(B, Dp, Dp).contiguous().requires_grad_(True)
        ge, = torch.autograd.grad((gmp.ProDMP(tabs).get_traj_pos_cov(times.to(DEV), Le, init_time.to(DEV)) * w).sum(),
                                  Le)
        gsum = ge.double().sum(0)
        assert (g1.double() - gsum).abs().max().item() <= 2e-4 * gsum.abs().max().item()


def test_empty_batch():
    D, K1, T = 7, 9, 5
    tabs = ops.Tables(**cfg_of(D, K1))
    L = torch.zeros(0, D * K1, D * K1, device=DEV, requires_grad=True)
    mp = gmp.ProDMP(tabs)
    cov = mp.get_traj_pos_cov(torch.zeros(0, T, device=DEV), L, torch.zeros(0, device=DEV))
    std = mp.get_traj_pos_std()
    assert cov.shape == (0, D * T, D * T) and std.shape == (0, T, D)
    g, = torch.autograd.grad(cov.sum() + std.sum(), L)
    assert g.shape == L.shape


def test_invalid_arguments_are_refused():
    tabs = ops.Tables(**cfg_of(3, 4))
    lib = _lib.load()
    assert lib.tce_prodmp_traj_cov_work_bytes(tabs.handle, 4, 10, 144, 4) == 0
    assert lib.tce_prodmp_traj_cov_work_bytes(tabs.handle, 4, 0, 144, 0) == 0
    L = torch.eye(12, device=DEV).expand(4, 12, 12).contiguous()
    times, it = torch.zeros(4, 3, device=DEV), torch.zeros(4, device=DEV)
    with pytest.raises(_lib.TceError, match="invalid"):
        ops.traj_pos_cov(L, times[:, :0], it, tabs.handle, 3, 1e-4)
    with pytest.raises(_lib.TceError):
        ops.traj_pos_cov(L[:2], times, it, tabs.handle, 3, 1e-4)


def test_graph_captured_calls_equal_eager():
    D, K1, B, T = 14, 9, 17, 33
    tabs = ops.Tables(**cfg_of(D, K1))
    times, L, init_time = case(D, K1, B, T, seed=2)
    Lg = L.to(DEV).requires_grad_(True)
    wc, ws = (w.float().to(DEV) for w in weights((B, D * T, D * T), (B, T, D), seed=3))
    mp = gmp.ProDMP(tabs)
    mp.update_inputs(times=times.to(DEV), params_L=Lg, init_time=init_time.to(DEV))

    def step():
        cov, std = mp.get_traj_pos_cov(), mp.get_traj_pos_std()
        g, = torch.autograd.grad((cov * wc).sum() + (std * ws).sum(), Lg)
        return cov, std, g

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eager = [t.clone() for t in step()]
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = step()
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(eager, out):
        assert torch.equal(a, b)

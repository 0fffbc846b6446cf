"""mp_pytorch's ProDMP.get_traj_pos_std, restated on the oracle as the sqrt of the diagonal of get_traj_pos_cov (the
reference the GPU tests use), against the Monte-Carlo spread of the oracle's sample_trajectories, and its two output
layouts (CPU only)."""
import torch

from oracle.gen_golden import MP_CONFIGS
from oracle.prodmp import get_mp
from oracle import util as ou


def pos_std(mp, times, L, t0, y0, v0, flat_shape=False, reg=1e-4):
    """sqrt(diag(get_traj_pos_cov)) with its batch-global regulariser: [*a, T, D], or [*a, D*T] DoF-major."""
    cov = mp.get_traj_pos_cov(times, L, t0, y0, v0, reg=reg)
    std = torch.sqrt(torch.einsum('...ii->...i', cov))
    return std if flat_shape else std.reshape(*std.shape[:-1], mp.num_dof, -1).transpose(-1, -2)


def _case(D, K1, B, T, seed=3):
    cfg = dict(MP_CONFIGS["box"], num_dof=D, num_basis=K1 - 1)
    g = torch.Generator().manual_seed(seed)
    Dp = D * K1
    L = torch.tril(0.05 * torch.randn(B, Dp, Dp, generator=g, dtype=torch.float64), -1) + \
        torch.diag_embed(torch.nn.functional.softplus(torch.randn(B, Dp, generator=g, dtype=torch.float64)) + 1e-4)
    init_time = torch.rand(B, generator=g, dtype=torch.float64) * 0.3
    times = ou.get_times(init_time, T, cfg["dt"])
    mean = 0.5 * torch.randn(B, Dp, generator=g, dtype=torch.float64)
    init_pos = torch.rand(B, D, generator=g, dtype=torch.float64) * 2 - 1
    init_vel = 0.1 * torch.randn(B, D, generator=g, dtype=torch.float64)
    return get_mp(type="prodmp", args=dict(cfg)), times, mean, L, init_time, init_pos, init_vel, g


def test_pos_std_is_the_spread_of_sampled_trajectories():
    B, T, S = 2, 40, 20000
    mp, times, mean, L, t0, y0, v0, g = _case(3, 4, B, T)
    std = pos_std(mp, times, L, t0, y0, v0, reg=0.0)                    # [B, T, D]
    eps = torch.randn(S, B, mean.shape[-1], generator=g, dtype=torch.float64)
    pos, _ = mp.sample_trajectories(times, mean, L, t0, y0, v0, num_smp=S, eps=eps)   # [B, S, T, D]
    var_mc = pos.var(dim=1)
    var = std ** 2
    # the sample variance of S Gaussian draws has a relative standard error sqrt(2 / (S - 1)) (0.01 here)
    tol = 5 * (2 / (S - 1)) ** 0.5 * var + 1e-12 * var.max()
    assert tuple(std.shape) == (B, T, 3)
    assert bool(((var_mc - var).abs() <= tol).all())


def test_pos_std_layouts_and_regulariser():
    B, T = 3, 7
    mp, times, mean, L, t0, y0, v0, _ = _case(2, 3, B, T)
    cov, r = mp.get_traj_pos_cov(times, L, t0, y0, v0, return_reg=True)
    std = pos_std(mp, times, L, t0, y0, v0)
    flat = pos_std(mp, times, L, t0, y0, v0, flat_shape=True)
    diag = torch.einsum('...ii->...i', cov)                                      # DoF-major
    assert r > 0 and torch.equal(flat, torch.sqrt(diag))
    assert torch.equal(std, flat.reshape(B, 2, T).transpose(-1, -2))

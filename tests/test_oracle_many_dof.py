"""The fp64 CPU oracle's segment likelihood above 8 degrees of freedom (14 and 16 DoF, the shapes of two 7-DoF arms and
of 16-joint hands): every segment log-prob equals ``scipy.stats.multivariate_normal.logpdf`` on the mean and the
covariance H Sigma H^T + reg I built here from the basis rows, DoF by DoF.  CPU only."""
import numpy as np
import pytest
import torch
from scipy.stats import multivariate_normal

from oracle import policy as opol
from oracle import util as ou
from oracle.gen_golden import MP_CONFIGS, NUM_TIMES


@pytest.mark.parametrize("D,K1", [(14, 4), (16, 4), (16, 2)])
def test_segment_log_prob_equals_scipy(D, K1):
    cfg = dict(MP_CONFIGS["box"], num_dof=D, num_basis=K1 - 1)
    T, B, Dp = NUM_TIMES["box"], 3, D * K1
    g = torch.Generator().manual_seed(D * 100 + K1)
    rn = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    mean = 0.5 * rn(B, Dp)
    L = torch.tril(0.05 * rn(B, Dp, Dp), -1) + torch.diag_embed(torch.nn.functional.softplus(rn(B, Dp)) + 1e-4)
    init_time = torch.rand(B, generator=g, dtype=torch.float64) * 0.3
    init_pos = torch.rand(B, D, generator=g, dtype=torch.float64) * 2 - 1
    init_vel = 0.1 * rn(B, D)
    times = ou.get_times(init_time, T, cfg["dt"])
    pairs = torch.tensor([[0, 4], [4, 8], [10, 50], [T - 2, T - 1]])
    pol = opol.TemporalCorrelatedPolicy(Dp, mp=dict(type="prodmp", args=dict(cfg, dtype=torch.float64)),
                                        contextual=True)
    smp = pol.sample(False, mean, L, times, init_time, init_pos, init_vel, eps=rn(B, Dp))
    lp, _, _, reg = pol.log_prob(smp, mean, L, times, init_time, init_pos, init_vel, pred_pairs=pairs,
                                 return_parts=True)
    assert lp.shape == (B, pairs.shape[0])

    mp = pol.mp
    P = pairs.shape[0]
    tp = times[:, pairs]                                                  # [B, P, 2]
    mp.update_inputs(times=tp, params=mean[:, None].expand(B, P, Dp), params_L=None,
                     init_time=init_time[:, None].expand(B, P), init_pos=init_pos[:, None].expand(B, P, D),
                     init_vel=init_vel[:, None].expand(B, P, D))
    mu = mp.get_traj_pos(flat_shape=True)                                 # [B, P, 2D], DoF-major
    Hp = mp._terms()[4]                                                   # [B, P, 2, K1]
    covs, max_diag = {}, 0.0
    for b in range(B):
        Sigma = (L[b] @ L[b].T).numpy()
        for p in range(P):
            H = np.zeros((2 * D, Dp))
            for d in range(D):
                H[2 * d:2 * d + 2, d * K1:(d + 1) * K1] = Hp[b, p].numpy()
            covs[b, p] = H @ Sigma @ H.T
            max_diag = max(max_diag, float(np.diag(covs[b, p]).max()))
    assert abs(reg - 1e-4 * max_diag) <= 1e-12 * reg
    for b in range(B):
        for p in range(P):
            x = smp[b, pairs[p], :D].T.reshape(-1).numpy()                # d0@t0, d0@t1, d1@t0, ...
            want = multivariate_normal.logpdf(x, mean=mu[b, p].numpy(), cov=covs[b, p] + reg * np.eye(2 * D))
            assert abs(lp[b, p].item() - want) <= 1e-8 * max(1.0, abs(want)), (b, p)

"""Time the full-covariance projections at 64 < n <= 128 (the workspace kernels) on the GPU.

CUDA events around each call, the L2 flushed (a 256 MB write) before every timed call; median of the repetitions.
Cases: KL, Frobenius and W2 forward and backward (factor space), each for one shared matrix
(B = 1) and for B = 1024 per-episode matrices, at n = 70 and 128; and one BlackBoxAgent policy epoch (forward, losses,
backward) with a full-covariance policy of Dp = 112 parameters, B = 1024, for each projection.  Prints one JSON document.
"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from tce_rl_b200 import ops  # noqa: E402
from tce_rl_b200.rl import agent_factory, critic_factory, policy_factory, projection_factory  # noqa: E402


def draw(B, n, seed=0):
    g = torch.Generator().manual_seed(seed)
    Lo = torch.tril(torch.randn(B, n, n, generator=g) * 0.3 / n ** 0.5, -1) + torch.diag_embed(0.5 + torch.rand(B, n, generator=g))
    L = Lo + torch.tril(torch.randn(B, n, n, generator=g) * 0.02 / n ** 0.5, -1)
    return L.cuda(), Lo.cuda()


def timed(fn, reps, flush):
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return statistics.median(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    flush = torch.empty(64 * 1024 * 1024, device="cuda", dtype=torch.float32)
    res = {"gpu": torch.cuda.get_device_name(), "l2_flushed": True, "reps": args.reps, "ms": {}}
    for n in (70, 128):
        for B in (1, 1024):
            L, Lo = draw(B, n)
            state = ops.kl_state(B, n, L.device)
            P = ops.proj_kl_cov_fwd(L, Lo, 5e-4, state, False)[0]
            G = torch.tril(torch.randn_like(L))
            Pf, scf = ops.proj_frob_cov(L, Lo, 5e-4)[:2]
            cases = {
                "kl_fwd": lambda: ops.proj_kl_cov_fwd(L, Lo, 5e-4, state, False),
                "kl_bwd": lambda: ops.proj_kl_cov_bwd(G, L, P, state),
                "frob_fwd": lambda: ops.proj_frob_cov(L, Lo, 5e-4),
                "frob_bwd": lambda: ops.proj_frob_cov_bwd(G, L, Lo, Pf, scf, 5e-4),
                "w2_fwd": lambda: ops.proj_w2_cov(L, Lo, 2.5e-4, True),
                "w2_bwd": lambda: ops.proj_w2_cov_bwd(G, L, Lo, 2.5e-4, True),
            }
            for name, fn in cases.items():
                res["ms"][f"{name}_n{n}_B{B}"] = round(timed(fn, args.reps, flush), 4)
    for typ, cb in (("KLProjectionLayer", 5e-4), ("FrobeniusProjectionLayer", 5e-4), ("WassersteinProjectionLayer", 2.5e-4)):
        agent, data = bbrl_epoch_setup(112, typ, cb, B=1024)
        res["ms"][f"bbrl_epoch_{typ}_Dp112_B1024"] = round(timed(lambda: agent.policy_epoch(data, None, None), args.reps,
                                                                 flush), 4)
    print(json.dumps(res, indent=1))


def bbrl_epoch_setup(Dp, typ, cb, B, obs_dim=9):
    """BlackBoxAgent with a shared full-covariance policy and a processed synthetic dataset."""
    torch.manual_seed(0)
    policy = policy_factory("BlackBoxPolicy", dim_in=obs_dim, dim_out=Dp,
                            mean_net_args=dict(avg_neuron=32, num_hidden=2, shape=0.0),
                            variance_net_args=dict(std_only=False, contextual=False), init_method="orthogonal",
                            out_layer_gain=0.01, act_func_hidden="leaky_relu", act_func_last=None, dtype="float32",
                            device="cuda", min_std=1e-4)
    critic = critic_factory("ValueFunction", dim_in=obs_dim, dim_out=1, hidden=dict(avg_neuron=32, num_hidden=2, shape=0.0),
                            init_method="orthogonal", out_layer_gain=1, act_func_hidden="leaky_relu",
                            act_func_last=None, dtype="float32", device="cuda")
    layer = projection_factory(typ, device="cuda", dtype="float32", action_dim=Dp, proj_type=typ, mean_bound=0.05,
                               cov_bound=cb, trust_region_coeff=10.0, scale_prec=True, entropy_schedule="linear",
                               total_train_steps=100, target_entropy=0.0, temperature=0.7, entropy_eq=False,
                               entropy_first=False, do_regression=False)
    agent = agent_factory("BlackBoxAgent", policy=policy, critic=critic, sampler=None, projection=layer, dtype="float32",
                          device="cuda", lr_policy=3e-4, lr_critic=1e-3, wd_policy=5e-5, wd_critic=5e-5, epochs_policy=1,
                          epochs_critic=1, num_minibatchs=1, norm_advantages=True, set_variance=False)
    obs = torch.randn(B, obs_dim, device="cuda")
    with torch.no_grad():
        mean_old, L_old = policy.policy(obs)
        mean_old = (mean_old + 0.05 * torch.randn_like(mean_old)).contiguous()
        L_old = (1.03 * L_old[:1]).expand(B, -1, -1).contiguous()
        actions = policy.sample(False, mean_old, L_old, eps=torch.randn(B, Dp, device="cuda"))
        lp_old = policy.log_prob(actions, mean_old, L_old)
        for p in policy.parameters:
            p.add_(0.02 * torch.randn_like(p))
    data = agent.process_dataset(dict(segment_state=obs, segment_action=actions, segment_log_prob=lp_old,
                                      segment_params_mean=mean_old, segment_params_L=L_old,
                                      segment_reward=torch.randn(B, device="cuda"),
                                      segment_value=torch.randn(B, device="cuda")))
    layer.initial_entropy = policy.entropy([data["segment_params_mean"], data["segment_params_L"]]).mean()
    return agent, data


if __name__ == "__main__":
    main()

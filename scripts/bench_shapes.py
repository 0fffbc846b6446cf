"""Segment likelihood and policy epoch on ProDMP shapes without specialised kernels, next to the box shape.

    python scripts/bench_shapes.py [--out profiles/r04_any_shape.json]

Prints one JSON document (also written to --out).  Reported, CUDA-event times (mean over repeated calls after warm-up):
* ``likelihood``: ``ops_seglik.seglik`` in grad mode 2 (forward + backward of the fused surrogate in one call, as the
  epoch runs it) at B in {1024, 16384}, P = 25 chained pairs, one common time grid, for per-episode factors
  ([B, n, n]) and one shared covariance (fp64 Sigma, gradient w.r.t. Sigma: the input of the KL epoch).  The box shape
  (7, 9) runs the fused / uniform-grid kernels; every other shape runs the staged kernels.
* ``epoch``: one eager ``policy_epoch`` (B = 1024, KL projection, shared and contextual covariance, flat gradient and
  FlatAdam as ``update_policy`` sets them up), host wall time of 20 epochs ending in a device synchronise, divided by
  20; ``fast_epoch`` says whether the hand-scheduled shared-covariance epoch ran.
The card name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

from oracle import util as ou                                              # noqa: E402
from oracle.gen_golden import MP_CONFIGS, NUM_TIMES                        # noqa: E402
from tce_rl_b200 import ops, ops_seglik                                    # noqa: E402
from tce_rl_b200.rl import TemporalCorrelatedAgent, policy_factory, projection_factory   # noqa: E402
from tce_rl_b200.rl.agent import SegmentTimeSampler                        # noqa: E402

DEV = "cuda:0"
LIK_SHAPES = [(7, 9), (6, 6), (5, 8), (8, 8), (4, 16), (1, 16)]
EPOCH_SHAPES = [(7, 9), (6, 6), (8, 8)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def cfg_of(D, K1):
    return dict(MP_CONFIGS["box"], num_dof=D, num_basis=K1 - 1), NUM_TIMES["box"]


def event_time(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / iters


def likelihood(D, K1, B):
    cfg, T = cfg_of(D, K1)
    Dp, P = D * K1, 25
    tabs = ops.Tables(**cfg)
    g = torch.Generator().manual_seed(0)
    L = (torch.tril(0.05 * torch.randn(B, Dp, Dp, generator=g), -1) + torch.diag_embed(0.5 + torch.rand(B, Dp, generator=g))).to(DEV)
    mean = (0.5 * torch.randn(B, Dp, generator=g)).to(DEV)
    smp = (0.5 * torch.randn(B, T, 2 * D, generator=g)).to(DEV)
    init_time = torch.zeros(B, device=DEV)
    times = ou.get_times(init_time.double().cpu(), T, cfg["dt"]).float().to(DEV)
    init_pos, init_vel = torch.zeros(B, D, device=DEV), torch.zeros(B, D, device=DEV)
    pairs = ou.get_time_pairs(T, dict(num_select=P + 1, fixed_interval=True))[:P].to(DEV)
    lp_old, adv = torch.zeros(B, P, device=DEV), torch.randn(B, P, generator=g).to(DEV)
    sigma = (L[0].double() @ L[0].double().T).contiguous()
    scale = torch.ones(1, device=DEV, dtype=torch.float64)
    chained, uniform = ops_seglik._facts(pairs, init_time, times, True, None)
    out = {"compiled": tabs.compiled, "D": D, "K1": K1, "B": B, "P": P}
    iters = 50 if B <= 1024 else 10
    out["per_episode_us"] = event_time(lambda: ops_seglik.seglik(
        smp, mean, L, None, None, times, init_time, init_pos, init_vel, pairs, tabs.handle, 1e-4, 2, None, lp_old, adv,
        chained, False, True), iters)
    out["shared_sigma_us"] = event_time(lambda: ops_seglik.seglik(
        smp, mean, None, sigma, scale, times, init_time, init_pos, init_vel, pairs, tabs.handle, 1e-4, 2, None, lp_old,
        adv, chained, uniform, False, True), iters)
    return out


def epoch(D, K1, contextual, B=1024, epochs=20):
    cfg, T = cfg_of(D, K1)
    Dp, obs_dim = D * K1, 10
    torch.manual_seed(0)
    policy = policy_factory("TemporalCorrelatedPolicy", dim_in=obs_dim, dim_out=Dp,
                            mean_net_args=dict(avg_neuron=128, num_hidden=2, shape=0.0),
                            variance_net_args=dict(std_only=False, contextual=contextual, avg_neuron=128, num_hidden=2,
                                                   shape=0.0),
                            init_method="orthogonal", out_layer_gain=0.01, act_func_hidden="leaky_relu",
                            act_func_last=None, dtype="float32", device=DEV, min_std=1e-4,
                            mp=dict(type="prodmp", args=dict(cfg)))
    layer = projection_factory("KLProjectionLayer", proj_type="kl", mean_bound=0.05, cov_bound=5e-4,
                               trust_region_coeff=1.0, scale_prec=True, entropy_schedule="linear", action_dim=Dp,
                               total_train_steps=7500, target_entropy=0.0, temperature=0.7, entropy_eq=False,
                               entropy_first=False, do_regression=False, dtype="float32", device=DEV)
    sampler = SegmentTimeSampler(cfg["dt"], T, dict(num_select=25, fixed_interval=True), device=DEV)
    pairs = sampler.get_time_pairs()
    agent = TemporalCorrelatedAgent(policy, None, sampler, layer, dtype="float32", device=DEV, lr_policy=1e-4,
                                    lr_critic=1e-3, wd_policy=5e-5, wd_critic=5e-5, discount_factor=1.0,
                                    epochs_policy=1, epochs_critic=1, norm_advantages=True,
                                    segment_advantage="value_subtraction", set_variance=False)
    g = torch.Generator().manual_seed(1)
    obs = torch.randn(B, obs_dim + 2 * D, generator=g).to(DEV)
    init_time = torch.zeros(B, device=DEV)
    init_pos, init_vel = (0.1 * torch.randn(B, D, generator=g)).to(DEV), torch.zeros(B, D, device=DEV)
    times = sampler.get_times(init_time, T)
    with torch.no_grad():
        mean_old, L_old = policy.policy(obs[..., :-2 * D])
        smp = policy.sample(False, mean_old, L_old, times, init_time, init_pos, init_vel)
        lp_old = policy.log_prob(smp, mean_old, L_old, times, init_time, init_pos, init_vel, pred_pairs=pairs)
    dataset = dict(segment_state=obs, step_actions=smp, segment_log_prob_estimate=lp_old, segment_params_mean=mean_old,
                   segment_params_L=L_old if contextual else L_old[:1].expand(B, -1, -1),
                   segment_advantage=torch.randn(B, pairs.shape[0], generator=g).to(DEV), segment_init_time=init_time,
                   segment_init_pos=init_pos, segment_init_vel=init_vel)
    layer.initial_entropy = policy.entropy([mean_old, L_old]).mean()
    agent.ensure_flat_grads(agent.policy_net_params)          # as update_policy: one flat gradient + FlatAdam
    agent._use_flat_adam()
    for _ in range(3):
        agent.policy_epoch(dataset, times, pairs)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(epochs):
        agent.policy_epoch(dataset, times, pairs)
    torch.cuda.synchronize()
    return {"D": D, "K1": K1, "B": B, "contextual": contextual, "compiled": policy.mp.tables.compiled,
            "fast_epoch": agent._fast is not None, "ms_per_epoch": (time.perf_counter() - t0) * 1e3 / epochs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_shapes.py measures on the GPU; no CUDA device found")
    res = {"card": card(), "likelihood": [], "epoch": []}
    for D, K1 in LIK_SHAPES:
        for B in (1024, 16384):
            res["likelihood"].append(likelihood(D, K1, B))
    for D, K1 in EPOCH_SHAPES:
        for contextual in (False, True):
            res["epoch"].append(epoch(D, K1, contextual))
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()

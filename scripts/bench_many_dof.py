"""Time the per-segment factorisation above 8 DoF and whole policy epochs of 14-DoF policies on the GPU.

    python scripts/bench_many_dof.py [--out profiles/x.json]

CUDA events around each call with the L2 cache overwritten (a 256 MB write) before every timed call; median of the
repetitions.  Cases:
* the per-segment stage alone (``tce_seglik_chol``, forward and with an upstream gradient), B = 1024, P = 25 chained
  pairs, per-episode factors: (14, 4) and (16, 4) run ``seglik_chol_warp_kernel`` (one warp per segment), (7, 9) runs
  ``seglik_chol_kernel<14>`` (one thread per segment) for comparison;
* one TemporalCorrelatedAgent policy epoch (forward, losses, backward), B = 1024, KL projection: full covariance at
  (14, 4) and (7, 9), shared and contextual; std_only at (14, 9) and (7, 9), shared and contextual.
The GPU name and power limit are read in the same run.  Prints one JSON document."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from tce_rl_b200 import _lib, ops  # noqa: E402
from tce_rl_b200.rl import TemporalCorrelatedAgent, policy_factory, projection_factory  # noqa: E402
from tce_rl_b200.rl.agent import SegmentTimeSampler  # noqa: E402

DEV = "cuda"


def box_cfg(D, K1):
    return dict(num_dof=D, tau=2.0, alpha_phase=3, num_basis=K1 - 1, basis_bandwidth_factor=3, num_basis_outside=0,
                alpha=10, relative_goal=False, auto_scale_basis=True, weights_scale=0.3, goal_scale=0.3, dt=0.02)


def timed(fn, reps, flush):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush.fill_(1.0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    return dict(median_us=statistics.median(ts), min_us=min(ts), max_us=max(ts))


def chol_case(D, K1, B, P):
    """(forward call, gradient call) of the per-segment stage on a filled workspace."""
    cfg, T, Dp = box_cfg(D, K1), 100, D * K1
    tabs = ops.Tables(**cfg)
    g = torch.Generator(device=DEV).manual_seed(0)
    mean = 0.5 * torch.randn(B, Dp, device=DEV, generator=g)
    L = (torch.tril(0.05 * torch.randn(B, Dp, Dp, device=DEV, generator=g), -1)
         + torch.diag_embed(0.5 + torch.rand(B, Dp, device=DEV, generator=g))).contiguous()
    init_time = torch.zeros(B, device=DEV)
    times = (torch.arange(T, device=DEV, dtype=torch.float32) * cfg["dt"]).expand(B, T).contiguous()
    ip, iv = torch.rand(B, D, device=DEV, generator=g), 0.1 * torch.randn(B, D, device=DEV, generator=g)
    smp = torch.randn(B, T, 2 * D, device=DEV, generator=g)
    idx = torch.linspace(0, T - 1, P + 1).long()
    pairs = torch.stack([idx[:-1], idx[1:]], -1).to(DEV)
    logp, work, diag_max, info = ops.seglik_fwd(smp, mean, L, times, init_time, ip, iv, pairs, tabs.handle, 1e-4)
    adj = torch.empty_like(work)
    glp = torch.ones(B, P, device=DEV)
    p = lambda t: t.data_ptr()
    st = lambda: torch.cuda.current_stream().cuda_stream
    fwd = lambda: _lib.call("tce_seglik_chol", tabs.handle, p(work), None, p(diag_max), 1e-4, None, None, None, 0.0,
                            None, p(logp), p(info), B, P, st())
    bwd = lambda: _lib.call("tce_seglik_chol", tabs.handle, p(work), p(adj), p(diag_max), 1e-4, p(glp), None, None, 0.0,
                            None, None, None, B, P, st())
    return fwd, bwd, tabs


def epoch_case(D, K1, std_only, contextual, B):
    cfg, T, Dp, obs_dim = box_cfg(D, K1), 100, D * K1, 10
    torch.manual_seed(0)
    policy = policy_factory("TemporalCorrelatedPolicy", dim_in=obs_dim, dim_out=Dp,
                            mean_net_args=dict(avg_neuron=128, num_hidden=2, shape=0.0),
                            variance_net_args=dict(std_only=std_only, contextual=contextual, avg_neuron=128,
                                                   num_hidden=2, shape=0.0),
                            init_method="orthogonal", out_layer_gain=0.01, act_func_hidden="leaky_relu",
                            act_func_last=None, dtype="float32", device=DEV, min_std=1e-4,
                            mp=dict(type="prodmp", args=cfg))
    layer = projection_factory("KLProjectionLayer", proj_type="kl", mean_bound=0.05, cov_bound=5e-4,
                               trust_region_coeff=1.0, scale_prec=True, entropy_schedule="linear", action_dim=Dp,
                               total_train_steps=7500, target_entropy=0.0, temperature=0.7, entropy_eq=False,
                               entropy_first=False, do_regression=False, device=DEV, dtype="float32")
    sampler = SegmentTimeSampler(cfg["dt"], T, dict(num_select=25, fixed_interval=True), device=DEV)
    pairs = sampler.get_time_pairs()
    agent = TemporalCorrelatedAgent(policy, None, sampler, layer, dtype="float32", device=DEV, lr_policy=1e-4,
                                    lr_critic=1e-3, wd_policy=5e-5, wd_critic=5e-5, discount_factor=1.0,
                                    epochs_policy=1, epochs_critic=1, norm_advantages=True,
                                    segment_advantage="value_subtraction", set_variance=False)
    g = torch.Generator(device=DEV).manual_seed(4)
    obs = torch.randn(B, obs_dim + 2 * D, device=DEV, generator=g)
    init_time = torch.zeros(B, device=DEV)
    ip, iv = torch.rand(B, D, device=DEV, generator=g) * 2 - 1, 0.1 * torch.randn(B, D, device=DEV, generator=g)
    times = sampler.get_times(init_time, T)
    with torch.no_grad():
        mean_old, L_old = policy.policy(obs[..., :-2 * D])
        mean_old = mean_old + 0.05 * torch.randn(B, Dp, device=DEV, generator=g)
        L_old = L_old * torch.exp(0.05 * torch.randn(B if contextual else 1, Dp, device=DEV, generator=g)).diag_embed()
        if not contextual:
            L_old = L_old[:1].expand(B, -1, -1).contiguous()
        smp = policy.sample(False, mean_old, L_old, times, init_time, ip, iv,
                            eps=torch.randn(B, Dp, device=DEV, generator=g))
        lp_old = policy.log_prob(smp, mean_old, L_old, times, init_time, ip, iv, pred_pairs=pairs)
    dataset = dict(segment_state=obs, step_actions=smp, segment_log_prob_estimate=lp_old, segment_params_mean=mean_old,
                   segment_params_L=L_old, segment_advantage=torch.randn(B, pairs.shape[0], device=DEV, generator=g),
                   segment_init_time=init_time, segment_init_pos=ip, segment_init_vel=iv)
    layer.initial_entropy = policy.entropy([mean_old, L_old]).mean()
    agent.ensure_flat_grads(agent.policy_net_params)
    agent._use_flat_adam()
    return lambda: agent.policy_epoch(dataset, times, pairs), agent


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_many_dof.py needs a GPU")
    gpu = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
        gpu["power_limit"], gpu["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except (OSError, subprocess.CalledProcessError, IndexError, ValueError):
        gpu["power_limit"] = "not read"
    flush = torch.empty(256 * 2 ** 20 // 4, device=DEV)
    B, P = args.batch, 25
    stage = []
    for D, K1 in [(7, 9), (14, 4), (16, 4)]:
        fwd, bwd, _ = chol_case(D, K1, B, P)
        kernel = f"seglik_chol_kernel<{2 * D}>" if D <= 8 else f"seglik_chol_warp_kernel<{2 * D}>"
        stage.append(dict(num_dof=D, k1=K1, B=B, P=P, kernel=kernel, logp=timed(fwd, args.reps, flush),
                          with_gradient=timed(bwd, args.reps, flush)))
    epochs = []
    for D, K1, std_only, contextual in [(7, 9, False, False), (7, 9, False, True), (14, 4, False, False),
                                        (14, 4, False, True), (7, 9, True, False), (7, 9, True, True),
                                        (14, 9, True, False), (14, 9, True, True)]:
        step, agent = epoch_case(D, K1, std_only, contextual, B)
        row = dict(num_dof=D, k1=K1, dp=D * K1, std_only=std_only, contextual=contextual, B=B, P=P,
                   layer="KLProjectionLayer", **timed(step, args.reps, flush))
        row["hand_scheduled_epoch"] = agent._fast is not None
        epochs.append(row)
    doc = dict(gpu=gpu, l2_flush="256 MB write before every timed call", reps=args.reps, stage=stage, epochs=epochs)
    text = json.dumps(doc, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()

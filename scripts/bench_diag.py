"""Diagonal-covariance (std_only) policies on one GPU: ``update_policy`` with graph-captured epochs, and the diagonal
kernels next to the dense kernels on the same diagonal inputs.

    python scripts/bench_diag.py [--out profiles/r03_bench_diag.json]

Prints one JSON document (also written to --out).  Reported:
* ``update_policy_us_per_epoch``: box pushing, B = 1024, P = 24, KL projection, 10 epochs captured in a CUDA graph:
  host wall time of a whole ``update_policy`` call (ending in its device synchronise) divided by the epoch count
  (std_only contextual, std_only shared, full-covariance contextual).  This includes the per-update work outside the
  replayed epochs, so it is an upper bound of the epoch time, not the epoch time itself;
* ``kernels``: CUDA-event times (mean over repeated op calls, after warm-up; each call includes the zero fill of its
  dense [B, n, n] output or gradient) of the diagonal KL projection and the
  diagonal segment likelihood at B in {1024, 16384, 65536}, with the bytes the algorithm must move and that as a
  fraction of 7.7 TB/s HBM, and of the dense kernels (``proj_kl_cov``, ``seg_logprob_staged``) on the same inputs.
The card name and power limit are read in the same run.  The working sets of the diagonal kernels at B <= 16384 fit
in the 126 MB L2, so their HBM fraction there is an upper bound of the achieved DRAM rate, not a measurement of it.
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
from oracle.gen_golden import MP_CONFIGS, NUM_TIMES, synthetic_inputs      # noqa: E402
from tce_rl_b200 import ops                                                # noqa: E402
from tce_rl_b200.rl import TemporalCorrelatedAgent, policy_factory, projection_factory   # noqa: E402
from tce_rl_b200.rl.agent import SegmentTimeSampler                        # noqa: E402

DEV = "cuda:0"
HBM = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def cuda_time(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / reps                    # us per call


def build_agent(std_only, contextual, B=1024, epochs=10):
    cfg, T = MP_CONFIGS["box"], NUM_TIMES["box"]
    D, Dp, obs_dim = cfg["num_dof"], cfg["num_dof"] * (cfg["num_basis"] + 1), 12
    torch.manual_seed(0)
    policy = policy_factory("TemporalCorrelatedPolicy", dim_in=obs_dim, dim_out=Dp,
                            mean_net_args=dict(avg_neuron=128, num_hidden=2, shape=0.0),
                            variance_net_args=dict(std_only=std_only, contextual=contextual, avg_neuron=128,
                                                   num_hidden=2, shape=0.0),
                            init_method="orthogonal", out_layer_gain=0.01, act_func_hidden="leaky_relu",
                            act_func_last=None, dtype="float32", device=DEV, min_std=1e-4,
                            mp=dict(type="prodmp", args=dict(cfg)))
    proj = projection_factory("KLProjectionLayer", proj_type="kl", mean_bound=0.05, cov_bound=5e-4,
                              trust_region_coeff=1.0, scale_prec=True, entropy_schedule="linear", action_dim=Dp,
                              total_train_steps=7500, target_entropy=0.0, temperature=0.7, entropy_eq=False,
                              entropy_first=False, do_regression=False, dtype="float32", device=DEV)
    sampler = SegmentTimeSampler(cfg["dt"], T, dict(num_select=25, fixed_interval=True), device=DEV)
    agent = TemporalCorrelatedAgent(policy, None, sampler, proj, dtype="float32", device=DEV, lr_policy=3e-4,
                                    lr_critic=1e-3, wd_policy=5e-5, wd_critic=5e-5, discount_factor=1.0,
                                    epochs_policy=epochs, epochs_critic=1, num_minibatchs=1, norm_advantages=True,
                                    segment_advantage="value_subtraction", set_variance=False,
                                    use_cuda_graph=True)
    inp = synthetic_inputs("box", B, seed=3, dtype=torch.float32)
    c = lambda t: t.to(DEV)
    g = torch.Generator().manual_seed(5)
    obs = c(torch.randn(B, obs_dim + 2 * D, generator=g))
    pairs = sampler.get_time_pairs()
    with torch.no_grad():
        times = sampler.get_times(c(inp["init_time"]), T)
        mean_old, L_old = policy.policy(obs[..., :-2 * D])
        smp = policy.sample(False, mean_old, L_old, times, c(inp["init_time"]), c(inp["init_pos"]),
                            c(inp["init_vel"]), eps=c(inp["eps"]))
        lp_old = policy.log_prob(smp, mean_old, L_old, times, c(inp["init_time"]), c(inp["init_pos"]),
                                 c(inp["init_vel"]), pred_pairs=pairs)
        adv, _ = agent.get_advantage_return(c(inp["rewards"]), c(inp["values"]), c(inp["dones"]),
                                            c(inp["time_limit_dones"]))
        seg_adv = agent.get_segment_advantage(c(inp["rewards"]), c(inp["values"]), adv, pairs)
    dataset = dict(segment_state=obs, step_actions=smp, segment_log_prob_estimate=lp_old,
                   segment_params_mean=mean_old.clone(), segment_params_L=L_old.clone(), segment_advantage=seg_adv,
                   segment_init_time=c(inp["init_time"]), segment_init_pos=c(inp["init_pos"]),
                   segment_init_vel=c(inp["init_vel"]))
    return agent, dataset


def epoch_time(std_only, contextual, epochs=10, reps=5):
    agent, dataset = build_agent(std_only, contextual, epochs=epochs)
    agent.num_iterations = 1
    agent.update_policy(dataset)                             # capture + warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        agent.update_policy(dataset)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e6 / (reps * epochs)


def kernel_times(B, reps):
    cfg, T = MP_CONFIGS["box"], NUM_TIMES["box"]
    D, K1 = cfg["num_dof"], cfg["num_basis"] + 1
    n = D * K1
    g = torch.Generator().manual_seed(B)
    s_old = torch.exp(0.3 * torch.randn(B, n, generator=g))
    s = s_old * torch.exp(0.1 * torch.randn(B, n, generator=g))
    L, Lo = torch.diag_embed(s).to(DEV), torch.diag_embed(s_old).to(DEV)
    beta = torch.full((1,), -1e9, device=DEV, dtype=torch.float64)
    res = {}
    out, state, _ = ops.proj_kl_diag(L, Lo, 5e-4, beta, False)
    gout = torch.randn_like(out)
    vec_bytes = B * n * 4
    fwd_bytes = 3 * vec_bytes + B * 32                       # s, s_old in, s_proj out, state
    bwd_bytes = 4 * vec_bytes + B * 32                       # s, s_old, grad in, grad out, state
    t = cuda_time(lambda: ops.proj_kl_diag(L, Lo, 5e-4, beta, False), reps)
    res["proj_kl_diag_fwd"] = dict(us=t, bytes=fwd_bytes, hbm_fraction=fwd_bytes / (t * 1e-6) / HBM)
    t = cuda_time(lambda: ops.proj_kl_diag_bwd(gout, L, Lo, state), reps)
    res["proj_kl_diag_bwd"] = dict(us=t, bytes=bwd_bytes, hbm_fraction=bwd_bytes / (t * 1e-6) / HBM)
    dreps = max(3, reps // 20)
    st = ops.kl_state(B, n, DEV)
    res["dense_proj_kl_cov_fwd"] = dict(us=cuda_time(lambda: ops.proj_kl_cov_fwd(L, Lo, 5e-4, st, False), dreps, 1))
    pl, _ = ops.proj_kl_cov_fwd(L, Lo, 5e-4, st, False)
    res["dense_proj_kl_cov_bwd"] = dict(us=cuda_time(lambda: ops.proj_kl_cov_bwd(gout, L, pl, st), dreps, 1))
    del st, pl

    # likelihood (box pushing, P = 24 chained pairs, per-episode factors)
    inp = synthetic_inputs("box", B, seed=1, dtype=torch.float32)
    times = ou.get_times(inp["init_time"].double(), T, cfg["dt"]).float()
    torch.manual_seed(0)
    pairs = ou.get_time_pairs(T, dict(num_select=25, fixed_interval=True))
    P = pairs.shape[0]
    tabs = ops.Tables(**cfg)
    c = lambda x: x.to(DEV)
    mean = c(inp["mean"])
    smp = ops.prodmp_traj(mean, c(times), c(inp["init_time"]), c(inp["init_pos"]), c(inp["init_vel"]), tabs.handle, D)
    args = (c(times), c(inp["init_time"]), c(inp["init_pos"]), c(inp["init_vel"]), c(pairs), tabs)
    mg, Lg = mean.clone().requires_grad_(True), L.clone().requires_grad_(True)
    w = torch.randn(B, P, device=DEV)

    def diag_fb():
        lp = ops.seg_logprob_diag(smp, mg, Lg, *args)
        torch.autograd.backward(lp, w)

    def dense_fb():
        lp = ops.seg_logprob_staged(smp, mg, Lg, *args)
        torch.autograd.backward(lp, w)
    lik_bytes = (B * n * 4 * 2 + B * P * 2 * D * 4 + B * P * 4 + B * T * 4) * 2 + B * n * 4 * 2   # fwd + bwd reads/writes
    t = cuda_time(diag_fb, reps)
    res["seglik_diag_fwd_bwd"] = dict(us=t, bytes=lik_bytes, hbm_fraction=lik_bytes / (t * 1e-6) / HBM,
                                      note="includes the zero fill of the dense [B, n, n] gradient of L")
    t = cuda_time(lambda: ops.seg_logprob_diag(smp, mg.detach(), Lg.detach(), *args), reps)
    res["seglik_diag_fwd"] = dict(us=t)
    res["dense_seglik_staged_fwd_bwd"] = dict(us=cuda_time(dense_fb, dreps, 1))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=200)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_diag.py measures on the GPU; no CUDA device found")
    doc = {"card": card(), "workload": "box pushing (7 DoF x 9 = 63 parameters), P = 24 chained pairs"}
    doc["update_policy_us_per_epoch"] = {"std_only_contextual": epoch_time(True, True), "std_only_shared": epoch_time(True, False),
                       "full_cov_contextual": epoch_time(False, True)}
    doc["kernels"] = {str(B): kernel_times(B, a.reps) for B in (1024, 16384, 65536)}
    doc["card_after"] = card()
    text = json.dumps(doc, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

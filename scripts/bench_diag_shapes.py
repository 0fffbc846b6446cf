"""Time one std_only (diagonal covariance) policy epoch of TemporalCorrelatedAgent at B = 1024 per ProDMP shape, layer
and covariance layout, and compare source trees.

    python scripts/bench_diag_shapes.py --trees . /path/to/other/checkout --rounds 2 --out profiles/x.json

Each (tree, round) runs in a subprocess of its own (the trees alternate: A B A B), each of which times every config:
warm-up epochs, then ``--steps`` epochs each bracketed by CUDA events with the L2 cache overwritten (a 256 MB write)
before every one; the median is reported.  A config a tree cannot run (e.g. Dp > 64 before the diagonal path took
every shape) is reported with its error.  The GPU name and power limit are read in the same run.  Nothing is written
into the trees but the build a tree needs (built beforehand with ``python -m tce_rl_b200._build``)."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

CONFIGS = [(7, 9, "KLProjectionLayer", True), (7, 9, "KLProjectionLayer", False),
           (7, 9, "WassersteinProjectionLayer", True), (7, 9, "WassersteinProjectionLayer", False),
           (7, 9, "FrobeniusProjectionLayer", True), (7, 9, "FrobeniusProjectionLayer", False),
           (7, 10, "KLProjectionLayer", True), (7, 10, "KLProjectionLayer", False),
           (8, 16, "KLProjectionLayer", True), (8, 16, "KLProjectionLayer", False)]
LAYERS = {"KLProjectionLayer": (0.05, 5e-4), "FrobeniusProjectionLayer": (0.05, 5e-4),
          "WassersteinProjectionLayer": (0.005, 2.5e-4)}


def epoch_fn(D, K1, typ, contextual, B):
    """(run one epoch, its inputs) of a std_only TemporalCorrelatedAgent at the box task settings with this shape."""
    import torch
    from tce_rl_b200.rl import TemporalCorrelatedAgent, policy_factory, projection_factory
    from tce_rl_b200.rl.agent import SegmentTimeSampler
    dev = "cuda"
    cfg = dict(num_dof=D, tau=2.0, alpha_phase=3, num_basis=K1 - 1, basis_bandwidth_factor=3, num_basis_outside=0,
               alpha=10, relative_goal=False, auto_scale_basis=True, weights_scale=0.3, goal_scale=0.3, dt=0.02)
    T, Dp, obs_dim = 100, D * K1, 10
    mb, cb = LAYERS[typ]
    torch.manual_seed(0)
    policy = policy_factory("TemporalCorrelatedPolicy", dim_in=obs_dim, dim_out=Dp,
                            mean_net_args=dict(avg_neuron=128, num_hidden=2, shape=0.0),
                            variance_net_args=dict(std_only=True, contextual=contextual, avg_neuron=128, num_hidden=2,
                                                   shape=0.0),
                            init_method="orthogonal", out_layer_gain=0.01, act_func_hidden="leaky_relu",
                            act_func_last=None, dtype="float32", device=dev, min_std=1e-4,
                            mp=dict(type="prodmp", args=cfg))
    layer = projection_factory(typ, proj_type="kl", mean_bound=mb, cov_bound=cb, trust_region_coeff=1.0,
                               scale_prec=True, entropy_schedule="linear", action_dim=Dp, total_train_steps=7500,
                               target_entropy=0.0, temperature=0.7, entropy_eq=False, entropy_first=False,
                               do_regression=False, device=dev, dtype="float32")
    sampler = SegmentTimeSampler(cfg["dt"], T, dict(num_select=25, fixed_interval=True), device=dev)
    pairs = sampler.get_time_pairs()
    agent = TemporalCorrelatedAgent(policy, None, sampler, layer, dtype="float32", device=dev, lr_policy=1e-4,
                                    lr_critic=1e-3, wd_policy=5e-5, wd_critic=5e-5, discount_factor=1.0,
                                    epochs_policy=1, epochs_critic=1, norm_advantages=True,
                                    segment_advantage="value_subtraction", set_variance=False)
    g = torch.Generator(device=dev).manual_seed(4)
    obs = torch.randn(B, obs_dim + 2 * D, device=dev, generator=g)
    init_time = torch.zeros(B, device=dev)
    init_pos, init_vel = torch.rand(B, D, device=dev, generator=g) * 2 - 1, 0.1 * torch.randn(B, D, device=dev, generator=g)
    times = sampler.get_times(init_time, T)
    with torch.no_grad():
        mean_old, L_old = policy.policy(obs[..., :-2 * D])
        mean_old = mean_old + 0.05 * torch.randn(B, Dp, device=dev, generator=g)
        L_old = L_old * torch.exp(0.05 * torch.randn(B if contextual else 1, Dp, device=dev, generator=g)).diag_embed()
        if not contextual:
            L_old = L_old[:1].expand(B, -1, -1).contiguous()
        smp = policy.sample(False, mean_old, L_old, times, init_time, init_pos, init_vel,
                            eps=torch.randn(B, Dp, device=dev, generator=g))
        lp_old = policy.log_prob(smp, mean_old, L_old, times, init_time, init_pos, init_vel, pred_pairs=pairs)
    dataset = dict(segment_state=obs, step_actions=smp, segment_log_prob_estimate=lp_old, segment_params_mean=mean_old,
                   segment_params_L=L_old, segment_advantage=torch.randn(B, pairs.shape[0], device=dev, generator=g),
                   segment_init_time=init_time, segment_init_pos=init_pos, segment_init_vel=init_vel)
    layer.initial_entropy = policy.entropy([mean_old, L_old]).mean()
    agent.ensure_flat_grads(agent.policy_net_params)
    agent._use_flat_adam()
    return lambda: agent.policy_epoch(dataset, times, pairs)


def run_tree(args):
    """Child: time every config in the tree this process imports from (cwd)."""
    import torch
    sys.path.insert(0, os.getcwd())
    flush = torch.empty(256 * 2 ** 20 // 4, device="cuda")
    res = []
    for D, K1, typ, contextual in CONFIGS:
        row = dict(num_dof=D, k1=K1, dp=D * K1, layer=typ, contextual=contextual, B=args.batch)
        try:
            step = epoch_fn(D, K1, typ, contextual, args.batch)
            for _ in range(args.warmup):
                step()
            torch.cuda.synchronize()
            ts = []
            for _ in range(args.steps):
                flush.fill_(1.0)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                step()
                b.record()
                b.synchronize()
                ts.append(a.elapsed_time(b) * 1e3)
            row.update(median_us=statistics.median(ts), min_us=min(ts), max_us=max(ts))
        except Exception as e:                          # noqa: BLE001 -- reported, not hidden
            row["error"] = f"{type(e).__name__}: {str(e)[:160]}"
        res.append(row)
    print(json.dumps(res))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trees", nargs="+", default=["."])
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child", action="store_true")
    args = ap.parse_args()
    if args.child:
        return run_tree(args)
    import torch
    gpu = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
        gpu["power_limit"], gpu["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except (OSError, subprocess.CalledProcessError, IndexError, ValueError):
        gpu["power_limit"] = "not read"
    runs = []
    for r in range(args.rounds):
        for tree in args.trees:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--batch", str(args.batch),
                                  "--steps", str(args.steps), "--warmup", str(args.warmup)],
                                 cwd=tree, capture_output=True, text=True)
            if out.returncode:
                sys.stderr.write(out.stderr[-3000:])
                raise SystemExit(f"{tree}: exit {out.returncode}")
            runs.append(dict(tree=tree, round=r, configs=json.loads(out.stdout.strip().splitlines()[-1])))
    doc = dict(gpu=gpu, batch=args.batch, steps=args.steps, warmup=args.warmup, l2_flush="256 MB write before every epoch",
               runs=runs)
    text = json.dumps(doc, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    for run in runs:
        for c in run["configs"]:
            t = f'{c["median_us"]:9.1f} us' if "median_us" in c else c["error"]
            print(f'{run["tree"]:>12} r{run["round"]} ({c["num_dof"]},{c["k1"]}) {c["layer"][:5]} '
                  f'{"ctx" if c["contextual"] else "shared"}: {t}')


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- TCE policy-update throughput on B200 (BASELINE.json: "TCE policy-update episodes/sec").

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torch.distributed.run)
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR     (also writes the last step's outputs)
    python bench.py --impl reference --gpus N --steps K --warmup W

A *step* is ONE policy epoch of ``TemporalCorrelatedAgent.update_policy``
(mprl/rl/agent/temporal_correlated_agent.py:524-589) on the headline workload (BASELINE.json configs[1]):
box-pushing shape (7 DoF, 8 basis + goal, Dp = 63, T = 100), 1024 episodes x 24 segments per GPU
(``num_select: 25`` yields 24 pairs, SURVEY App. D.1), KL projection, non-contextual full covariance (as every
shipped config), fp32: policy MLP forward -> vector->Cholesky head -> KL trust-region projection (+ entropy
projection) -> segment-wise likelihood -> surrogate + trust-region loss -> backward -> (gradient all-reduce) ->
Adam step.  Nothing is skipped inside the timed region.  Weak scaling: every rank owns 1024 episodes.

One JSON line is printed by rank 0:
* ``value``       whole-job episodes/s with inputs resident in HBM (CUDA-graph replay, CUDA events, L2 flushed
                  between steps, max over ranks);
* ``e2e``         the same through the public agent API with the dataset coming from pinned host memory every
                  step and the loss vector read back;
* ``config.variants``  the other halves of SURVEY 8(d) config 2, same step, same timing: per-episode covariance
                  factors (contextual layout, nothing amortised by broadcasting) and the literal 25-segment pair set;
* ``also``        BASELINE configs 1, 3, 4, 5 (B = 152 GPU next to CPU fp32 / fp64; metaworld B = 4096 KL; table
                  tennis W2 1024 episodes / GPU; likelihood sweep with roofline fractions).  ``config.variants`` and
                  ``also`` are N = 1 lines; at N > 1 they run only with ``--multi-extras`` (config 3 is then strong
                  scaled, 4096 / N episodes per GPU);
* ``roofline``    the dominant kernel over ALL kernels of the step, timed inside this run with CUDA events on the
                  launching stream, next to the whole-step fraction of SURVEY 8(d);
* ``cpu_baseline`` the CPU oracle (a port of the reference path) on the box's host cores, same config.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import math
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# ---- MP shapes (mprl/config/{box_push_random_init,metaworld,table_tennis_4d}/tcp/entire/shared.yaml:53-73) --
MP_SHAPES = {
    "box": (dict(num_dof=7, tau=2.0, alpha_phase=3, num_basis=8, basis_bandwidth_factor=3, num_basis_outside=0,
                 alpha=10, relative_goal=False, auto_scale_basis=True, weights_scale=0.3, goal_scale=0.3, dt=0.02), 100),
    "metaworld": (dict(num_dof=4, tau=5.0, alpha_phase=3, num_basis=8, basis_bandwidth_factor=5, num_basis_outside=0,
                       alpha=10, relative_goal=True, auto_scale_basis=True, weights_scale=0.1, goal_scale=0.1,
                       dt=0.0125), 500),
    "table_tennis": (dict(num_dof=7, tau=0.75, delay=0.3, alpha_phase=3, num_basis=3, basis_bandwidth_factor=3,
                          num_basis_outside=0, alpha=25, relative_goal=True, auto_scale_basis=True, weights_scale=0.7,
                          goal_scale=0.1, dt=0.008), 350),
}
MP_BOX, T_STEPS = MP_SHAPES["box"]
OBS_DIM, B_PER_GPU = 20, 1024
PROJ = dict(proj_type="kl", mean_bound=0.05, cov_bound=5e-4, trust_region_coeff=1.0, scale_prec=True,
            entropy_schedule="linear", total_train_steps=7500, target_entropy=0.0, temperature=0.7,
            entropy_eq=False, entropy_first=False, do_regression=False)
AGENT = dict(lr_policy=1e-4, lr_critic=1e-3, wd_policy=5e-5, wd_critic=5e-5, discount_factor=1.0, epochs_policy=50,
             epochs_critic=50, num_minibatchs=1, norm_advantages=True, segment_advantage="value_subtraction",
             set_variance=False, gae_scaling=0.95)
POLICY = dict(mean_net_args=dict(avg_neuron=128, num_hidden=2, shape=0.0),
              variance_net_args=dict(std_only=False, contextual=False), init_method="orthogonal",
              out_layer_gain=0.01, act_func_hidden="leaky_relu", act_func_last=None, min_std=1e-4)
D, K1 = MP_BOX["num_dof"], MP_BOX["num_basis"] + 1
DP = D * K1


def shape_dims(shape):
    cfg, T = MP_SHAPES[shape]
    d, k1 = cfg["num_dof"], cfg["num_basis"] + 1
    return cfg, T, d, k1, d * k1


def synthetic_host_data(B, seed, shape="box"):
    """Synthetic rollout data of SURVEY 8(d) (CPU tensors, fp32)."""
    _, T, d, _, dp = shape_dims(shape)
    g = torch.Generator().manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=g)
    out = dict(obs=rn(B, OBS_DIM + 2 * d), mean_noise=0.05 * rn(B, dp), L_noise=torch.tril(0.01 * rn(dp, dp), -1),
               init_time=torch.zeros(B), init_pos=torch.rand(B, d, generator=g) * 2 - 1, init_vel=0.1 * rn(B, d),
               eps=rn(B, dp), rewards=rn(B, T), values=rn(B, T + 1))
    out["dones"] = torch.zeros(B, T, dtype=torch.bool)
    out["dones"][:, -1] = True
    out["time_limit_dones"] = torch.zeros(B, T, dtype=torch.bool)
    return out


def pair_set(T, mode):
    """'faithful': select_pred_pairs(num_select=25, fixed_interval) after torch.manual_seed(0) (24 pairs for T in
    {100, 350, 500}); 'literal25': the 25-segment index set {0, 4, ..., 96, 99} scaled to T (SURVEY 8(d) config 2)."""
    if mode == "faithful":
        return None
    step = T // 25
    idx = torch.cat([torch.arange(0, 25 * step, step), torch.tensor([T - 1])])
    return torch.stack([idx[:-1], idx[1:]], 1).to(torch.long)


# =============================================================================================================
# clocks
# =============================================================================================================
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm = sorted(int(r[1]) for r in self.rows if len(r) >= 9 and r[1].isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 9 for n, v in zip(names, r[5:9]) if v.lower() == "active"})
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(self.rows[0][2]), "reasons": reasons,
                "samples": len(sm)}


# =============================================================================================================
# GPU arm: workload construction
# =============================================================================================================
def build_gpu_workload(device, rank, world, shape="box", B=B_PER_GPU, pairs_mode="faithful", contextual=False,
                       proj_type="KLProjectionLayer", mean_bound=None, cov_bound=None, agent_kwargs=None):
    """-> (agent, dataset, times, pairs): the policy-update state of one rank after a synthetic rollout."""
    from tce_rl_b200.rl import TemporalCorrelatedAgent, policy_factory, projection_factory
    from tce_rl_b200.rl.agent import SegmentTimeSampler

    cfg, T, d, k1, dp = shape_dims(shape)
    torch.manual_seed(0)                                        # identical initial weights on every rank
    pol_kw = dict(POLICY)
    if contextual:
        pol_kw["variance_net_args"] = dict(std_only=False, contextual=True, avg_neuron=128, num_hidden=2, shape=0.0)
    policy = policy_factory("TemporalCorrelatedPolicy", dim_in=OBS_DIM, dim_out=dp, dtype="float32", device=device,
                            mp=dict(type="prodmp", args=dict(cfg)), **pol_kw)
    pk = dict(PROJ)
    if mean_bound is not None:
        pk["mean_bound"] = mean_bound
    if cov_bound is not None:
        pk["cov_bound"] = cov_bound
    projection = projection_factory(proj_type, device=device, dtype="float32", action_dim=dp, **pk)
    sampler = SegmentTimeSampler(cfg["dt"], T, dict(num_select=25, fixed_interval=True), device=device)
    torch.manual_seed(0)
    pairs = sampler.get_time_pairs()                            # seed 0 -> indices 0, 4, ..., 96 (P = 24)
    literal = pair_set(T, pairs_mode)
    if literal is not None:
        pairs = sampler.pred_pairs = literal.to(device)
    dist_on = world > 1
    agent = TemporalCorrelatedAgent(policy, None, sampler, projection, dtype="float32", device=device,
                                    process_group=True if dist_on else None, **dict(AGENT, **(agent_kwargs or {})))
    host = synthetic_host_data(B, seed=1234 + rank, shape=shape)
    c = lambda t: t.to(device)
    with torch.no_grad():
        times = sampler.get_times(c(host["init_time"]), T)
        mean0, L0 = policy.policy(c(host["obs"])[..., :-2 * d])
        mean_old = mean0 + c(host["mean_noise"])
        if contextual:
            L_old = (1.05 * L0 + c(host["L_noise"])).contiguous()
        else:
            L_old = (1.05 * L0[:1] + c(host["L_noise"])).expand(B, -1, -1).contiguous()
        smp = policy.sample(False, mean_old, L_old, times, c(host["init_time"]), c(host["init_pos"]),
                            c(host["init_vel"]), eps=c(host["eps"]))
        lp_old = policy.log_prob(smp, mean_old, L_old, times, c(host["init_time"]), c(host["init_pos"]),
                                 c(host["init_vel"]), pred_pairs=pairs)
        adv, ret = agent.get_advantage_return(c(host["rewards"]), c(host["values"]), c(host["dones"]),
                                              c(host["time_limit_dones"]))
        seg_adv = agent.get_segment_advantage(c(host["rewards"]), c(host["values"]), adv, pairs)
        # the new policy starts away from the old one so that both projection branches are active
        for p in policy.mean_net.parameters():
            p.add_(0.05 * torch.randn_like(p))
        if contextual:
            last = list(policy.variance_net.parameters())[-1]
            last.add_(0.02 * torch.randn_like(last))
        else:
            policy.variance_net.variable.add_(0.02 * torch.randn_like(policy.variance_net.variable))
    dataset = dict(segment_state=c(host["obs"]), step_actions=smp, segment_log_prob_estimate=lp_old,
                   segment_params_mean=mean_old, segment_params_L=L_old, segment_advantage=seg_adv,
                   segment_init_time=c(host["init_time"]), segment_init_pos=c(host["init_pos"]),
                   segment_init_vel=c(host["init_vel"]))
    # the dataset as the sampler hands it over (reference layout, [B, n, n] old factors) lives on the HOST; the
    # device copy is made by the agent's own loader (non-contextual policy: one old factor, broadcast)
    host_dataset = {k: v.cpu().pin_memory() for k, v in dataset.items()}
    dataset = agent.dataset_to_device(host_dataset)
    agent.host_dataset = host_dataset
    projection.initial_entropy = agent._global_mean(policy.entropy([mean_old, L_old]))
    if dist_on:                                                  # as update_policy does once per dataset
        from tce_rl_b200 import ops
        ops.sync_uniform(dataset["segment_init_time"], times)
    agent.num_iterations = 100
    agent.ensure_flat_grads(agent.policy_net_params)
    return agent, dataset, times, pairs


def graph_kernel_nodes(graph):
    """Number of kernel / memset / memcpy nodes of a captured CUDA graph (= GPU activities per replay)."""
    try:
        from cuda.bindings import runtime as rt
        raw = graph.raw_cuda_graph()
        err, _, num = rt.cudaGraphGetNodes(rt.cudaGraph_t(raw), 0)
        if int(err) != 0:
            return None
        err, nodes, num = rt.cudaGraphGetNodes(rt.cudaGraph_t(raw), num)
        kinds = {}
        for nd in nodes[:num]:
            err, typ = rt.cudaGraphNodeGetType(nd)
            name = getattr(typ, "name", str(typ)).replace("cudaGraphNodeType", "").lower()
            kinds[name] = kinds.get(name, 0) + 1
        return kinds
    except Exception:
        return None


def capture_epoch(agent, dataset, times, pairs, rank=0):
    """Two eager warm-up epochs, then one epoch captured in a CUDA graph.  -> (step_fn, metrics, abi_launches, mode,
    graph, node kinds)"""
    from tce_rl_b200 import _lib
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            agent.policy_epoch(dataset, times, pairs)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    try:
        l0 = _lib.LAUNCHES
        try:
            graph = torch.cuda.CUDAGraph(keep_graph=True)
        except TypeError:
            graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            metrics = agent.policy_epoch(dataset, times, pairs)
        launches = _lib.LAUNCHES - l0
        kinds = graph_kernel_nodes(graph)
        try:
            graph.instantiate()
        except Exception:
            pass
        return graph.replay, metrics, launches, "cuda_graph", graph, kinds
    except Exception as exc:                                     # pragma: no cover
        if rank == 0:
            print(f"[bench] CUDA-graph capture failed ({exc!r}); timing eager steps", file=sys.stderr)
        torch.cuda.synchronize()
        l0 = _lib.LAUNCHES
        box = [agent.policy_epoch(dataset, times, pairs)]
        launches = _lib.LAUNCHES - l0

        def step_fn():                                           # in place: the returned metrics track the last step
            box[0].copy_(agent.policy_epoch(dataset, times, pairs))
        return step_fn, box[0], launches, "eager", None, None


class Timer:
    """K timed steps after W warm-ups: CUDA events around each step on the launching stream, L2 flushed (768 MB
    write) before each, barrier + synchronize on both sides, max over ranks."""

    def __init__(self, device, world):
        self.device, self.world = device, world
        self.flush = torch.empty(192 * 1024 * 1024, device=device, dtype=torch.int32)

    def barrier(self):
        import torch.distributed as dist
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run(self, step_fn, K, W, sync_each=False):
        import torch.distributed as dist
        for _ in range(W):
            self.flush.zero_()
            step_fn()
        self.barrier()
        events = []
        for _ in range(K):
            self.flush.zero_()                                   # L2 flush, outside the timed events
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step_fn()
            b.record()
            if sync_each:
                b.synchronize()
            events.append((a, b))
        self.barrier()
        per = sorted(a.elapsed_time(b) for a, b in events)
        self.last_steps = {"min": round(per[0], 5), "median": round(per[len(per) // 2], 5), "max": round(per[-1], 5)}
        tt = torch.tensor([sum(per)], device=self.device, dtype=torch.float64)
        if self.world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return tt.item() / K                                     # ms per step


# =============================================================================================================
# roofline: every kernel of the step, timed live
# =============================================================================================================
def csrc_hash(files=None):
    """Hash of the kernel sources (all of csrc/, or the named files)."""
    h = hashlib.sha256()
    base = os.path.join(ROOT, "tce_rl_b200", "csrc")
    for f in sorted(files if files is not None else os.listdir(base)):
        h.update(open(os.path.join(base, f), "rb").read())
    return h.hexdigest()[:16]


# which sources an entry point's kernels live in (first matching prefix; the shared headers always count): an ncu
# capture of a kernel stays valid while THESE files are unchanged
_SRC_OF = (("tce_seglik_uniform", "tce_seglik_fused.cu"), ("tce_seglik_prepass", "tce_seglik_fused.cu"),
           ("tce_seglik_fused", "tce_seglik_fused.cu"), ("tce_seglik_dsigma_reduce", "tce_seglik_fused.cu"),
           ("tce_seglik", "tce_seglik.cu"), ("tce_proj", "tce_proj.cu"), ("tce_gauss_maha", "tce_proj.cu"),
           ("tce_gauss_kl", "tce_proj.cu"), ("tce_gauss_stats", "tce_proj.cu"), ("tce_tri_inverse", "tce_proj.cu"),
           ("tce_epoch", "tce_epoch.cu"), ("tce_prodmp", "tce_traj.cu"), ("tce_mvn", "tce_gauss.cu"),
           ("tce_chol", "tce_gauss.cu"), ("tce_policy_head", "tce_gauss.cu"), ("tce_adam", "tce_adam.cu"),
           ("tce_grad_sumsq", "tce_adam.cu"), ("tce_p2p", "tce_p2p.cu"), ("tce_gae", "tce_adv.cu"),
           ("tce_segment", "tce_adv.cu"), ("tce_normalize", "tce_adv.cu"))


def src_hash_of(abi_name):
    base = os.path.join(ROOT, "tce_rl_b200", "csrc")
    headers = [f for f in os.listdir(base) if f.endswith(".cuh")]
    for prefix, f in _SRC_OF:
        if abi_name.startswith(prefix):
            return csrc_hash(headers + [f])
    return csrc_hash()


def measure_fma_peaks(timer):
    """FP32 / FP64 FMA throughput of this GPU (TFLOP/s), measured with the library's own micro-benchmark (the
    driver's MEASURED_PEAKS.json has HBM and bf16 tensor entries only)."""
    import ctypes
    from tce_rl_b200 import _lib
    scratch = torch.empty(16, device=timer.device, dtype=torch.float64)
    st = torch.cuda.current_stream().cuda_stream
    pipes = {}
    for name, fp64 in (("fp32", 0), ("fp64", 1)):
        fl = ctypes.c_double()
        best = 0.0
        for _ in range(4):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            _lib.call("tce_bench_fma", fp64, 4096, scratch.data_ptr(), ctypes.byref(fl), st)
            b.record()
            torch.cuda.synchronize()
            best = max(best, fl.value / (a.elapsed_time(b) * 1e-3) / 1e12)
        pipes[name] = best
    return pipes


def survey_figures(shape, P):
    """SURVEY 8(d) algorithmic bytes / FLOPs per EPISODE (fp32 = 4 B, L counted as its lower triangle)."""
    _, T, d, k1, dp = shape_dims(shape)
    n, tri = 2 * d, dp * (dp + 1) // 2
    fwd_bytes = 4 * (tri + dp + (P + 1) * d + (1 + 2 * d) + P)
    bwd_bytes = fwd_bytes + 4 * (P + dp + tri)
    mac_seg = dp * (dp + 1) + k1 * (4 * sum(i * (i + 1) // 2 for i in range(d)) + 3 * d * (d + 1) // 2) \
        + n ** 3 // 6 + n * n // 2 + n * k1
    fwd_flops = P * 2 * mac_seg
    epoch_bytes = 4 * (2 * (dp + tri) + dp + tri + (P + 1) * d + (1 + 2 * d) + 2 * P)
    epoch_flops = 3 * fwd_flops + 4 * dp ** 3 // 3
    return dict(fwd_bytes=fwd_bytes, bwd_bytes=bwd_bytes, fwd_flops=fwd_flops, epoch_bytes=epoch_bytes,
                epoch_flops=epoch_flops, proj_bytes=6 * dp * (dp + 1), proj_flops=2 * dp ** 3 // 3,
                traj_bytes=4 * (dp + (1 + 2 * d) + T + 2 * d * T), traj_flops=2 * T * d * (2 * k1 + 4))


def kernel_table(agent, dataset, times, pairs, reps=5):
    """Per-kernel durations of the step: every C-ABI launch of ``reps`` eager epochs is bracketed by CUDA events on
    ITS launching stream (``_lib.TIMING``).  The epoch is queued behind a ~3 ms device-side sleep so that the host
    runs ahead and the events measure the kernels, not launch gaps.  -> {abi name: (mean us per epoch, calls/epoch)}"""
    from tce_rl_b200 import _lib
    agent.policy_epoch(dataset, times, pairs)
    torch.cuda.synchronize()
    acc = {}
    for _ in range(reps):
        _lib.TIMING = []
        torch.cuda._sleep(6_000_000)
        agent.policy_epoch(dataset, times, pairs)
        torch.cuda.synchronize()
        rec, _lib.TIMING = _lib.TIMING, None
        for name, a, b in rec:
            us, cnt = acc.get(name, (0.0, 0))
            acc[name] = (us + a.elapsed_time(b) * 1e3, cnt + 1)
    return {k: (us / reps, cnt / reps) for k, (us, cnt) in acc.items()}


def roofline_numbers(agent, dataset, times, pairs, timer, peaks, ms_per_step, shape="box", contextual=False):
    B, P = dataset["segment_params_mean"].shape[0], int(pairs.shape[0])
    _, T, d, k1, dp = shape_dims(shape)
    fig = survey_figures(shape, P)
    table = kernel_table(agent, dataset, times, pairs)
    pipes = measure_fma_peaks(timer)
    n_cov = B if contextual else 1
    lik = [k for k in table if k.startswith("tce_seglik")]
    lik_us = sum(table[k][0] for k in lik)
    # algorithmic (bytes, FLOPs) per launch; the likelihood launches are one unit of work (SURVEY: fwd + bwd, bwd = 2x
    # fwd FLOPs) and share one figure
    alg = {}
    for k in table:
        if k.startswith("tce_proj_kl") and "bwd" not in k and not k.endswith("_chol"):
            alg[k] = (n_cov * fig["proj_bytes"], n_cov * fig["proj_flops"], "fp64")
        elif k.startswith("tce_proj_kl") and "bwd" in k:
            alg[k] = (n_cov * fig["proj_bytes"], n_cov * fig["proj_flops"], "fp64")
        elif k.startswith("tce_proj_kl") and k.endswith("_chol"):
            alg[k] = (n_cov * 4 * dp * (dp + 1), n_cov * dp ** 3 // 3, "fp64")
    dom = max(table, key=lambda k: table[k][0])
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    kern = {k: {"us": round(us, 2), "calls": round(c, 2)} for k, (us, c) in sorted(table.items(), key=lambda kv: -kv[1][0])}
    if dom in lik:
        a_bytes, a_flops, pipe = B * fig["bwd_bytes"], 3 * B * fig["fwd_flops"], "fp32+fp64"
        dom_us, dom_label = lik_us, "segment likelihood (" + " + ".join(sorted(lik)) + ")"
    else:
        a_bytes, a_flops, pipe = alg.get(dom, (0, 0, "fp64"))
        dom_us, dom_label = table[dom][0], dom
    achieved = a_bytes / (dom_us * 1e-6) / 1e9 if dom_us > 0 else 0.0
    # blended FMA peak of the whole step: likelihood FLOPs split between the pipes as the kernels run them (the two
    # O(Dp^3)-class products fp32, the per-segment quadratic forms / factorisations fp64), projection FLOPs fp64
    step_flops = B * 3 * fig["fwd_flops"] + n_cov * 4 * dp ** 3 // 3
    step_time_at_peak = (B * 3 * fig["fwd_flops"] * 0.5 / (pipes["fp32"] * 1e12)
                         + (B * 3 * fig["fwd_flops"] * 0.5 + n_cov * 4 * dp ** 3 // 3) / (pipes["fp64"] * 1e12))
    traffic = None
    traffic_src = "no ncu capture for this kernel"
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")))
        ent = tj.get("kernels", {}).get(dom)
        if ent is not None:                              # captures are keyed by launch grid (1 matrix / B matrices / CTAs)
            ent = ent.get(f"grid={n_cov}") or (next(iter(ent.values())) if len(ent) == 1 else None)
        if ent is not None and (ent.get("src_hash") == src_hash_of(dom) if "src_hash" in ent
                                else tj.get("csrc_hash") == csrc_hash()):
            traffic, traffic_src = ent["dram_bytes"], tj.get("source", "profiles/r02_ncu_traffic.json")
        elif ent is not None:
            traffic_src = "profiles/r02_ncu_traffic.json is stale (kernel sources changed since the capture)"
    except Exception:
        pass
    roof = {"bound": "hbm", "kernel": dom_label, "achieved": round(achieved, 3), "peak": hbm_peak, "unit": "GB/s",
            "frac": round(achieved / hbm_peak, 6), "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst)" if "hbm_gbs" in peaks
            else "fallback 6650 GB/s (B200_PROFILING.md)",
            "algorithmic_bytes_per_launch": a_bytes, "algorithmic_flops_per_launch": a_flops,
            "kernel_us": round(dom_us, 2), "pipe": pipe,
            "selection": "longest of ALL C-ABI launches of one eager epoch (CUDA events on each launching stream)",
            "note": ("the dominant kernel is a single-CTA latency chain (one 63x63 covariance for the whole batch): its "
                     "roofline fraction is ~0 by construction; see whole_step and config.variants.contextual for the "
                     "batched projection") if n_cov == 1 and dom.startswith("tce_proj_kl") else "",
            "compute": {"achieved_tflops": round(a_flops / (dom_us * 1e-6) / 1e12, 4) if dom_us > 0 else 0.0,
                        "measured_fp32_fma_tflops": round(pipes["fp32"], 2),
                        "measured_fp64_fma_tflops": round(pipes["fp64"], 2),
                        "frac_of_pipe": round(a_flops / (dom_us * 1e-6) / 1e12 /
                                              (pipes["fp64"] if pipe == "fp64" else pipes["fp32"]), 5) if dom_us > 0 else 0.0},
            "whole_step": {"algorithmic_flops": step_flops, "algorithmic_bytes": B * fig["epoch_bytes"],
                           "ms_per_step": round(ms_per_step, 5),
                           "frac_of_fp32_fma": round(step_flops / (ms_per_step * 1e-3) / 1e12 / pipes["fp32"], 5),
                           "frac_of_blended_fma": round(step_time_at_peak / (ms_per_step * 1e-3), 5),
                           "frac_of_hbm": round(B * fig["epoch_bytes"] / (ms_per_step * 1e-3) / 1e9 / hbm_peak, 5),
                           "formula": "SURVEY 8(d): FLOPs = B*3*fwd_flops + n_cov*4*Dp^3/3; blended peak = half of the "
                                      "likelihood FLOPs on the fp32 pipe, the rest on the fp64 pipe"},
            "likelihood": {"us_all_launches": round(lik_us, 2),
                           "alg_tflops": round(3 * B * fig["fwd_flops"] / (lik_us * 1e-6) / 1e12, 3) if lik_us else None,
                           "hbm_frac": round(B * fig["bwd_bytes"] / (lik_us * 1e-6) / 1e9 / hbm_peak, 5) if lik_us else None},
            "kernels": kern}
    return roof


# =============================================================================================================
# `also`: BASELINE configs 1, 3, 4, 5
# =============================================================================================================
def epoch_point(timer, device, rank, world, K, W, **kw):
    agent, ds, times, pairs = build_gpu_workload(device, rank, world, **kw)
    step_fn, metrics, launches, mode, graph, kinds = capture_epoch(agent, ds, times, pairs, rank)
    ms = timer.run(step_fn, K, W)
    ok = bool(torch.isfinite(metrics).all().item())
    B = ds["segment_params_mean"].shape[0]
    res = {"ms_per_step": round(ms, 5), "episodes_per_s": round(world * B / (ms * 1e-3), 1), "episodes_per_gpu": B,
           "segments": int(pairs.shape[0]), "finite": ok, "abi_launches_per_step": launches, "replay": mode}
    if kinds:
        res["graph_nodes_per_step"] = kinds
    return res, (agent, ds, times, pairs, graph)


def likelihood_sweep(timer, device, peaks, pipes, points=((1024, 25), (16384, 25), (65536, 25))):
    """BASELINE config 5: the segment likelihood alone (per-episode covariance factors, box-pushing shape), forward and
    forward + backward, against SURVEY 8(d)'s per-episode figures."""
    from tce_rl_b200 import ops
    cfg, T, d, k1, dp = shape_dims("box")
    tabs = ops.Tables(**cfg)
    out = []
    for B, P in points:
        g = torch.Generator().manual_seed(7)
        base = min(B, 2048)
        rn = lambda *s: torch.randn(*s, generator=g)
        mean = (0.5 * rn(base, dp)).repeat(B // base, 1).to(device)
        L = (torch.tril(0.05 * rn(base, dp, dp), -1) + torch.diag_embed(torch.nn.functional.softplus(rn(base, dp)) + 1e-4)
             ).repeat(B // base, 1, 1).to(device)
        init_time = torch.zeros(B, device=device)
        init_pos = (torch.rand(base, d, generator=g) * 2 - 1).repeat(B // base, 1).to(device)
        init_vel = (0.1 * rn(base, d)).repeat(B // base, 1).to(device)
        eps = rn(base, dp).repeat(B // base, 1).to(device)
        times = (init_time[:, None] + cfg["dt"] * torch.arange(1, T + 1, device=device)[None, :]).contiguous()
        idx = torch.arange(0, T, T // (P + 1))[:P + 1]
        pairs = torch.stack([idx[:-1], idx[1:]], 1).to(device)
        theta = ops.mvn_rsample(mean, L, eps, 0, 0)
        traj = ops.prodmp_traj(theta, times, init_time, init_pos, init_vel, tabs.handle, d)
        glp = torch.full((B, P), 1.0 / (B * P), device=device)

        def fwd():
            return ops.seglik(traj, mean, L, None, None, times, init_time, init_pos, init_vel, pairs, tabs.handle, 1e-4,
                              0, None, None, None, True, False, False)

        def fwd_bwd():
            return ops.seglik(traj, mean, L, None, None, times, init_time, init_pos, init_vel, pairs, tabs.handle, 1e-4,
                              1, glp, None, None, True, False, True)
        info = fwd()[1]
        assert int(info.abs().max()) == 0
        reps = 10 if B <= 16384 else 4
        tf, tfb = timer.run(fwd, reps, 3) * 1e-3, timer.run(fwd_bwd, reps, 3) * 1e-3
        fig = survey_figures("box", P)
        out.append({"B": B, "P": P, "fwd_us": round(tf * 1e6, 1), "fwd_bwd_us": round(tfb * 1e6, 1),
                    "seg_logprobs_per_s_fwd": round(B * P / tf), "seg_logprobs_per_s_fwd_bwd": round(B * P / tfb),
                    "hbm_frac_fwd": round(B * fig["fwd_bytes"] / tf / 1e9 / float(peaks.get("hbm_gbs", 6650.0)), 4),
                    "hbm_frac_fwd_bwd": round(B * fig["bwd_bytes"] / tfb / 1e9 / float(peaks.get("hbm_gbs", 6650.0)), 4),
                    "alg_tflops_fwd": round(B * fig["fwd_flops"] / tf / 1e12, 2),
                    "alg_tflops_fwd_bwd": round(3 * B * fig["fwd_flops"] / tfb / 1e12, 2),
                    "frac_fp32_fma_fwd": round(B * fig["fwd_flops"] / tf / 1e12 / pipes["fp32"], 4),
                    "frac_fp32_fma_fwd_bwd": round(3 * B * fig["fwd_flops"] / tfb / 1e12 / pipes["fp32"], 4)})
        del mean, L, traj, theta, eps, glp
        torch.cuda.empty_cache()
    return out


# =============================================================================================================
# main GPU arm
# =============================================================================================================
def _mark(msg):
    if os.environ.get("TCE_BENCH_DEBUG"):
        print(f"[bench r{os.environ.get('RANK', '0')}] {msg}", file=sys.stderr, flush=True)


def dump_outputs(out_dir, metrics, policy):
    """What the last timed step handed its caller, as ``out_dir/<name>.npy``: the metrics vector (fp64, the agent's
    loss keys then its KL keys) and every policy parameter after that step's Adam update (fp32, in
    ``policy.parameters`` order).  The workload is seeded, so the same arguments give the same inputs on every run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"metrics": metrics.double()}
    arrays.update((f"policy_param_{i:02d}", p.detach().float()) for i, p in enumerate(policy.parameters))
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def run_ours(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE {world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (GPU arm) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass

    _mark("init done")
    agent, dataset, times, pairs = build_gpu_workload(device, rank, world)
    _mark("workload built")
    K, W = args.steps, max(args.warmup, 3)
    timer = Timer(device, world)
    flush = timer.flush
    step_fn, metrics, launches_per_step, mode, graph, kinds = capture_epoch(agent, dataset, times, pairs, rank)
    _mark("graph captured")

    # ---- device-resident timing ---------------------------------------------------------------------------------
    with ClockSampler(local) as clocks:
        t_wall0 = time.perf_counter()
        ms_per_step = timer.run(step_fn, K, W)
        t_wall = time.perf_counter() - t_wall0
    step_spread = dict(timer.last_steps)
    value = world * B_PER_GPU / (ms_per_step * 1e-3)
    _mark("timed region done")
    final = metrics.cpu()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, final, agent.policy)
    if not torch.isfinite(final).all():
        raise SystemExit("non-finite loss in the timed region")

    # ---- end to end: host-resident dataset in, loss vector out, every step -------------------------------------------
    pinned = agent.host_dataset                                  # reference layout, pinned host memory
    out_host = torch.empty_like(final).pin_memory()
    # bytes that cross PCIe per step: every tensor of the host dataset, except that the B equal old factors of
    # the non-contextual policy travel once (TemporalCorrelatedAgent.dataset_to_device)
    h2d = sum((v[:1] if k == "segment_params_L" else v).numel() * v.element_size() for k, v in pinned.items())
    h2d_reference_layout = sum(v.numel() * v.element_size() for v in pinned.values())
    d2h = out_host.numel() * out_host.element_size()

    # Double-buffered input pipeline (what a training loop around the agent does): two device copies of the
    # dataset, each with its own captured epoch; while step k runs on buffer k % 2 a copy stream uploads the
    # dataset of step k + 1 into the other buffer.  Every step's inputs still cross PCIe inside the timed region
    # (K uploads in K timed steps) and every step's loss vector is read back and waited for (one step later: the host
    # queues step k + 1 before it blocks on the loss of step k, as a training loop that logs its losses does).
    sets = [(dataset, step_fn, metrics)]
    if graph is not None:
        try:
            dataset_b = agent.dataset_to_device(pinned)
            torch.cuda.synchronize()
            # same procedure as for the first buffer: the eager warm-up epochs also settle the per-dataset facts the
            # epoch caches (common time grid: decided once per dataset with one device read, which a capture cannot
            # do -- captured cold, this graph fell back to the general-grid likelihood, +50 us per replay)
            step_b, metrics_b, _, mode_b, graph_b, _ = capture_epoch(agent, dataset_b, times, pairs, rank)
            if mode_b != "cuda_graph":
                raise RuntimeError("capture failed")
            sets.append((dataset_b, step_b, metrics_b))
        except Exception as exc:                                 # pragma: no cover
            if rank == 0:
                print(f"[bench] second epoch graph failed ({exc!r}); e2e without input prefetch", file=sys.stderr)
    main_stream, copy_stream = torch.cuda.current_stream(), torch.cuda.Stream()
    uploaded = [torch.cuda.Event() for _ in sets]
    consumed = [torch.cuda.Event() for _ in sets]

    def upload(i, after=None):
        copy_stream.wait_event(consumed[i])                      # the last replay on buffer i has read its inputs
        if after is not None:
            copy_stream.wait_event(after)                        # not before the current step started: the copy must
        with torch.cuda.stream(copy_stream):                     # fall inside a timed step, not inside the L2 flush
            agent.dataset_to_device(pinned, out=sets[i][0])      # static device addresses: the graph replays on them
            uploaded[i].record(copy_stream)

    e2e_count = [0]
    out_hosts = [out_host, torch.empty_like(out_host).pin_memory()]
    read_back = [torch.cuda.Event(), torch.cuda.Event()]
    for ev in read_back:
        ev.record(main_stream)

    def e2e_step():
        i = e2e_count[0] % len(sets)
        e2e_count[0] += 1
        started = torch.cuda.Event()
        started.record(main_stream)
        if len(sets) == 1:
            upload(0)                                            # no second buffer: upload, then compute
        main_stream.wait_event(uploaded[i])
        sets[i][1]()
        consumed[i].record(main_stream)
        j = e2e_count[0] % 2
        out_hosts[j].copy_(sets[i][2], non_blocking=True)       # the step's loss vector -> pinned host memory
        read_back[j].record(main_stream)
        read_back[1 - j].synchronize()                           # the PREVIOUS step's loss is on the host (owned by the
                                                                 # caller) before the step after this one is queued:
                                                                 # one step of look-ahead, no launch gap on the GPU
        if len(sets) > 1:                                        # next step's inputs, overlapped with this step; queued
            upload(e2e_count[0] % len(sets), after=started)      # AFTER this step's replay so that the host's ~20
                                                                 # copy calls do not delay the start of the epoch

    if len(sets) > 1:
        upload(0)
    for _ in range(4):
        e2e_step()
    timer.barrier()
    _mark("e2e warm-up done")
    e2e_ms = timer.run(e2e_step, K, 0)                           # (each step waits for the previous step's loss itself)
    e2e_value = world * B_PER_GPU / (e2e_ms * 1e-3)
    if os.environ.get("TCE_E2E_DEBUG"):                          # where the e2e step's extra time goes (stderr only)
        def variant(no_upload=False, no_readback=False, one_graph=False, which=0):
            def f():
                i = which if one_graph else e2e_count[0] % len(sets)
                e2e_count[0] += 1
                started = torch.cuda.Event(); started.record(main_stream)
                if not no_upload:
                    main_stream.wait_event(uploaded[i])
                sets[i][1]()
                consumed[i].record(main_stream)
                if not no_readback:
                    out_hosts[0].copy_(sets[i][2], non_blocking=True)
                if not no_upload:
                    upload(0 if one_graph else e2e_count[0] % len(sets), after=started)
            return f
        for tag, kw in (("full", {}), ("no_upload", dict(no_upload=True)), ("no_readback", dict(no_readback=True)),
                        ("no_upload_no_readback", dict(no_upload=True, no_readback=True)),
                        ("one_graph_no_upload_no_readback", dict(no_upload=True, no_readback=True, one_graph=True)),
                        ("graph_b_only", dict(no_upload=True, no_readback=True, one_graph=True, which=len(sets) - 1))):
            torch.cuda.synchronize()
            print(f"[e2e debug] {tag}: {timer.run(variant(**kw), K, 3):.5f} ms", file=sys.stderr)
    # the upload alone (same loader, same pinned dataset, nothing else running): what PCIe + ~20 copy calls cost per step
    torch.cuda.synchronize()
    ua, ub = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(copy_stream):
        ua.record(copy_stream)
        for _ in range(10):
            agent.dataset_to_device(pinned, out=sets[0][0])
        ub.record(copy_stream)
    torch.cuda.synchronize()
    upload_ms = ua.elapsed_time(ub) / 10
    _mark("e2e done")

    # ---- the other halves of config 2, and BASELINE configs 1 / 3 / 4 / 5 ------------------------------------------
    variants, also = {}, {}
    Kv, Wv = max(5, min(K, 20)), 3
    if not args.no_variants:
        variants["contextual_P24"], ctx = epoch_point(timer, device, rank, world, Kv, Wv, contextual=True)
        variants["contextual_P24"]["note"] = ("per-episode covariance factors [B, 63, 63] (variance NET, contextual "
                                              "layout): 1024 KL projections per step, nothing broadcast")
        if not args.no_roofline:                 # every rank: the timed eager epochs contain the collectives
            try:
                r = roofline_numbers(ctx[0], ctx[1], ctx[2], ctx[3], timer, peaks, variants["contextual_P24"]["ms_per_step"],
                                     contextual=True)
                variants["contextual_P24"]["roofline"] = {k: r[k] for k in ("kernel", "achieved", "frac", "kernel_us",
                                                                            "compute", "whole_step", "likelihood")}
                variants["contextual_P24"]["roofline"]["kernels"] = dict(list(r["kernels"].items())[:8])
            except Exception as exc:                             # pragma: no cover
                variants["contextual_P24"]["roofline"] = {"error": repr(exc)}
        del ctx
        torch.cuda.empty_cache()
        variants["shared_P25"], _ = epoch_point(timer, device, rank, world, Kv, Wv, pairs_mode="literal25")
        variants["shared_P25"]["note"] = "literal 25 segments: index set {0, 4, ..., 96, 99}"
        variants["contextual_P25"], _ = epoch_point(timer, device, rank, world, Kv, Wv, contextual=True,
                                                    pairs_mode="literal25")
        del _
        torch.cuda.empty_cache()
        _mark("variants done")
    if not args.no_also:
        also["config3_metaworld_kl"], _ = epoch_point(timer, device, rank, world, Kv, Wv, shape="metaworld",
                                                      B=4096 // world, mean_bound=0.005, cov_bound=5e-4)
        also["config3_metaworld_kl"].update(global_episodes=4096, scaling="strong")
        also["config4_table_tennis_w2"], _ = epoch_point(timer, device, rank, world, Kv, Wv, shape="table_tennis",
                                                         B=1024, proj_type="WassersteinProjectionLayer",
                                                         mean_bound=0.005, cov_bound=2.5e-4)
        also["config4_table_tennis_w2"].update(global_episodes=1024 * world, scaling="weak",
                                               note="BASELINE names no batch for config 4: 1024 episodes per GPU")
        if world == 1:
            also["config1_boxpush_B152"], _ = epoch_point(timer, device, rank, world, Kv, Wv, B=152)
        del _
        torch.cuda.empty_cache()
        _mark("also epochs done")

    roof = None
    if not args.no_roofline:                         # every rank (collectives inside the eager epochs); rank 0 reports
        roof = roofline_numbers(agent, dataset, times, pairs, timer, peaks, ms_per_step)
        if world == 1 and not args.no_also:
            pipes = {"fp32": roof["compute"]["measured_fp32_fma_tflops"], "fp64": roof["compute"]["measured_fp64_fma_tflops"]}
            also["config5_likelihood_sweep"] = likelihood_sweep(timer, device, peaks, pipes)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(budget_s=12.0)
        if not args.no_also:
            also["config1_boxpush_B152"]["cpu_fp32"] = cpu_baseline(budget_s=4.0, B=152, dtype=torch.float32)
            also["config1_boxpush_B152"]["cpu_fp64"] = cpu_baseline(budget_s=4.0, B=152, dtype=torch.float64)
    _mark("roofline / cpu baseline done")
    if world > 1:
        dist.barrier()
    _mark("final barrier passed")
    if rank == 0:
        P = int(pairs.shape[0])
        total_nodes = sum(kinds.values()) if kinds else None
        line = {
            "metric": "TCE policy-update episodes/sec", "value": round(value, 1), "unit": "episodes/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": round(ms_per_step, 5), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"boxpush_tce_policy_epoch_B{B_PER_GPU}_P{P}", "episodes_per_gpu": B_PER_GPU,
                       "global_episodes": world * B_PER_GPU, "segments": P, "num_dof": D, "num_basis_g": K1,
                       "dim_params": DP, "num_times": T_STEPS, "projection": "KLProjectionLayer",
                       "contextual_cov": False,
                       "L_layout": "non-contextual covariance (every shipped config): the new, old and projected factors "
                                   "are each ONE [63,63] matrix broadcast over the batch with stride 0 (the reference "
                                   "repeats them B times); the per-episode layout is config.variants.contextual_P24",
                       "kl_warm_start": True,
                       "grad_exchange": ("none (1 GPU)" if world == 1 else
                                         "fused NVLink peer-memory all-reduce + gradient norm (tce_p2p_allreduce_sumsq)"
                                         if getattr(agent, "_p2p", None) is not None else "NCCL all_reduce(AVG)"),
                       "kl_warm_start_note": "every timed step projects against the same old factor, so the eigenbasis "
                                             "warm start always hits: a real update is 1 cold + 49 warm epochs per "
                                             "dataset (cold epoch: +0.1-0.2 ms once per 50)",
                       "step": "policy MLP + head + KL/entropy projection + segment likelihood + losses + backward "
                               "+ grad all-reduce + Adam", "replay": mode, "l2": "flushed between timed steps",
                       "segment_logprobs_per_s_fwd_bwd": round(value * P, 1),
                       "variants": variants},
            "clocks": clocks.summary(),
            "e2e": {"value": round(e2e_value, 1), "unit": "episodes/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": round(e2e_ms, 5),
                    "host_dataset_bytes": h2d_reference_layout, "upload_alone_ms": round(upload_ms, 5),
                    "host_tensors_per_step": sum(1 for v in pinned.values() if torch.is_tensor(v)),
                    "input_pipeline": "double_buffered" if len(sets) > 1 else "serial",
                    "note": "host dataset in the reference layout; the loader sends the shared old factor once; "
                            "the upload of step k+1 overlaps step k (two device buffers, two captured epochs); every "
                            "step's loss vector is copied to pinned host memory and waited for one step later"},
            "gpu_launches": (total_nodes if total_nodes is not None else launches_per_step) * K,
            "gpu_launches_per_step": total_nodes if total_nodes is not None else launches_per_step,
            "gpu_launches_detail": {"own_kernels_per_step": launches_per_step, "graph_nodes_per_step": kinds,
                                    "note": "own = launches through the C ABI (libtce_b200.so); graph nodes = every GPU "
                                            "activity of one replayed epoch incl. cuBLAS GEMMs of the MLP and ATen glue"},
            "roofline": roof,
            "also": also,
            "wall_s_timed_region": round(t_wall, 3), "step_ms_rank0": step_spread,
            "loss": {"surrogate": round(final[0].item(), 6), "trust_region": round(final[2].item(), 6)},
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    if world > 1:
        # NCCL kernels captured in the CUDA graph keep the communicator busy at teardown (observed: hang in
        # destroy_process_group); all results are out, so leave without the collective teardown.
        sys.stdout.flush()
        sys.stderr.flush()
        torch.cuda.synchronize()
        os._exit(0)


# =============================================================================================================
# CPU arm: the oracle (a port of the reference's path: mprl.rl + restated mp_pytorch / trust_region_projections)
# =============================================================================================================
def make_oracle_workload(B, dtype=torch.float32, seed=1234):
    from oracle import agent as oa, policy as opol, projection as oproj, util as ou
    torch.manual_seed(0)
    dims = [OBS_DIM, 128, 128, DP]
    layers = []
    for i, (a, b) in enumerate(zip(dims[:-1], dims[1:])):
        lin = torch.nn.Linear(a, b, dtype=dtype)
        torch.nn.init.orthogonal_(lin.weight, gain=0.01 if i == 2 else math.sqrt(2))
        torch.nn.init.zeros_(lin.bias)
        layers += [lin] + ([torch.nn.LeakyReLU()] if i < 2 else [])
    mean_net = torch.nn.Sequential(*layers)
    policy = opol.TemporalCorrelatedPolicy(DP, mp=dict(type="prodmp", args=dict(MP_BOX, dtype=dtype)), mean_net=mean_net,
                                           contextual=False, min_std=1e-4, dtype=dtype)
    policy.cov_vector = policy.cov_vector.clone().requires_grad_(True)
    layer = oproj.projection_factory("KLProjectionLayer", dtype=dtype, action_dim=DP, **PROJ)
    host = synthetic_host_data(B, seed)
    c = lambda t: t.to(dtype) if t.is_floating_point() else t
    torch.manual_seed(0)
    pairs = ou.get_time_pairs(T_STEPS, dict(num_select=25, fixed_interval=True))
    with torch.no_grad():
        times = ou.get_times(c(host["init_time"]), T_STEPS, MP_BOX["dt"])
        mean0, L0 = policy.policy(c(host["obs"])[..., :-2 * D])
        mean_old = mean0 + c(host["mean_noise"])
        L_old = (1.05 * L0[:1] + c(host["L_noise"])).expand(B, -1, -1).contiguous()
        smp = policy.sample(False, mean_old, L_old, times, c(host["init_time"]), c(host["init_pos"]), c(host["init_vel"]),
                            eps=c(host["eps"]))
        lp_old = policy.log_prob(smp, mean_old, L_old, times, c(host["init_time"]), c(host["init_pos"]),
                                 c(host["init_vel"]), pred_pairs=pairs)
        adv, _ = oa.get_advantage_return(c(host["rewards"]), c(host["values"]), host["dones"], host["time_limit_dones"],
                                         1.0, 0.95)
        seg = oa.get_segment_advantage(c(host["rewards"]), c(host["values"]), adv, pairs, 1.0, "value_subtraction", True)
        for p in mean_net.parameters():
            p.add_(0.05 * torch.randn_like(p))
    data = dict(segment_state=c(host["obs"]), step_actions=smp, segment_log_prob_estimate=lp_old,
                segment_params_mean=mean_old, segment_params_L=L_old, segment_advantage=seg,
                segment_init_time=c(host["init_time"]), segment_init_pos=c(host["init_pos"]),
                segment_init_vel=c(host["init_vel"]))
    layer.initial_entropy = policy.entropy([mean_old, L_old]).mean()
    params = list(mean_net.parameters()) + [policy.cov_vector]
    opt = torch.optim.Adam(params, lr=1e-4, weight_decay=5e-5)

    def epoch():
        loss, _ = oa.policy_epoch(policy, layer, data, times, pairs, 100, set_variance=False)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        return float(loss.detach())
    return epoch


def cpu_baseline(budget_s=12.0, B=B_PER_GPU, dtype=torch.float32):
    """The oracle's policy epoch on ALL host cores, same config as the GPU arm (full batch), bounded by ``budget_s``."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    epoch = make_oracle_workload(B, dtype=dtype)
    epoch()                                                      # warm-up
    t0, n = time.perf_counter(), 0
    while True:
        epoch()
        n += 1
        dt = time.perf_counter() - t0
        if dt >= budget_s or n >= 50:
            break
    name = "fp32" if dtype == torch.float32 else "fp64"
    return {"value": round(B * n / dt, 2), "unit": "episodes/s", "cores": torch.get_num_threads(), "kind": "port",
            "same_config": B == B_PER_GPU and dtype == torch.float32, "ms_per_step": round(dt / n * 1e3, 2),
            "sample": f"{n} policy epochs of {B} episodes x 24 segments ({name}, torch CPU oracle = reference mprl.rl "
                      f"path + restated mp_pytorch / trust-region layers), {dt:.1f} s",
            "note": "the restated KL projection solves the dual exactly (cheaper than the reference's ITPAL/NLopt "
                    "C++ path) and the 12 logging KLs are not evaluated: a lower bound on the reference's CPU cost"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    B = B_PER_GPU                                                # the full headline batch: same config as our arm
    epoch = make_oracle_workload(B)
    for _ in range(max(1, min(args.warmup, 3))):
        epoch()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        epoch()
    dt = time.perf_counter() - t0
    value = B * args.steps / dt
    print(json.dumps({
        "impl": "reference", "metric": "TCE policy-update episodes/sec", "value": round(value, 2),
        "unit": "episodes/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(dt / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"boxpush_tce_policy_epoch_B{B_PER_GPU}_P24", "episodes_per_gpu": B_PER_GPU,
                   "same_config": True,
                   "sample": f"each step = one policy epoch over all {B} episodes x 24 segments of the workload "
                             "(CPU, one process; N > 1 does not change the CPU arm)"},
        "cpu_baseline": {"value": round(value, 2), "unit": "episodes/s", "cores": torch.get_num_threads(),
                         "kind": "port", "sample": f"{args.steps} epochs x {B} episodes x 24 segments"},
        "e2e": {"value": round(value, 2), "unit": "episodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--no-also", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--multi-extras", action="store_true",
                    help="N > 1: also run config.variants / also on every rank (by default they are N = 1 lines: at "
                         "N > 1 the run is the headline step, e2e and the roofline, i.e. what the scaling curve needs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (metrics vector and updated policy "
                         "parameters) to DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl ours)")
    if int(os.environ.get("WORLD_SIZE", "1")) > 1 and not args.multi_extras:
        args.no_variants = args.no_also = True
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

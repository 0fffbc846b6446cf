"""Time the ProDMP position covariance and standard deviation ops (tce::traj_pos_cov / traj_pos_std, forward and
backward w.r.t. L) on the box task's shape (7, 9) and on (16, 8) (128 parameters), T = 100, B = 64 and 1024.

    python scripts/bench_traj_cov.py [--reps 20] [--out profiles/r09_bench_traj_cov.json]

CUDA events around each call with the L2 cache overwritten (a 256 MB write) before every timed call; median over the
repetitions.  The covariance forward writes B (D T)^2 fp32 values and its backward reads as many, so each is reported
as those bytes over the call time, as a fraction of the HBM bandwidth measured in the same run (a 4 GB device-to-device
copy: read + write bytes over its time).  The GPU name and power limit are read in the same run.  Prints one JSON
document."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from tce_rl_b200 import ops  # noqa: E402

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


def hbm_bandwidth(reps, flush):
    n = 4 * 2 ** 30 // 4
    src, dst = torch.ones(n, device=DEV), torch.empty(n, device=DEV)
    t = timed(lambda: dst.copy_(src), reps, flush)
    del src, dst
    return 2 * 4 * n / (t["median_us"] * 1e-6)


def case(D, K1, B, T, reps, flush, hbm):
    tabs = ops.Tables(**box_cfg(D, K1))
    Dp, N = D * K1, D * T
    g = torch.Generator(device=DEV).manual_seed(0)
    L = (torch.tril(0.05 * torch.randn(B, Dp, Dp, device=DEV, generator=g), -1)
         + torch.diag_embed(0.5 + torch.rand(B, Dp, device=DEV, generator=g))).contiguous()
    init_time = 0.3 * torch.rand(B, device=DEV, generator=g)
    times = (init_time[:, None] + torch.arange(T, device=DEV, dtype=torch.float32) * 0.02).contiguous()
    h = tabs.handle
    cov = ops.traj_pos_cov(L, times, init_time, h, D, 1e-4)
    gcov = torch.randn(cov.shape, device=DEV, generator=g)
    std = ops.traj_pos_std(L, times, init_time, h, D, 1e-4)
    gstd = torch.randn(std.shape, device=DEV, generator=g)
    out = dict(num_dof=D, k1=K1, B=B, T=T, cov_bytes=4 * B * N * N)
    out["cov_fwd"] = timed(lambda: ops.traj_pos_cov(L, times, init_time, h, D, 1e-4), reps, flush)
    out["cov_bwd"] = timed(lambda: ops.traj_pos_cov_bwd(gcov, L, times, init_time, h), reps, flush)
    out["std_fwd"] = timed(lambda: ops.traj_pos_std(L, times, init_time, h, D, 1e-4), reps, flush)
    out["std_bwd"] = timed(lambda: ops.traj_pos_std_bwd(gstd, std, L, times, init_time, h), reps, flush)
    L1 = L[:1].contiguous()
    out["cov_bwd_shared_L"] = timed(lambda: ops.traj_pos_cov_bwd(gcov, L1, times, init_time, h), reps, flush)
    for k in ("cov_fwd", "cov_bwd", "cov_bwd_shared_L"):
        bw = out["cov_bytes"] / (out[k]["median_us"] * 1e-6)
        out[k]["cov_bytes_per_s"] = bw
        out[k]["fraction_of_measured_hbm"] = bw / hbm
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_traj_cov.py needs a GPU")
    gpu = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, check=True).stdout.splitlines()[0]
        gpu["power_limit"], gpu["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except Exception:
        gpu["power_limit"] = "not read"
    flush = torch.empty(256 * 2 ** 20 // 4, device=DEV)
    hbm = hbm_bandwidth(args.reps, flush)
    cases = [case(D, K1, B, 100, args.reps, flush, hbm) for D, K1 in [(7, 9), (16, 8)] for B in (64, 1024)]
    doc = dict(gpu=gpu, l2_flush="256 MB write before every timed call", reps=args.reps,
               measured_hbm_bytes_per_s=hbm, cases=cases)
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

"""Run the three segment-likelihood kernels a few times on the headline shape (for ncu captures)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from tce_rl_b200 import ops, _lib
from oracle.gen_golden import MP_CONFIGS, NUM_TIMES, synthetic_inputs
from oracle import util as ou

dev = "cuda:0"
name, B = (sys.argv[1] if len(sys.argv) > 1 else "box"), int(sys.argv[2]) if len(sys.argv) > 2 else 1024
cfg, T = MP_CONFIGS[name], NUM_TIMES[name]
inp = synthetic_inputs(name, B, dtype=torch.float32)
times = ou.get_times(inp["init_time"].double(), T, cfg["dt"]).float()
torch.manual_seed(0)
pairs = ou.get_time_pairs(T, dict(num_select=25, fixed_interval=True))
g = {k: v.to(dev) for k, v in inp.items()}
times_g, pairs_g = times.to(dev), pairs.to(dev)
tabs = ops.Tables(**cfg)
theta = ops.mvn_rsample(g["mean"], g["L"], g["eps"], 0, 0)
traj = ops.prodmp_traj(theta, times_g, g["init_time"], g["init_pos"], g["init_vel"], tabs.handle, cfg["num_dof"])
P, Dp = pairs.shape[0], g["mean"].shape[1]
work = ops._work(tabs.handle, B, P, dev); adj = torch.empty_like(work)
dmax = torch.zeros(1, device=dev, dtype=torch.float64)
logp = torch.empty(B, P, device=dev); info = torch.empty(B, P, device=dev, dtype=torch.int32)
glp = torch.ones(B, P, device=dev); gm = torch.empty_like(g["mean"]); gL = torch.empty_like(g["L"])
st = torch.cuda.current_stream().cuda_stream
p = lambda t: t.data_ptr()
for _ in range(3):
    _lib.call("tce_seglik_gram", tabs.handle, p(traj), p(g["mean"]), p(g["L"]), Dp * Dp, p(times_g), p(g["init_time"]), p(g["init_pos"]), p(g["init_vel"]), p(pairs_g), p(work), p(dmax), B, T, P, st)
    _lib.call("tce_seglik_chol", tabs.handle, p(work), p(adj), p(dmax), 1e-4, p(glp), None, None, 0.0, None, p(logp), p(info), B, P, st)
    _lib.call("tce_seglik_bwd", tabs.handle, p(adj), p(g["L"]), Dp * Dp, p(times_g), p(g["init_time"]), p(pairs_g), None, p(gm), p(gL), B, T, P, st)
torch.cuda.synchronize()
print("ok", float(logp.sum()))

import ctypes
buf = (ctypes.c_longlong * 32)()
_lib.call("tce_debug_seglik_phase_cycles", buf)
s = list(buf)
for nm, i in (("gram load L", 0), ("gram basis", 1), ("gram Sigma", 2), ("gram C blocks", 3), ("gram residual", 4), ("gram max", 5)):
    print(f"{nm:16s} {s[i + 1] - s[i]:8d} cycles")
for nm, i in (("bwd load+basis", 16), ("bwd grad_mean", 17), ("bwd M (fp64)", 18), ("bwd M.L", 19), ("bwd store", 20)):
    print(f"{nm:16s} {s[i + 1] - s[i]:8d} cycles")

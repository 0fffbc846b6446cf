"""PyTorch custom ops (``torch.ops.tce.*``) over the C ABI of libtce_b200.so.

PyTorch is plumbing here: it owns device memory and streams; every op body is one or more calls
into the hand-written sm_100a kernels.  There is no CPU or eager fallback: tensors must be CUDA
fp32 (indices int64, flags bool/uint8) and the library must be built.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import MpCfg, TceError

Tensor = torch.Tensor


# --------------------------------------------------------------------------------------------------
# helpers
# --------------------------------------------------------------------------------------------------
def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _chk(t: Tensor, dtype=torch.float32, name="tensor") -> Tensor:
    if not t.is_cuda:
        raise TceError(f"{name} must be a CUDA tensor (tce_rl_b200 has no CPU path)")
    if t.dtype != dtype:
        raise TceError(f"{name} must be {dtype}, got {t.dtype}")
    return t.contiguous()


def _batched_matrix(L: Tensor, name="L", batch: Optional[int] = None) -> Tuple[Tensor, int]:
    """Return (storage tensor, batch stride in elements); keeps a stride-0 batch expand un-materialised.
    ``batch``: a single matrix [1, n, n] is broadcast over that many episodes (batch stride 0)."""
    if not L.is_cuda or L.dtype != torch.float32:
        raise TceError(f"{name} must be a CUDA float32 tensor")
    n = L.shape[-1]
    if L.dim() == 3 and L.stride(0) == 0 and L.stride(1) == n and L.stride(2) == 1:
        return L, 0
    if L.dim() == 3 and L.shape[0] == 1 and batch is not None and batch > 1:
        return L.contiguous(), 0
    L = L.contiguous()
    return L, n * n


class Tables:
    """Owner of a ``tce_tables_t`` handle (pre-computed ProDMP basis tables on the current device)."""

    def __init__(self, *, num_dof, tau, dt, num_basis, alpha, alpha_phase, basis_bandwidth_factor,
                 delay=0.0, num_basis_outside=0, auto_scale_basis=True, weights_scale=1.0, goal_scale=1.0,
                 relative_goal=False, relative_goal_scaled=False, pre_compute_length_factor=5, **_ignored):
        self.cfg = MpCfg(num_dof=int(num_dof), num_basis=int(num_basis), num_basis_outside=int(num_basis_outside),
                         pre_compute_length_factor=int(pre_compute_length_factor),
                         auto_scale_basis=int(bool(auto_scale_basis)), relative_goal=int(bool(relative_goal)),
                         relative_goal_scaled=int(bool(relative_goal_scaled)), reserved=0, tau=float(tau),
                         delay=float(delay), dt=float(dt), alpha=float(alpha), alpha_phase=float(alpha_phase),
                         basis_bandwidth_factor=float(basis_bandwidth_factor), weights_scale=float(weights_scale),
                         goal_scale=float(goal_scale))
        self.num_dof, self.num_basis_g = int(num_dof), int(num_basis) + 1
        self.dim_params = self.num_dof * self.num_basis_g
        self.tau, self.delay, self.dt = float(tau), float(delay), float(dt)
        self.factor = int(pre_compute_length_factor)
        handle = C.c_void_p()
        self.device = torch.cuda.current_device()
        _lib.call("tce_prodmp_tables_create", C.byref(self.cfg), _stream(), C.byref(handle))
        self.handle = handle.value
        self.num_pc = _lib.load().tce_prodmp_tables_num_pc(self.handle)
        # one of the five shapes with fused / uniform-grid likelihood kernels (else: staged kernels, see ops_seglik.compiled)
        self.compiled = _lib.load().tce_seglik_compiled(self.handle) == 1

    def export(self):
        """fp64 tables as CPU tensors (for tests / inspection)."""
        n, k1 = self.num_pc, self.num_basis_g
        out = {k: torch.empty(n, dtype=torch.float64) for k in ("y1", "y2", "dy1", "dy2")}
        out["pos_basis"] = torch.empty(n, k1, dtype=torch.float64)
        out["vel_basis"] = torch.empty(n, k1, dtype=torch.float64)
        out["scale"] = torch.empty(k1, dtype=torch.float64)
        _lib.call("tce_prodmp_tables_export", self.handle,
                  *[out[k].data_ptr() for k in ("y1", "y2", "dy1", "dy2", "pos_basis", "vel_basis", "scale")])
        return out

    def max_time(self) -> float:
        return self.delay + self.factor * self.tau

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                _lib.load().tce_prodmp_tables_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


# --------------------------------------------------------------------------------------------------
UNIFORM_TRAJ = True      # common-time-grid fast path of the trajectory synthesis (False: always the general kernel)
_NUM_SMS = {}


def _num_sms(device) -> int:
    idx = torch.device(device).index
    idx = torch.cuda.current_device() if idx is None else idx
    if idx not in _NUM_SMS:
        _NUM_SMS[idx] = torch.cuda.get_device_properties(idx).multi_processor_count
    return _NUM_SMS[idx]


def traj_uniform_layout(B: int, T: int, num_dof: int, k1: int, sms: int) -> Tuple[int, int]:
    """(episodes per CTA, dynamic shared memory in bytes) of ``tce_prodmp_traj_fwd_uniform``: the same formula as
    ``launch_traj_uniform`` (csrc/tce_traj.cu).  A CTA holds all T basis rows and one output tile."""
    epc = min(256 // num_dof, 16)
    while epc > 4 and -(-B // epc) < 2 * sms:
        epc //= 2
    estride = (20 * 2 * num_dof + 3) // 4 * 4
    while estride % 32 != 8:
        estride += 4
    return epc, 4 * (T * ((2 * (k1 + 2) + 3) // 4 * 4) + epc * estride)


TRAJ_UNIFORM_SMEM = 200 * 1024    # the uniform kernel's limit; longer horizons run the general kernel


# (1) trajectory synthesis
# --------------------------------------------------------------------------------------------------
@torch.library.custom_op("tce::prodmp_traj", mutates_args=())
def prodmp_traj(params: Tensor, times: Tensor, init_time: Tensor, init_pos: Tensor, init_vel: Tensor,
                tables: int, num_dof: int) -> Tensor:
    params, times = _chk(params, name="params"), _chk(times, name="times")
    init_time, init_pos, init_vel = _chk(init_time), _chk(init_pos), _chk(init_vel)
    B, T = times.shape
    traj = torch.empty(B, T, 2 * num_dof, device=params.device, dtype=torch.float32)
    # one time grid for the whole batch (a cached device read per tensor; never decided under graph capture): the
    # basis rows are evaluated once and the batch becomes a small matrix product per episode.  The rows live in shared
    # memory, so a horizon whose rows do not fit runs the general kernel.
    k1 = params.shape[-1] // num_dof
    if UNIFORM_TRAJ and B >= 64 and \
            traj_uniform_layout(B, T, num_dof, k1, _num_sms(params.device))[1] <= TRAJ_UNIFORM_SMEM and \
            times_uniform(init_time, times):
        rows = torch.empty(T * ((2 * (k1 + 2) + 3) // 4 * 4), device=params.device, dtype=torch.float32)
        _lib.call("tce_prodmp_traj_fwd_uniform", tables, _p(params), _p(times), _p(init_time), _p(init_pos), _p(init_vel),
                  _p(rows), _p(traj), B, T, _stream())
        return traj
    _lib.call("tce_prodmp_traj_fwd", tables, _p(params), _p(times), _p(init_time), _p(init_pos), _p(init_vel),
              _p(traj), B, T, _stream())
    return traj


@prodmp_traj.register_fake
def _(params, times, init_time, init_pos, init_vel, tables, num_dof):
    return params.new_empty(times.shape[0], times.shape[1], 2 * num_dof)


@torch.library.custom_op("tce::prodmp_traj_bwd", mutates_args=())
def prodmp_traj_bwd(grad_traj: Tensor, times: Tensor, init_time: Tensor, tables: int, num_dof: int,
                    dim_params: int) -> Tuple[Tensor, Tensor, Tensor]:
    grad_traj, times, init_time = _chk(grad_traj), _chk(times), _chk(init_time)
    B, T = times.shape
    gp = torch.empty(B, dim_params, device=times.device, dtype=torch.float32)
    gy = torch.empty(B, num_dof, device=times.device, dtype=torch.float32)
    gv = torch.empty(B, num_dof, device=times.device, dtype=torch.float32)
    _lib.call("tce_prodmp_traj_bwd", tables, _p(grad_traj), _p(times), _p(init_time), _p(gp), _p(gy), _p(gv),
              B, T, _stream())
    return gp, gy, gv


def _traj_setup(ctx, inputs, output):
    params, times, init_time, init_pos, init_vel, tables, num_dof = inputs
    ctx.save_for_backward(times, init_time)
    ctx.tables, ctx.num_dof, ctx.dim_params = tables, num_dof, params.shape[-1]


def _traj_backward(ctx, grad):
    times, init_time = ctx.saved_tensors
    gp, gy, gv = prodmp_traj_bwd(grad, times, init_time, ctx.tables, ctx.num_dof, ctx.dim_params)
    return gp, None, None, gy, gv, None, None


prodmp_traj.register_autograd(_traj_backward, setup_context=_traj_setup)


# --------------------------------------------------------------------------------------------------
# (2) Gaussian sampling, Cholesky, head, stats
# --------------------------------------------------------------------------------------------------
@torch.library.custom_op("tce::mvn_rsample", mutates_args=())
def mvn_rsample(mean: Tensor, L: Tensor, eps: Optional[Tensor], seed: int, offset: int) -> Tensor:
    mean = _chk(mean, name="mean")
    L, ldb = _batched_matrix(L)
    eps_c = None if eps is None else _chk(eps, name="eps")
    B, n = mean.shape
    out = torch.empty_like(mean)
    _lib.call("tce_mvn_rsample", _p(mean), _p(L), ldb, _p(eps_c), seed, offset, _p(out), B, n, _stream())
    return out


@mvn_rsample.register_fake
def _(mean, L, eps, seed, offset):
    return torch.empty_like(mean)


def _rsample_setup(ctx, inputs, output):
    mean, L, eps, seed, offset = inputs
    ctx.save_for_backward(L if eps is not None and eps.requires_grad else None, eps)
    ctx.seed, ctx.offset = seed, offset


def _rsample_backward(ctx, g):
    """out = mean + tril(L) eps: d/dmean = g, d/dL[b] = tril(g[b] eps[b]^T) (dense: autograd sums it for a stride-0
    expanded factor), d/deps = tril(L)^T g.  In-kernel draws are regenerated from (seed, offset): the Philox counter
    is the element index b * n + j whatever the factor, so the identity at stride 0 returns the forward's eps."""
    L, eps = ctx.saved_tensors
    g_L = g_eps = None
    if ctx.needs_input_grad[1]:
        if eps is None:
            B, n = g.shape
            eye = torch.eye(n, device=g.device, dtype=torch.float32).expand(B, n, n)
            eps = mvn_rsample(g.new_zeros(B, n), eye, None, ctx.seed, ctx.offset)
        g_L = torch.tril(g.unsqueeze(-1) * eps.unsqueeze(-2))
    if ctx.needs_input_grad[2]:
        g_eps = torch.einsum('bij,bi->bj', torch.tril(L), g)
    return (g if ctx.needs_input_grad[0] else None), g_L, g_eps, None, None


mvn_rsample.register_autograd(_rsample_backward, setup_context=_rsample_setup)


@torch.library.custom_op("tce::chol_fwd", mutates_args=())
def chol_fwd(A: Tensor) -> Tuple[Tensor, Tensor]:
    A = _chk(A, name="A")
    B, n = A.shape[0], A.shape[-1]
    L = torch.empty_like(A)
    info = torch.empty(B, device=A.device, dtype=torch.int32)
    _lib.call("tce_chol_fwd", _p(A), _p(L), _p(info), B, n, _stream())
    return L, info


@chol_fwd.register_fake
def _(A):
    return torch.empty_like(A), A.new_empty(A.shape[0], dtype=torch.int32)


@torch.library.custom_op("tce::chol_bwd", mutates_args=())
def chol_bwd(L: Tensor, grad_L: Tensor) -> Tensor:
    L, grad_L = _chk(L), _chk(grad_L)
    gA = torch.empty_like(L)
    _lib.call("tce_chol_bwd", _p(L), _p(grad_L), _p(gA), L.shape[0], L.shape[-1], _stream())
    return gA


@chol_bwd.register_fake
def _(L, grad_L):
    return torch.empty_like(L)


def _chol_setup(ctx, inputs, output):
    ctx.save_for_backward(output[0])


def _chol_backward(ctx, gL, ginfo):
    (L,) = ctx.saved_tensors
    return chol_bwd(L, gL)


chol_fwd.register_autograd(_chol_backward, setup_context=_chol_setup)


def cholesky(A: Tensor) -> Tensor:
    """Batched Cholesky of [B, n, n] SPD matrices (differentiable)."""
    return chol_fwd(A)[0]


@torch.library.custom_op("tce::policy_head", mutates_args=())
def policy_head(vec: Tensor, batch: int, dim: int, min_std: float) -> Tensor:
    """cov vector [nvec] (shared) or [B, nvec] -> L [B, dim, dim]."""
    vec = _chk(vec, name="cov vector")
    ldb = 0 if vec.dim() == 1 else vec.shape[-1]
    L = torch.empty(batch, dim, dim, device=vec.device, dtype=torch.float32)
    _lib.call("tce_policy_head_fwd", _p(vec), ldb, float(min_std), _p(L), batch, dim, _stream())
    return L


@policy_head.register_fake
def _(vec, batch, dim, min_std):
    return vec.new_empty(batch, dim, dim)


@torch.library.custom_op("tce::policy_head_bwd", mutates_args=())
def policy_head_bwd(vec: Tensor, grad_L: Tensor) -> Tensor:
    vec, grad_L = _chk(vec), _chk(grad_L)
    ldb = 0 if vec.dim() == 1 else vec.shape[-1]
    g = torch.empty_like(vec)
    _lib.call("tce_policy_head_bwd", _p(vec), ldb, _p(grad_L), _p(g), grad_L.shape[0], grad_L.shape[-1], _stream())
    return g


@policy_head_bwd.register_fake
def _(vec, grad_L):
    return torch.empty_like(vec)


def _head_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0])


def _head_backward(ctx, gL):
    (vec,) = ctx.saved_tensors
    return policy_head_bwd(vec, gL), None, None, None


policy_head.register_autograd(_head_backward, setup_context=_head_setup)


@torch.library.custom_op("tce::policy_head_diag", mutates_args=())
def policy_head_diag(vec: Tensor, batch: int, dim: int, min_std: float) -> Tensor:
    """std vector [dim] (shared) or [B, dim] -> L [B, dim, dim] = diag(softplus(vec) + min_std)."""
    vec = _chk(vec, name="std vector")
    ldb = 0 if vec.dim() == 1 else vec.shape[-1]
    L = torch.empty(batch, dim, dim, device=vec.device, dtype=torch.float32)
    _lib.call("tce_policy_head_diag_fwd", _p(vec), ldb, float(min_std), _p(L), batch, dim, _stream())
    return L


@policy_head_diag.register_fake
def _(vec, batch, dim, min_std):
    return vec.new_empty(batch, dim, dim)


@torch.library.custom_op("tce::policy_head_diag_bwd", mutates_args=())
def policy_head_diag_bwd(vec: Tensor, grad_L: Tensor) -> Tensor:
    vec, grad_L = _chk(vec), _chk(grad_L)
    ldb = 0 if vec.dim() == 1 else vec.shape[-1]
    g = torch.empty_like(vec)
    _lib.call("tce_policy_head_diag_bwd", _p(vec), ldb, _p(grad_L), _p(g), grad_L.shape[0], grad_L.shape[-1], _stream())
    return g


@policy_head_diag_bwd.register_fake
def _(vec, grad_L):
    return torch.empty_like(vec)


def _head_diag_backward(ctx, gL):
    (vec,) = ctx.saved_tensors
    return policy_head_diag_bwd(vec, gL), None, None, None


policy_head_diag.register_autograd(_head_diag_backward, setup_context=_head_setup)


@torch.library.custom_op("tce::gauss_stats", mutates_args=())
def gauss_stats(mean: Tensor, L: Tensor, mean_o: Tensor, L_o: Tensor) -> Tensor:
    """[B, 5] float64: maha, tr(Sigma_o^-1 Sigma), logdet Sigma, logdet Sigma_o, entropy(mean, L)."""
    mean, mean_o = _chk(mean), _chk(mean_o)
    L, ldb = _batched_matrix(L)
    L_o, ldbo = _batched_matrix(L_o, "L_o")
    B, n = mean.shape
    out = torch.empty(B, 5, device=mean.device, dtype=torch.float64)
    _lib.call("tce_gauss_stats", _p(mean), _p(L), ldb, _p(mean_o), _p(L_o), ldbo, _p(out), B, n, _stream())
    return out


@gauss_stats.register_fake
def _(mean, L, mean_o, L_o):
    return mean.new_empty(mean.shape[0], 5, dtype=torch.float64)


# --------------------------------------------------------------------------------------------------
# (3) segment-wise trajectory likelihood
# --------------------------------------------------------------------------------------------------
# Two implementations of the likelihood.  A shared covariance runs the fused kernels in ops_seglik.py (re-exported at
# the end of this module); per-episode factors run the STAGED ops below (gram / chol / bwd with an fp64 HBM workspace,
# see ops_seglik.PER_EPISODE_STAGED).  The staged gram kernel also serves mp.ProDMP.get_traj_pos_cov, and the tests use
# the staged ops as an independent reference for the fused kernels.
from .ops_seglik import (set_regulariser_group, _reduce_diag_max, unit_seed, sync_uniform,  # noqa: E402
                         diag_strides, _dense_diag_grad)


def _episode_factors(L: Tensor, B: int, n: int) -> Tuple[Tensor, int]:
    """(storage, batch stride) of the per-episode factors L [B, n, n] read by the staged kernels; a stride-0 batch
    expand of one matrix is fine.  A [1, n, n] factor with B > 1 is refused: the kernels would read past its end."""
    if tuple(L.shape) != (B, n, n):
        raise TceError(f"L must be [B, n, n] = [{B}, {n}, {n}], got {list(L.shape)}")
    return _batched_matrix(L)


def _work(tables: int, B: int, P: int, device) -> Tensor:
    nbytes = _lib.load().tce_seglik_work_bytes(tables, B, P)
    return torch.empty(max(nbytes // 8, 1), device=device, dtype=torch.float64)


@torch.library.custom_op("tce::seglik_fwd", mutates_args=())
def seglik_fwd(smp_traj: Tensor, mean: Tensor, L: Tensor, times: Tensor, init_time: Tensor, init_pos: Tensor,
               init_vel: Tensor, pred_pairs: Tensor, tables: int, reg_rel: float) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """-> (logp [B,P], work (fp64 gram matrices + residuals), diag_max [1] fp64, info [B,P] int32)."""
    smp_traj, mean, times = _chk(smp_traj, name="smp_traj"), _chk(mean, name="mean"), _chk(times, name="times")
    init_time, init_pos, init_vel = _chk(init_time), _chk(init_pos), _chk(init_vel)
    pairs = _chk(pred_pairs, torch.int64, "pred_pairs")
    B, T = times.shape
    L, ldb = _episode_factors(L, B, mean.shape[-1])
    P = pairs.shape[0]
    dev = mean.device
    work = _work(tables, B, P, dev)
    diag_max = torch.zeros(1, device=dev, dtype=torch.float64)
    logp = torch.empty(B, P, device=dev, dtype=torch.float32)
    info = torch.empty(B, P, device=dev, dtype=torch.int32)
    st = _stream()
    _lib.call("tce_seglik_gram", tables, _p(smp_traj), _p(mean), _p(L), ldb, _p(times), _p(init_time), _p(init_pos),
              _p(init_vel), _p(pairs), _p(work), _p(diag_max), B, T, P, st)
    _reduce_diag_max(diag_max)
    _lib.call("tce_seglik_chol", tables, _p(work), None, _p(diag_max), float(reg_rel), None, None, None, 0.0, None,
              _p(logp), _p(info), B, P, st)
    return logp, work, diag_max, info


@seglik_fwd.register_fake
def _(smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs, tables, reg_rel):
    B, P = times.shape[0], pred_pairs.shape[0]
    n = smp_traj.shape[-1]
    return (mean.new_empty(B, P), mean.new_empty(B * P * (n * (n + 1) // 2 + n), dtype=torch.float64),
            mean.new_empty(1, dtype=torch.float64), mean.new_empty(B, P, dtype=torch.int32))


@torch.library.custom_op("tce::seglik_bwd", mutates_args=())
def seglik_bwd(grad_logp: Tensor, work: Tensor, diag_max: Tensor, L: Tensor, times: Tensor, init_time: Tensor,
               pred_pairs: Tensor, tables: int, reg_rel: float, dim_params: int) -> Tuple[Tensor, Tensor]:
    grad_logp, times, init_time = _chk(grad_logp), _chk(times), _chk(init_time)
    pairs = _chk(pred_pairs, torch.int64)
    B, T = times.shape
    L, ldb = _episode_factors(L, B, dim_params)
    P = pairs.shape[0]
    dev = times.device
    adj = torch.empty_like(work)
    g_mean = torch.empty(B, dim_params, device=dev, dtype=torch.float32)
    g_L = torch.empty(B, dim_params, dim_params, device=dev, dtype=torch.float32)
    st = _stream()
    _lib.call("tce_seglik_chol", tables, _p(work), _p(adj), _p(diag_max), float(reg_rel), _p(grad_logp), None, None,
              0.0, None, None, None, B, P, st)
    _lib.call("tce_seglik_bwd", tables, _p(adj), _p(L), ldb, _p(times), _p(init_time), _p(pairs), None, _p(g_mean),
              _p(g_L), B, T, P, st)
    return g_mean, g_L


@seglik_bwd.register_fake
def _(grad_logp, work, diag_max, L, times, init_time, pred_pairs, tables, reg_rel, dim_params):
    B = times.shape[0]
    return times.new_empty(B, dim_params), times.new_empty(B, dim_params, dim_params)


def _seglik_setup(ctx, inputs, output):
    smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs, tables, reg_rel = inputs
    logp, work, diag_max, info = output
    ctx.save_for_backward(work, diag_max, L, times, init_time, pred_pairs)
    ctx.tables, ctx.reg_rel, ctx.dim_params = tables, reg_rel, mean.shape[-1]
    ctx.L_expanded = L.dim() == 3 and L.stride(0) == 0
    ctx.set_materialize_grads(False)


def _seglik_backward(ctx, g_logp, g_work, g_diag, g_info):
    work, diag_max, L, times, init_time, pred_pairs = ctx.saved_tensors
    if g_logp is None:
        return (None,) * 10
    g_mean, g_L = seglik_bwd(g_logp, work, diag_max, L, times, init_time, pred_pairs, ctx.tables, ctx.reg_rel,
                             ctx.dim_params)
    return None, g_mean, g_L, None, None, None, None, None, None, None


seglik_fwd.register_autograd(_seglik_backward, setup_context=_seglik_setup)


def seg_logprob_staged(smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs, tables: Tables,
                       reg_rel: float = 1e-4, return_info: bool = False):
    """Segment-wise log-likelihood [B, P] (differentiable w.r.t. ``mean`` and ``L``), staged kernels."""
    logp, _work_, diag_max, info = seglik_fwd(smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs,
                                              tables.handle, reg_rel)
    return (logp, info, diag_max) if return_info else logp


@torch.library.custom_op("tce::seglik_surrogate_fwd", mutates_args=())
def seglik_surrogate_fwd(smp_traj: Tensor, mean: Tensor, L: Tensor, times: Tensor, init_time: Tensor,
                         init_pos: Tensor, init_vel: Tensor, pred_pairs: Tensor, logp_old: Tensor, advantage: Tensor,
                         tables: int, reg_rel: float) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """Fused segment likelihood + importance-sampling surrogate (temporal_correlated_agent.py:718-739).

    -> (stats [2] fp64 = {-mean(ratio * adv), mean(ratio)}, logp [B,P], adj (per-segment adjoints for the
    backward stage, already scaled by d loss / d logp), info [B,P]).
    """
    smp_traj, mean, times = _chk(smp_traj, name="smp_traj"), _chk(mean, name="mean"), _chk(times, name="times")
    init_time, init_pos, init_vel = _chk(init_time), _chk(init_pos), _chk(init_vel)
    logp_old, advantage = _chk(logp_old, name="logp_old"), _chk(advantage, name="advantage")
    pairs = _chk(pred_pairs, torch.int64, "pred_pairs")
    B, T = times.shape
    L, ldb = _episode_factors(L, B, mean.shape[-1])
    P = pairs.shape[0]
    dev = mean.device
    work = _work(tables, B, P, dev)
    diag_max = torch.zeros(1, device=dev, dtype=torch.float64)
    stats = torch.zeros(2, device=dev, dtype=torch.float64)
    logp = torch.empty(B, P, device=dev, dtype=torch.float32)
    info = torch.empty(B, P, device=dev, dtype=torch.int32)
    st = _stream()
    _lib.call("tce_seglik_gram", tables, _p(smp_traj), _p(mean), _p(L), ldb, _p(times), _p(init_time), _p(init_pos),
              _p(init_vel), _p(pairs), _p(work), _p(diag_max), B, T, P, st)
    _reduce_diag_max(diag_max)
    _lib.call("tce_seglik_chol", tables, _p(work), _p(work), _p(diag_max), float(reg_rel), None, _p(logp_old),
              _p(advantage), 1.0 / (B * P), _p(stats), _p(logp), _p(info), B, P, st)
    return stats, logp, work, info


@seglik_surrogate_fwd.register_fake
def _(smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs, logp_old, advantage, tables, reg_rel):
    B, P = times.shape[0], pred_pairs.shape[0]
    n = smp_traj.shape[-1]
    return (mean.new_empty(2, dtype=torch.float64), mean.new_empty(B, P),
            mean.new_empty(B * P * (n * (n + 1) // 2 + n), dtype=torch.float64), mean.new_empty(B, P, dtype=torch.int32))


@torch.library.custom_op("tce::seglik_surrogate_bwd", mutates_args=())
def seglik_surrogate_bwd(upstream: Tensor, adj: Tensor, L: Tensor, times: Tensor, init_time: Tensor,
                         pred_pairs: Tensor, tables: int, dim_params: int) -> Tuple[Tensor, Tensor]:
    times, init_time = _chk(times), _chk(init_time)
    pairs = _chk(pred_pairs, torch.int64)
    up = _chk(upstream, torch.float32, "upstream")
    B, T = times.shape
    L, ldb = _episode_factors(L, B, dim_params)
    P = pairs.shape[0]
    g_mean = torch.empty(B, dim_params, device=times.device, dtype=torch.float32)
    g_L = torch.empty(B, dim_params, dim_params, device=times.device, dtype=torch.float32)
    _lib.call("tce_seglik_bwd", tables, _p(adj), _p(L), ldb, _p(times), _p(init_time), _p(pairs), _p(up), _p(g_mean),
              _p(g_L), B, T, P, _stream())
    return g_mean, g_L


@seglik_surrogate_bwd.register_fake
def _(upstream, adj, L, times, init_time, pred_pairs, tables, dim_params):
    B = times.shape[0]
    return times.new_empty(B, dim_params), times.new_empty(B, dim_params, dim_params)


def _sur_setup(ctx, inputs, output):
    (smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs, logp_old, advantage, tables, reg_rel) = inputs
    ctx.save_for_backward(output[2], L, times, init_time, pred_pairs)
    ctx.tables, ctx.dim_params = tables, mean.shape[-1]
    ctx.set_materialize_grads(False)


def _sur_backward(ctx, g_stats, g_logp, g_adj, g_info):
    adj, L, times, init_time, pred_pairs = ctx.saved_tensors
    none = (None,) * 12
    if g_stats is None:
        return none
    if g_stats is _E0.get(str(g_stats.device)):            # unit seed (see unit_seed): d total / d surrogate = 1
        up = unit_seed(g_stats.device, torch.float32).reshape(1)
    else:
        up = g_stats[0].to(torch.float32).reshape(1)       # d total / d surrogate loss (device scalar, no sync)
    g_mean, g_L = seglik_surrogate_bwd(up, adj, L, times, init_time, pred_pairs, ctx.tables, ctx.dim_params)
    return None, g_mean, g_L, None, None, None, None, None, None, None, None, None


seglik_surrogate_fwd.register_autograd(_sur_backward, setup_context=_sur_setup)


def seg_surrogate_staged(smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs, logp_old, advantage,
                         tables: Tables, reg_rel: float = 1e-4):
    """Staged kernels -> (surrogate loss = -mean(exp(lp - lp_old) * adv) [fp32 scalar, differentiable], mean ratio, logp)."""
    stats, logp, _adj, _info = seglik_surrogate_fwd(smp_traj, mean, L, times, init_time, init_pos, init_vel,
                                                    pred_pairs, logp_old, advantage, tables.handle, reg_rel)
    loss, ratio = _StatsToFloat.apply(stats)
    return loss, ratio.detach(), logp.detach()


_E0 = {}


class _StatsToFloat(torch.autograd.Function):
    """fp64 {loss, ratio} [2] -> two fp32 scalars with ONE kernel each way (select + cast + zero-fill + scatter
    of the plain formulation are four launches on the critical path between the likelihood's stage 2 and 3)."""

    @staticmethod
    def forward(ctx, stats):
        key = str(stats.device)
        if key not in _E0:
            _E0[key] = torch.tensor([1.0, 0.0], dtype=torch.float64, device=stats.device)
        ctx.e0 = _E0[key]
        ctx.set_materialize_grads(False)
        s32 = stats.to(torch.float32)
        return s32[0], s32[1]

    @staticmethod
    def backward(ctx, g_loss, g_ratio):
        if g_loss is None:
            return None
        if g_loss is unit_seed(g_loss.device, g_loss.dtype):   # seeded with the cached 1: no kernel at all
            return ctx.e0
        return ctx.e0 * g_loss                            # fp64 [2] = {d/d loss, 0}


# --------------------------------------------------------------------------------------------------
# (4b) GAE and segment advantages
# --------------------------------------------------------------------------------------------------
@torch.library.custom_op("tce::gae", mutates_args=())
def gae(rewards: Tensor, values: Tensor, dones: Tensor, time_limit_dones: Tensor, gamma: float, lam: float,
        use_gae: bool) -> Tuple[Tensor, Tensor]:
    rewards, values = _chk(rewards, name="rewards"), _chk(values, name="values")
    dn = _chk(dones.view(torch.uint8) if dones.dtype == torch.bool else dones, torch.uint8, "dones")
    tl = _chk(time_limit_dones.view(torch.uint8) if time_limit_dones.dtype == torch.bool else time_limit_dones,
              torch.uint8, "time_limit_dones")
    B, T = rewards.shape
    adv, ret = torch.empty_like(rewards), torch.empty_like(rewards)
    _lib.call("tce_gae", _p(rewards), _p(values), _p(dn), _p(tl), float(gamma), float(lam), int(use_gae), _p(adv),
              _p(ret), B, T, _stream())
    return adv, ret


@gae.register_fake
def _(rewards, values, dones, time_limit_dones, gamma, lam, use_gae):
    return torch.empty_like(rewards), torch.empty_like(rewards)


_STATS_GROUP = None


def set_stats_group(group) -> None:
    """At >1 GPU, all-reduce(SUM) {count, sum, sum sq} of the advantage normalisation over ``group``."""
    global _STATS_GROUP
    _STATS_GROUP = group


def _reduce_stats(stats: Tensor) -> None:
    if _STATS_GROUP is not None:
        import torch.distributed as dist
        dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=None if _STATS_GROUP is True else _STATS_GROUP)


@torch.library.custom_op("tce::segment_advantage", mutates_args=())
def segment_advantage(mode: int, rewards: Tensor, values: Tensor, advantages: Tensor, pred_pairs: Tensor,
                      gamma: float, normalize: bool) -> Tensor:
    """mode 0 accumulate / 1 value_subtraction / 2 accumulated rewards (raw); optional global normalisation."""
    rewards, values, advantages = _chk(rewards), _chk(values), _chk(advantages)
    pairs = _chk(pred_pairs, torch.int64)
    B, T = rewards.shape
    P = pairs.shape[0]
    seg = torch.empty(B, P, device=rewards.device, dtype=torch.float32)
    stats = torch.zeros(3, device=rewards.device, dtype=torch.float64)
    st = _stream()
    _lib.call("tce_segment_advantage_raw", int(mode), _p(rewards), _p(values), _p(advantages), _p(pairs),
              float(gamma), _p(seg), _p(stats), B, T, P, st)
    if normalize:
        _reduce_stats(stats)
        _lib.call("tce_normalize_by_stats", _p(seg), _p(stats), B * P, st)
    return seg


@segment_advantage.register_fake
def _(mode, rewards, values, advantages, pred_pairs, gamma, normalize):
    return rewards.new_empty(rewards.shape[0], pred_pairs.shape[0])


@torch.library.custom_op("tce::normalize", mutates_args=())
def normalize(x: Tensor) -> Tensor:
    """(x - mean) / (unbiased std + 1e-8) over all elements (advantage normalisation)."""
    x = _chk(x).clone()
    stats = torch.zeros(3, device=x.device, dtype=torch.float64)
    st = _stream()
    _lib.call("tce_sum_stats", _p(x), _p(stats), x.numel(), st)
    _reduce_stats(stats)
    _lib.call("tce_normalize_by_stats", _p(x), _p(stats), x.numel(), st)
    return x


@normalize.register_fake
def _(x):
    return torch.empty_like(x)


@torch.library.custom_op("tce::gauss_maha", mutates_args=())
def gauss_maha(mean: Tensor, mean_o: Tensor, L_o: Tensor) -> Tensor:
    """|L_o^-1 (mean - mean_o)|^2  [B] fp64 (``policy.maha``); differentiable w.r.t. all three arguments."""
    mean, mean_o = _chk(mean), _chk(mean_o)
    B, n = mean.shape
    L_o, ldbo = _batched_matrix(L_o, "L_o", batch=B)
    out = torch.empty(B, device=mean.device, dtype=torch.float64)
    _lib.call("tce_gauss_maha", _p(mean), _p(mean_o), _p(L_o), ldbo, None, _p(out), None, B, n, _stream())
    return out


@gauss_maha.register_fake
def _(mean, mean_o, L_o):
    return mean.new_empty(mean.shape[0], dtype=torch.float64)


@torch.library.custom_op("tce::gauss_maha_bwd", mutates_args=())
def gauss_maha_bwd(grad: Tensor, mean: Tensor, mean_o: Tensor, L_o: Tensor) -> Tensor:
    mean, mean_o = _chk(mean), _chk(mean_o)
    B, n = mean.shape
    L_o, ldbo = _batched_matrix(L_o, "L_o", batch=B)
    g = _chk(grad, torch.float64, "grad")
    g_mean = torch.empty_like(mean)
    _lib.call("tce_gauss_maha", _p(mean), _p(mean_o), _p(L_o), ldbo, _p(g), None, _p(g_mean), B, n, _stream())
    return g_mean


@gauss_maha_bwd.register_fake
def _(grad, mean, mean_o, L_o):
    return torch.empty_like(mean)


@torch.library.custom_op("tce::gauss_maha_bwd_full", mutates_args=())
def gauss_maha_bwd_full(grad: Tensor, mean: Tensor, mean_o: Tensor, L_o: Tensor, need_L: bool) -> Tuple[Tensor, Tensor]:
    """-> (d maha / d mean [B, n] (= -d maha / d mean_o), d maha / d L_o [B, n, n] or empty)."""
    mean, mean_o = _chk(mean), _chk(mean_o)
    B, n = mean.shape
    Lc, ldbo = _batched_matrix(L_o, "L_o", batch=B)
    g = _chk(grad, torch.float64, "grad")
    g_mean = torch.empty_like(mean)
    g_L = torch.empty(B, n, n, device=mean.device, dtype=torch.float32) if need_L else mean.new_empty(0)
    _lib.call("tce_gauss_maha_bwd_full", _p(mean), _p(mean_o), _p(Lc), ldbo, _p(g), _p(g_mean),
              _p(g_L) if need_L else None, B, n, _stream())
    return g_mean, g_L


@gauss_maha_bwd_full.register_fake
def _(grad, mean, mean_o, L_o, need_L):
    B, n = mean.shape
    return torch.empty_like(mean), (mean.new_empty(B, n, n) if need_L else mean.new_empty(0))


def _gm_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs)


def _gm_backward(ctx, g):
    mean, mean_o, L_o = ctx.saved_tensors
    if not (ctx.needs_input_grad[1] or ctx.needs_input_grad[2]):
        return gauss_maha_bwd(g, mean, mean_o, L_o), None, None
    g_mean, g_L = gauss_maha_bwd_full(g, mean, mean_o, L_o, bool(ctx.needs_input_grad[2]))
    if ctx.needs_input_grad[2] and L_o.shape[0] != mean.shape[0]:      # one factor [1, n, n] for the whole batch
        g_L = g_L.sum(dim=0, keepdim=True)
    return (g_mean if ctx.needs_input_grad[0] else None, -g_mean if ctx.needs_input_grad[1] else None,
            g_L if ctx.needs_input_grad[2] else None)


gauss_maha.register_autograd(_gm_backward, setup_context=_gm_setup)


@torch.library.custom_op("tce::tri_inverse", mutates_args=())
def tri_inverse(L: Tensor) -> Tensor:
    """L^-1 [Bc, n, n] fp64 of lower-triangular factors (not differentiable: used for detached / old factors)."""
    L = _chk(L, name="L")
    Bc, n = L.shape[0], L.shape[-1]
    out = torch.empty(Bc, n, n, device=L.device, dtype=torch.float64)
    _lib.call("tce_tri_inverse", _p(L), n * n, _p(out), Bc, n, _stream())
    return out


@tri_inverse.register_fake
def _(L):
    return L.new_empty(L.shape, dtype=torch.float64)


@torch.library.custom_op("tce::gauss_maha_shared_fwd", mutates_args=())
def gauss_maha_shared_fwd(mean: Tensor, mean_o: Tensor, Linv: Tensor, with_grad: bool) -> Tuple[Tensor, Tensor]:
    """-> (maha [B] fp64, d maha / d mean [B, n] fp32 or an empty tensor): the gradient is formed in the forward
    (two more matrix-vector products per episode) so that the backward is a single elementwise product."""
    mean, mean_o, Linv = _chk(mean), _chk(mean_o), _chk(Linv, torch.float64, "Linv")
    B, n = mean.shape
    out = torch.empty(B, device=mean.device, dtype=torch.float64)
    dmean = torch.empty_like(mean) if with_grad else mean.new_empty(0)
    _lib.call("tce_gauss_maha_shared", _p(mean), _p(mean_o), _p(Linv), None, _p(out),
              _p(dmean) if with_grad else None, B, n, _stream())
    return out, dmean


@gauss_maha_shared_fwd.register_fake
def _(mean, mean_o, Linv, with_grad):
    return mean.new_empty(mean.shape[0], dtype=torch.float64), (torch.empty_like(mean) if with_grad else mean.new_empty(0))


def _gms_setup(ctx, inputs, output):
    ctx.save_for_backward(output[1])
    ctx.set_materialize_grads(False)


def _gms_backward(ctx, g, g_dmean):
    (dmean,) = ctx.saved_tensors
    if g is None or dmean.numel() == 0:
        return None, None, None, None
    return g.to(dmean.dtype).unsqueeze(-1) * dmean, None, None, None


gauss_maha_shared_fwd.register_autograd(_gms_backward, setup_context=_gms_setup)


def gauss_maha_shared(mean: Tensor, mean_o: Tensor, Linv: Tensor) -> Tensor:
    """``gauss_maha`` for ONE covariance shared by all episodes, given ``Linv = tri_inverse(L_o)[0]`` [n, n];
    differentiable w.r.t. ``mean``."""
    need = torch.is_grad_enabled() and mean.requires_grad
    return gauss_maha_shared_fwd(mean, mean_o, Linv, need)[0]


@torch.library.custom_op("tce::gauss_maha_shared_bwd", mutates_args=())
def gauss_maha_shared_bwd(grad: Tensor, mean: Tensor, mean_o: Tensor, Linv: Tensor) -> Tensor:
    """Stand-alone gradient kernel (tests, C-ABI coverage): grad[b] * d maha / d mean."""
    mean, mean_o, Linv = _chk(mean), _chk(mean_o), _chk(Linv, torch.float64, "Linv")
    B, n = mean.shape
    g = _chk(grad, torch.float64, "grad")
    g_mean = torch.empty_like(mean)
    _lib.call("tce_gauss_maha_shared", _p(mean), _p(mean_o), _p(Linv), _p(g), None, _p(g_mean), B, n, _stream())
    return g_mean


@gauss_maha_shared_bwd.register_fake
def _(grad, mean, mean_o, Linv):
    return torch.empty_like(mean)


# --------------------------------------------------------------------------------------------------
# (4a) trust-region projection building blocks (each: hand-written forward + backward kernels)
# --------------------------------------------------------------------------------------------------
@torch.library.custom_op("tce::gauss_stats_bwd", mutates_args=())
def gauss_stats_bwd(grad_out: Tensor, mean: Tensor, L: Tensor, mean_o: Tensor, L_o: Tensor,
                    need_L: bool) -> Tuple[Tensor, Tensor]:
    mean, mean_o = _chk(mean), _chk(mean_o)
    g = _chk(grad_out, torch.float64, "grad_out")
    Lc, ldb = _batched_matrix(L)
    L_oc, ldbo = _batched_matrix(L_o, "L_o")
    B, n = mean.shape
    g_mean = torch.empty_like(mean)
    g_L = torch.empty(B, n, n, device=mean.device, dtype=torch.float32) if need_L else mean.new_empty(0)
    _lib.call("tce_gauss_stats_bwd", _p(mean), _p(Lc), ldb, _p(mean_o), _p(L_oc), ldbo, _p(g), _p(g_mean),
              _p(g_L) if need_L else None, B, n, _stream())
    return g_mean, g_L


@gauss_stats_bwd.register_fake
def _(grad_out, mean, L, mean_o, L_o, need_L):
    B, n = mean.shape
    return torch.empty_like(mean), (mean.new_empty(B, n, n) if need_L else mean.new_empty(0))


def _gs_setup(ctx, inputs, output):
    mean, L, mean_o, L_o = inputs
    ctx.save_for_backward(mean, L, mean_o, L_o)
    ctx.need_L = L.requires_grad


def _gs_backward(ctx, g):
    mean, L, mean_o, L_o = ctx.saved_tensors
    g_mean, g_L = gauss_stats_bwd(g.contiguous(), mean, L, mean_o, L_o, ctx.need_L)
    return g_mean, (g_L if ctx.need_L else None), None, None


gauss_stats.register_autograd(_gs_backward, setup_context=_gs_setup)


@torch.library.custom_op("tce::proj_mean", mutates_args=())
def proj_mean(mean: Tensor, mean_o: Tensor, mean_part: Tensor, eps: float) -> Tensor:
    mean, mean_o = _chk(mean), _chk(mean_o)
    mp = _chk(mean_part, torch.float64, "mean_part")
    out = torch.empty_like(mean)
    _lib.call("tce_proj_mean_fwd", _p(mean), _p(mean_o), _p(mp), float(eps), _p(out), mean.shape[0], mean.shape[1],
              _stream())
    return out


@proj_mean.register_fake
def _(mean, mean_o, mean_part, eps):
    return torch.empty_like(mean)


@torch.library.custom_op("tce::proj_mean_bwd", mutates_args=())
def proj_mean_bwd(grad_out: Tensor, mean: Tensor, mean_o: Tensor, mean_part: Tensor, eps: float) -> Tuple[Tensor, Tensor]:
    g, mean, mean_o = _chk(grad_out), _chk(mean), _chk(mean_o)
    mp = _chk(mean_part, torch.float64)
    g_mean, g_part = torch.empty_like(mean), torch.empty_like(mp)
    _lib.call("tce_proj_mean_bwd", _p(mean), _p(mean_o), _p(mp), float(eps), _p(g), _p(g_mean), _p(g_part),
              mean.shape[0], mean.shape[1], _stream())
    return g_mean, g_part


@proj_mean_bwd.register_fake
def _(grad_out, mean, mean_o, mean_part, eps):
    return torch.empty_like(mean), torch.empty_like(mean_part)


def _pm_setup(ctx, inputs, output):
    mean, mean_o, mean_part, eps = inputs
    ctx.save_for_backward(mean, mean_o, mean_part)
    ctx.eps = eps


def _pm_backward(ctx, g):
    mean, mean_o, mean_part = ctx.saved_tensors
    g_mean, g_part = proj_mean_bwd(g, mean, mean_o, mean_part, ctx.eps)
    return g_mean, None, g_part, None


proj_mean.register_autograd(_pm_backward, setup_context=_pm_setup)


@torch.library.custom_op("tce::proj_entropy", mutates_args=())
def proj_entropy(L: Tensor, beta: Tensor, equality: bool) -> Tuple[Tensor, Tensor]:
    """-> (projected L [Bc,n,n], entropy before projection [Bc] fp64); beta [Bc] or [1] fp64."""
    L = _chk(L, name="L")
    beta = _chk(beta, torch.float64, "beta")
    Bc, n = L.shape[0], L.shape[-1]
    out = torch.empty_like(L)
    ent = torch.empty(Bc, device=L.device, dtype=torch.float64)
    _lib.call("tce_proj_entropy_fwd", _p(L), _p(beta), 0 if beta.numel() == 1 else 1, int(equality), _p(out), _p(ent),
              Bc, n, _stream())
    return out, ent


@proj_entropy.register_fake
def _(L, beta, equality):
    return torch.empty_like(L), L.new_empty(L.shape[0], dtype=torch.float64)


@torch.library.custom_op("tce::proj_entropy_bwd", mutates_args=())
def proj_entropy_bwd(grad_out: Tensor, L: Tensor, beta: Tensor, equality: bool) -> Tensor:
    g, L = _chk(grad_out), _chk(L)
    beta = _chk(beta, torch.float64)
    out = torch.empty_like(L)
    _lib.call("tce_proj_entropy_bwd", _p(L), _p(beta), 0 if beta.numel() == 1 else 1, int(equality), _p(g), _p(out),
              L.shape[0], L.shape[-1], _stream())
    return out


@proj_entropy_bwd.register_fake
def _(grad_out, L, beta, equality):
    return torch.empty_like(L)


def _pe_setup(ctx, inputs, output):
    L, beta, equality = inputs
    ctx.save_for_backward(L, beta)
    ctx.equality = equality


def _pe_backward(ctx, g, g_ent):
    L, beta = ctx.saved_tensors
    return proj_entropy_bwd(g, L, beta, ctx.equality), None, None


proj_entropy.register_autograd(_pe_backward, setup_context=_pe_setup)


def kl_state_size(batch: int, n: int) -> int:
    return _lib.load().tce_proj_kl_save_doubles(batch, n)


def kl_state_sigma(state: Tensor, batch: int, n: int) -> Tuple[Tensor, Tensor]:
    """Views into a KL state buffer: (Sigma of the projected covariance before the entropy control [batch, n, n],
    alpha^2 of the fused entropy control [batch]) -- Sigma of the layer's output is alpha^2 * Sigma."""
    nn = batch * n * n
    sc = kl_state_scalars(state, batch, n)
    return state[3 * nn:4 * nn].view(batch, n, n), sc[:, 6]


KL_STATE_SCALARS = 16


def kl_state_scalars(state: Tensor, batch: int, n: int) -> Tensor:
    """[batch, 16] view: eta, KL step active, KL before the projection, fingerprint(L_old), alpha, entropy control
    active, alpha^2, [7:9] shape and volume part of KL_cov(N(Sigma_in) || N(Sigma_out)) (the trust-region loss),
    [9] entropy of the output, [10:12] shape / volume of KL(in || old), [12:14] shape / volume of KL(out || old)."""
    o = 4 * batch * n * n + batch * n
    return state[o:o + batch * KL_STATE_SCALARS].view(batch, KL_STATE_SCALARS)


def kl_state(batch: int, n: int, device) -> Tensor:
    """Zero-initialised state buffer of the KL covariance projection ({M, lambda, eta/active/kl0/fingerprint})."""
    return torch.zeros(_lib.load().tce_proj_kl_save_doubles(batch, n), device=device, dtype=torch.float64)


@torch.library.custom_op("tce::proj_kl_cov_fwd", mutates_args=("state",))
def proj_kl_cov_fwd(L: Tensor, L_o: Tensor, eps_cov: float, state: Tensor, warm: bool) -> Tuple[Tensor, Tensor]:
    L, L_o = _chk(L, name="L"), _chk(L_o, name="L_o")
    Bc, n = L.shape[0], L.shape[-1]
    if state.dtype != torch.float64 or not state.is_cuda or state.numel() != _lib.load().tce_proj_kl_save_doubles(Bc, n):
        raise TceError("state must come from ops.kl_state(batch, n, device)")
    out = torch.empty_like(L)
    info = torch.empty(Bc, device=L.device, dtype=torch.int32)
    _lib.call("tce_proj_kl_cov_fwd", _p(L), _p(L_o), float(eps_cov), _p(out), _p(state), _p(info), int(warm), Bc, n,
              _stream())
    return out, info


@proj_kl_cov_fwd.register_fake
def _(L, L_o, eps_cov, state, warm):
    return torch.empty_like(L), L.new_empty(L.shape[0], dtype=torch.int32)


@torch.library.custom_op("tce::proj_kl_cov_bwd", mutates_args=())
def proj_kl_cov_bwd(grad_out: Tensor, L: Tensor, proj_L: Tensor, state: Tensor) -> Tensor:
    g, L, proj_L = _chk(grad_out), _chk(L), _chk(proj_L)
    out = torch.empty_like(L)
    _lib.call("tce_proj_kl_cov_bwd", _p(L), _p(proj_L), _p(g), _p(state), _p(out), L.shape[0], L.shape[-1], _stream())
    return out


@proj_kl_cov_bwd.register_fake
def _(grad_out, L, proj_L, state):
    return torch.empty_like(L)


def _check_generation(ctx):
    """The state buffer of a warm-started layer is overwritten by its NEXT forward; a backward that runs after that
    would silently read the wrong eigen-system (two projections in one graph, micro-batch accumulation, ...)."""
    h = ctx.holder
    if h is not None and getattr(h, "_kl_generation", None) != ctx.generation:
        raise RuntimeError("KL projection: backward() after a later forward() of the same layer overwrote its state "
                           "buffer; run backward before projecting again, or use warm_start=False (fresh state "
                           "per call)")


class _ProjKLCov(torch.autograd.Function):
    """Autograd wrapper (a mutating custom op cannot carry an autograd formula itself)."""

    @staticmethod
    def forward(ctx, L, L_o, eps_cov, state, warm, holder):
        proj_L, info = proj_kl_cov_fwd(L, L_o, eps_cov, state, warm)
        ctx.save_for_backward(L, proj_L)
        ctx.state = state        # overwritten by the NEXT forward of a warm-started layer: guarded by a generation
        ctx.holder, ctx.generation = holder, None
        if holder is not None:
            holder._kl_generation = getattr(holder, "_kl_generation", 0) + 1
            ctx.generation = holder._kl_generation
        ctx.mark_non_differentiable(info)
        return proj_L, info

    @staticmethod
    def backward(ctx, g, g_info):
        L, proj_L = ctx.saved_tensors
        _check_generation(ctx)
        return proj_kl_cov_bwd(g.contiguous(), L, proj_L, ctx.state), None, None, None, None, None


SIGMA_READY = {}       # id(state) -> CUDA event recorded after the first half of a split forward


@torch.library.custom_op("tce::proj_kl_entropy_fwd", mutates_args=("state",))
def proj_kl_entropy_fwd(L: Tensor, L_o: Tensor, eps_cov: float, state: Tensor, warm: bool, beta: Tensor,
                        equality: bool, split: bool = False) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """KL covariance projection + entropy control -> (out_L, proj_L (pre-entropy), info).  ``split``: two launches
    (state incl. Sigma first, Cholesky second) with an event in ``SIGMA_READY[id(state)]`` between them."""
    L, L_o = _chk(L, name="L"), _chk(L_o, name="L_o")
    beta = _chk(beta, torch.float64, "beta")
    Bc, n = L.shape[0], L.shape[-1]
    if state.dtype != torch.float64 or not state.is_cuda or state.numel() != _lib.load().tce_proj_kl_save_doubles(Bc, n):
        raise TceError("state must come from ops.kl_state(batch, n, device)")
    out, proj = torch.empty_like(L), torch.empty_like(L)
    info = torch.empty(Bc, device=L.device, dtype=torch.int32)
    if split:
        _lib.call("tce_proj_kl_entropy_fwd_sigma", _p(L), _p(L_o), float(eps_cov), _p(beta),
                  0 if beta.numel() == 1 else 1, int(equality), _p(proj), _p(out), _p(state), _p(info), int(warm), Bc, n,
                  _stream())
        ev = torch.cuda.Event()
        ev.record()
        SIGMA_READY[id(state)] = ev
        out_inv = torch.empty(Bc, n, n, device=L.device, dtype=torch.float64)     # (out_L)^-1 for the trust-region loss
        _lib.call("tce_proj_kl_entropy_fwd_chol", _p(state), _p(proj), _p(out), _p(out_inv), _p(info), Bc, n, _stream())
        return out, proj, info, out_inv
    _lib.call("tce_proj_kl_entropy_fwd", _p(L), _p(L_o), float(eps_cov), _p(beta), 0 if beta.numel() == 1 else 1,
              int(equality), _p(proj), _p(out), _p(state), _p(info), int(warm), Bc, n, _stream())
    return out, proj, info, L.new_empty(0, dtype=torch.float64)


@proj_kl_entropy_fwd.register_fake
def _(L, L_o, eps_cov, state, warm, beta, equality, split=False):
    return (torch.empty_like(L), torch.empty_like(L), L.new_empty(L.shape[0], dtype=torch.int32),
            L.new_empty(L.shape if split else (0,), dtype=torch.float64))


@torch.library.custom_op("tce::proj_kl_entropy_bwd", mutates_args=())
def proj_kl_entropy_bwd(grad_out: Tensor, L: Tensor, proj_L: Tensor, state: Tensor,
                        out_inv: Optional[Tensor] = None) -> Tensor:
    """``out_inv``: inverse [Bc, n, n] fp64 of the layer's OUTPUT factor if somebody already formed it."""
    g, L, proj_L = _chk(grad_out), _chk(L), _chk(proj_L)
    out = torch.empty_like(L)
    if out_inv is not None:
        inv = _chk(out_inv, torch.float64, "out_inv")
        if inv.numel() != L.numel():
            raise TceError("out_inv must have the shape of L")
        _lib.call("tce_proj_kl_entropy_bwd_inv", _p(L), _p(proj_L), _p(g), _p(state), _p(inv), _p(out), L.shape[0],
                  L.shape[-1], _stream())
    else:
        _lib.call("tce_proj_kl_entropy_bwd", _p(L), _p(proj_L), _p(g), _p(state), _p(out), L.shape[0], L.shape[-1],
                  _stream())
    return out


@proj_kl_entropy_bwd.register_fake
def _(grad_out, L, proj_L, state, out_inv=None):
    return torch.empty_like(L)


@torch.library.custom_op("tce::proj_kl_entropy_bwd_tr", mutates_args=())
def proj_kl_entropy_bwd_tr(grad_out: Tensor, L: Tensor, proj_L: Tensor, state: Tensor, tr_coeff: float) -> Tensor:
    """``proj_kl_entropy_bwd`` + the gradient of tr_coeff * KL_cov(N(L L^T) || N(Sigma_out detached)) per matrix."""
    g, L, proj_L = _chk(grad_out), _chk(L), _chk(proj_L)
    out = torch.empty_like(L)
    _lib.call("tce_proj_kl_entropy_bwd_tr", _p(L), _p(proj_L), _p(g), _p(state), float(tr_coeff), _p(out), L.shape[0],
              L.shape[-1], _stream())
    return out


@proj_kl_entropy_bwd_tr.register_fake
def _(grad_out, L, proj_L, state, tr_coeff):
    return torch.empty_like(L)


@torch.library.custom_op("tce::proj_kl_bwd_sigma", mutates_args=())
def proj_kl_bwd_sigma(grad_sigma: Tensor, L: Tensor, state: Tensor, fused_entropy: bool, tr_coeff: float = 0.0) -> Tensor:
    """Backward of the KL covariance projection given d loss / d Sigma_out [Bc, n, n] fp64 (symmetric); ``tr_coeff``:
    also add the gradient of tr_coeff * KL_cov(N(L L^T) || N(Sigma_out detached)) (trust-region regression loss)."""
    L = _chk(L)
    g = _chk(grad_sigma, torch.float64, "grad_sigma")
    if g.numel() != L.numel():
        raise TceError("grad_sigma must have the shape of L")
    out = torch.empty_like(L)
    _lib.call("tce_proj_kl_bwd_sigma", _p(L), _p(g), _p(state), int(fused_entropy), float(tr_coeff), _p(out),
              L.shape[0], L.shape[-1], _stream())
    return out


@proj_kl_bwd_sigma.register_fake
def _(grad_sigma, L, state, fused_entropy, tr_coeff=0.0):
    return torch.empty_like(L)


class _ProjKLEntropy(torch.autograd.Function):
    """-> (out_L, proj_L, info, Sigma0 [Bc,n,n] fp64 (a view of the state), alpha^2 [Bc]): the output covariance is
    alpha^2 * Sigma0.  Sigma0 is a DIFFERENTIABLE output: a consumer that works on the covariance (the segment
    likelihood) returns d loss / d (alpha^2 Sigma0) as its gradient and the backward then runs in covariance space
    (no Cholesky adjoint); gradients w.r.t. out_L take the factor path; both may arrive."""

    @staticmethod
    def forward(ctx, L, L_o, eps_cov, state, warm, beta, equality, split, holder):
        out, proj_L, info, out_inv = proj_kl_entropy_fwd(L, L_o, eps_cov, state, warm, beta, equality, split)
        sigma, scale = kl_state_sigma(state, L.shape[0], L.shape[-1])
        ctx.save_for_backward(L, proj_L)
        ctx.state = state
        ctx.holder, ctx.out_ptr = holder, out.data_ptr()
        ctx.generation = None
        if holder is not None:
            holder._kl_generation = getattr(holder, "_kl_generation", 0) + 1
            ctx.generation = holder._kl_generation
        ctx.mark_non_differentiable(proj_L, info, scale, out_inv)
        ctx.set_materialize_grads(False)
        return out, proj_L, info, sigma, scale, out_inv

    @staticmethod
    def backward(ctx, g, g_proj, g_info, g_sigma, g_scale, g_inv):
        L, proj_L = ctx.saved_tensors
        _check_generation(ctx)
        res = None
        # a trust-region loss whose covariance gradient was folded into this backward (rl.projection, fold=True)
        fold = float(getattr(ctx.holder, "_tr_fold", 0.0) or 0.0) if ctx.holder is not None else 0.0
        if ctx.holder is not None:
            ctx.holder._tr_fold = 0.0
        if g_sigma is not None:
            res = proj_kl_bwd_sigma(g_sigma.contiguous(), L, ctx.state, True, fold)
            fold = 0.0
        if g is None and fold != 0.0:
            g = torch.zeros_like(L)
        if g is not None and fold != 0.0:          # per-matrix (contextual) covariance: the fold rides on the factor path
            r2 = proj_kl_entropy_bwd_tr(g.contiguous(), L, proj_L, ctx.state, fold)
            return ((r2 if res is None else res + r2),) + (None,) * 8
        if g is not None:
            # somebody (the trust-region loss) may have inverted this call's output factor: (inverse, event, data_ptr)
            known = getattr(ctx.holder, "_output_inverse", None) if ctx.holder is not None else None
            inv = None
            if known is not None and known[2] == ctx.out_ptr and known[0].numel() == L.numel():
                torch.cuda.current_stream().wait_event(known[1])
                inv = known[0].reshape(L.shape)
            r2 = proj_kl_entropy_bwd(g.contiguous(), L, proj_L, ctx.state, inv)
            res = r2 if res is None else res + r2
        return (res,) + (None,) * 8


def proj_kl_entropy(L: Tensor, L_o: Tensor, eps_cov: float, state: Tensor, warm: bool, beta: Tensor,
                    equality: bool, split: bool = False, holder=None, return_sigma: bool = False):
    """``proj_entropy(proj_kl_cov(L, L_o, ...)[0], beta, equality)[0]`` as ONE forward and ONE backward kernel
    -> (out_L, proj_L before the entropy control [not differentiable], info [, Sigma0, alpha^2, out_L^-1 (split only)]).
    ``split``: the
    forward is two launches (state with Sigma_proj and alpha first, the Cholesky factor second) and
    ``SIGMA_READY[id(state)]`` holds an event recorded between them, for consumers of the covariance.  ``holder``:
    the owning layer: guards the state against a second forward before this call's backward, and its attribute
    ``_output_inverse = (inverse of out_L [.., n, n] fp64, CUDA event, out_L.data_ptr())`` -- if set by the time of the
    backward and matching this call -- saves the factor-path backward its own triangular inverse."""
    res = _ProjKLEntropy.apply(L, L_o, eps_cov, state, warm, beta, equality, split, holder)
    return res if return_sigma else res[:3]


def proj_kl_cov(L: Tensor, L_o: Tensor, eps_cov: float, state: Tensor, warm: bool, holder=None) -> Tuple[Tensor, Tensor]:
    """-> (proj_L [Bc,n,n], info [Bc]); ``state`` (``kl_state``) is overwritten with {M = L_o Q, lambda, eta, ...}:
    it feeds the backward and, with ``warm``, the next call with the same ``L_o`` starts its eigen-solve from it
    (2-3 Jacobi sweeps instead of ~9; guarded by a fingerprint of ``L_o`` inside the kernel)."""
    return _ProjKLCov.apply(L, L_o, eps_cov, state, warm, holder)


KL_DIAG_STATE = 4       # per matrix: eta, KL step active, alpha, entropy control active


@torch.library.custom_op("tce::proj_kl_diag", mutates_args=())
def proj_kl_diag(L: Tensor, L_o: Tensor, eps_cov: float, beta: Optional[Tensor],
                 equality: bool) -> Tuple[Tensor, Tensor, Tensor]:
    """KL covariance projection of DIAGONAL factors (std_only policy), closed form, optionally followed by the entropy
    control of ``proj_entropy`` (``beta`` [Bc] or [1] fp64; None = none).  L [Bc, n, n] and L_o [Bc or 1, n, n] are
    read on their diagonals only (any strides) -> (out [Bc, n, n] diagonal, state [Bc, 4] fp64, info [Bc] int32)."""
    ldb, inc = diag_strides(L)
    ldb_o, inc_o = diag_strides(L_o, "L_o")
    Bc, n = L.shape[0], L.shape[-1]
    if L_o.shape[0] not in (1, Bc) or L_o.shape[-1] != n:
        raise TceError("L_o must be [Bc, n, n] or [1, n, n]")
    out, ldb_out, inc_out = _dense_diag_grad(L)
    state = torch.empty(Bc, KL_DIAG_STATE, device=L.device, dtype=torch.float64)
    info = torch.empty(Bc, device=L.device, dtype=torch.int32)
    if beta is not None:
        beta = _chk(beta, torch.float64, "beta")
    _lib.call("tce_proj_kl_diag_fwd", _p(L), ldb, inc, _p(L_o), ldb_o, inc_o, float(eps_cov), _p(beta),
              0 if beta is None or beta.numel() == 1 else 1, int(equality), _p(out), ldb_out, inc_out, _p(state),
              _p(info), Bc, n, _stream())
    return out, state, info


@proj_kl_diag.register_fake
def _(L, L_o, eps_cov, beta, equality):
    Bc = L.shape[0]
    return (L.new_empty(Bc, L.shape[-1], L.shape[-1]), L.new_empty(Bc, KL_DIAG_STATE, dtype=torch.float64),
            L.new_empty(Bc, dtype=torch.int32))


@torch.library.custom_op("tce::proj_kl_diag_bwd", mutates_args=())
def proj_kl_diag_bwd(grad_out: Tensor, L: Tensor, L_o: Tensor, state: Tensor) -> Tensor:
    """d loss / d L [Bc, n, n] (diagonal) from d loss / d out; L_o is a constant."""
    ldb, inc = diag_strides(L)
    ldb_o, inc_o = diag_strides(L_o, "L_o")
    ldb_g, inc_g = diag_strides(grad_out, "grad_out")
    state = _chk(state, torch.float64, "state")
    g, ldb_gs, inc_gs = _dense_diag_grad(L)
    _lib.call("tce_proj_kl_diag_bwd", _p(L), ldb, inc, _p(L_o), ldb_o, inc_o, _p(state), _p(grad_out), ldb_g, inc_g,
              _p(g), ldb_gs, inc_gs, L.shape[0], L.shape[-1], _stream())
    return g


@proj_kl_diag_bwd.register_fake
def _(grad_out, L, L_o, state):
    return L.new_empty(L.shape[0], L.shape[-1], L.shape[-1])


def _pkd_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0], inputs[1], output[1])
    ctx.set_materialize_grads(False)


def _pkd_backward(ctx, g, g_state, g_info):
    if g is None:
        return None, None, None, None, None
    L, L_o, state = ctx.saved_tensors
    return proj_kl_diag_bwd(g, L, L_o, state), None, None, None, None


proj_kl_diag.register_autograd(_pkd_backward, setup_context=_pkd_setup)


@torch.library.custom_op("tce::proj_frob_cov", mutates_args=())
def proj_frob_cov(L: Tensor, L_o: Tensor, eps_cov: float) -> Tuple[Tensor, Tensor, Tensor]:
    L = _chk(L, name="L")
    L_o, ldbo = _batched_matrix(L_o, "L_o")
    Bc, n = L.shape[0], L.shape[-1]
    out = torch.empty_like(L)
    sc = torch.empty(Bc, 4, device=L.device, dtype=torch.float64)
    info = torch.empty(Bc, device=L.device, dtype=torch.int32)
    _lib.call("tce_proj_frob_cov_fwd", _p(L), _p(L_o), ldbo, float(eps_cov), _p(out), _p(sc), _p(info), Bc, n, _stream())
    return out, sc, info


@proj_frob_cov.register_fake
def _(L, L_o, eps_cov):
    return torch.empty_like(L), L.new_empty(L.shape[0], 4, dtype=torch.float64), L.new_empty(L.shape[0], dtype=torch.int32)


@torch.library.custom_op("tce::proj_frob_cov_bwd", mutates_args=())
def proj_frob_cov_bwd(grad_out: Tensor, L: Tensor, L_o: Tensor, proj_L: Tensor, sc: Tensor, eps_cov: float) -> Tensor:
    g, L, proj_L = _chk(grad_out), _chk(L), _chk(proj_L)
    L_o, ldbo = _batched_matrix(L_o, "L_o")
    out = torch.empty_like(L)
    _lib.call("tce_proj_frob_cov_bwd", _p(L), _p(L_o), ldbo, float(eps_cov), _p(proj_L), _p(g), _p(sc), _p(out),
              L.shape[0], L.shape[-1], _stream())
    return out


@proj_frob_cov_bwd.register_fake
def _(grad_out, L, L_o, proj_L, sc, eps_cov):
    return torch.empty_like(L)


def _pf_setup(ctx, inputs, output):
    L, L_o, eps_cov = inputs
    ctx.save_for_backward(L, L_o, output[0], output[1])
    ctx.eps_cov = eps_cov


def _pf_backward(ctx, g, g_sc, g_info):
    L, L_o, proj_L, sc = ctx.saved_tensors
    return proj_frob_cov_bwd(g, L, L_o, proj_L, sc, ctx.eps_cov), None, None


proj_frob_cov.register_autograd(_pf_backward, setup_context=_pf_setup)


@torch.library.custom_op("tce::proj_w2_cov", mutates_args=())
def proj_w2_cov(L: Tensor, L_o: Tensor, eps_cov: float, scale_prec: bool) -> Tuple[Tensor, Tensor]:
    L = _chk(L, name="L")
    L_o, ldbo = _batched_matrix(L_o, "L_o")
    Bc, n = L.shape[0], L.shape[-1]
    out = torch.empty_like(L)
    sc = torch.empty(Bc, 4, device=L.device, dtype=torch.float64)
    _lib.call("tce_proj_w2_cov_fwd", _p(L), _p(L_o), ldbo, float(eps_cov), int(scale_prec), _p(out), _p(sc), Bc, n,
              _stream())
    return out, sc


@proj_w2_cov.register_fake
def _(L, L_o, eps_cov, scale_prec):
    return torch.empty_like(L), L.new_empty(L.shape[0], 4, dtype=torch.float64)


@torch.library.custom_op("tce::proj_w2_cov_bwd", mutates_args=())
def proj_w2_cov_bwd(grad_out: Tensor, L: Tensor, L_o: Tensor, eps_cov: float, scale_prec: bool) -> Tensor:
    g, L = _chk(grad_out), _chk(L)
    L_o, ldbo = _batched_matrix(L_o, "L_o")
    out = torch.empty_like(L)
    _lib.call("tce_proj_w2_cov_bwd", _p(L), _p(L_o), ldbo, float(eps_cov), int(scale_prec), _p(g), _p(out), L.shape[0],
              L.shape[-1], _stream())
    return out


@proj_w2_cov_bwd.register_fake
def _(grad_out, L, L_o, eps_cov, scale_prec):
    return torch.empty_like(L)


def _pw_setup(ctx, inputs, output):
    L, L_o, eps_cov, scale_prec = inputs
    ctx.save_for_backward(L, L_o)
    ctx.eps_cov, ctx.scale_prec = eps_cov, scale_prec


def _pw_backward(ctx, g, g_sc):
    L, L_o = ctx.saved_tensors
    return proj_w2_cov_bwd(g, L, L_o, ctx.eps_cov, ctx.scale_prec), None, None, None


proj_w2_cov.register_autograd(_pw_backward, setup_context=_pw_setup)


@torch.library.custom_op("tce::cov_distance", mutates_args=())
def cov_distance(kind: int, L: Tensor, L_o: Tensor, scale_prec: bool) -> Tensor:
    """Frobenius (kind 0) / commutative W2 (kind 1) covariance distance [Bc] fp64, differentiable w.r.t. L."""
    L = _chk(L, name="L")
    L_o, ldbo = _batched_matrix(L_o, "L_o")
    val = torch.empty(L.shape[0], device=L.device, dtype=torch.float64)
    _lib.call("tce_cov_distance", int(kind), _p(L), _p(L_o), ldbo, int(scale_prec), None, _p(val), None, L.shape[0],
              L.shape[-1], _stream())
    return val


@cov_distance.register_fake
def _(kind, L, L_o, scale_prec):
    return L.new_empty(L.shape[0], dtype=torch.float64)


@torch.library.custom_op("tce::cov_distance_bwd", mutates_args=())
def cov_distance_bwd(grad_val: Tensor, kind: int, L: Tensor, L_o: Tensor, scale_prec: bool) -> Tensor:
    L = _chk(L)
    g = _chk(grad_val, torch.float64)
    L_o, ldbo = _batched_matrix(L_o, "L_o")
    out = torch.empty_like(L)
    _lib.call("tce_cov_distance", int(kind), _p(L), _p(L_o), ldbo, int(scale_prec), _p(g), None, _p(out), L.shape[0],
              L.shape[-1], _stream())
    return out


@cov_distance_bwd.register_fake
def _(grad_val, kind, L, L_o, scale_prec):
    return torch.empty_like(L)


def _cd_setup(ctx, inputs, output):
    kind, L, L_o, scale_prec = inputs
    ctx.save_for_backward(L, L_o)
    ctx.kind, ctx.scale_prec = kind, scale_prec


def _cd_backward(ctx, g):
    L, L_o = ctx.saved_tensors
    return None, cov_distance_bwd(g.contiguous(), ctx.kind, L, L_o, ctx.scale_prec), None, None


cov_distance.register_autograd(_cd_backward, setup_context=_cd_setup)


# --------------------------------------------------------------------------------------------------
# (3) product path of the segment likelihood: fused kernels
# --------------------------------------------------------------------------------------------------
from .ops_seglik import (seg_logprob, seg_surrogate, seglik, pairs_chained, times_uniform, declare_uniform,  # noqa: E402,F401
                         shared_factor, seg_logprob_diag)

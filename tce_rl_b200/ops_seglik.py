"""Segment-wise trajectory likelihood on the fused kernels (``csrc/tce_seglik_fused.cu``).

Reference: ``TemporalCorrelatedPolicy.log_prob`` (mprl/rl/policy/temporal_correlated_policy.py:104-203) and
``TemporalCorrelatedAgent.surrogate_loss`` (mprl/rl/agent/temporal_correlated_agent.py:718-739).

Two device paths, same results:
* general  : ``tce_seglik_diagmax`` (regulariser pre-pass) -> [all-reduce(MAX)] -> ``tce_seglik_fused`` (one persistent
             kernel, forward + backward, no HBM workspace) -> ``tce_seglik_dsigma_reduce`` (shared covariance only);
* uniform  : every episode has the same time grid and the covariance is shared (all shipped TCE configs):
             ``tce_seglik_uniform_prep / _main / _finish`` + ``tce_seglik_dsigma_reduce``.
A segment count that neither takes (P > 256, or no episode group of the fused kernel fits in shared memory) runs the
staged kernels of ``csrc/tce_seglik.cu``, as every shape without specialised kernels does.

The gradient of the fused surrogate is produced in the FORWARD call (the upstream gradient of a scalar loss is known:
``-ratio * adv / (B P)``); the autograd backward only scales it.
"""
from __future__ import annotations

import ctypes as C
import warnings
import weakref
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import TceError

Tensor = torch.Tensor

# torch.distributed group over which the batch-global regulariser seed is MAX-reduced (None: single GPU)
_REG_GROUP = None
# True: every rank is known to hold the SAME time grid for all its episodes (``sync_uniform``).  With a shared
# covariance the gram matrices -- and hence the regulariser seed -- are then identical on all ranks by construction
# and the uniform path skips the all-reduce(MAX).
_GLOBAL_UNIFORM = False


def set_regulariser_group(group) -> None:
    """At >1 GPU, all-reduce(MAX) the batch-global regulariser seed over ``group`` (SURVEY 8(e)); ``True`` = the
    default group, ``None`` = no reduction."""
    global _REG_GROUP, _GLOBAL_UNIFORM
    _REG_GROUP = group
    _GLOBAL_UNIFORM = False


def sync_uniform(init_time: Tensor, times: Tensor) -> bool:
    """Collective (call on every rank of the regulariser group, outside graph capture): do ALL ranks hold one and the
    same time grid?  One all-reduce of four floats per dataset; the answer lets the uniform likelihood path drop its
    per-epoch all-reduce(MAX) (see ``_GLOBAL_UNIFORM``).  Returns the answer and remembers it."""
    global _GLOBAL_UNIFORM
    _GLOBAL_UNIFORM = False
    if _REG_GROUP is None:
        return False
    import torch.distributed as dist
    group = None if _REG_GROUP is True else _REG_GROUP
    local = times.shape[0] > 0 and times_uniform(init_time, times)
    if times.shape[0] > 0:
        row, t0 = times[0].double(), init_time[0].double().reshape(1)
        sig = torch.cat([t0, row.sum().reshape(1), (row * torch.arange(1, row.numel() + 1, device=row.device)).sum()
                         .reshape(1), torch.full((1,), float(local), device=row.device, dtype=torch.float64)])
    else:                                                # an empty shard constrains nothing
        sig = None
    big = 1e300
    lo = sig.clone() if sig is not None else torch.full((4,), big, device=times.device, dtype=torch.float64)
    hi = sig.clone() if sig is not None else torch.full((4,), -big, device=times.device, dtype=torch.float64)
    dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=group)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=group)
    _GLOBAL_UNIFORM = bool(torch.equal(lo, hi) and lo[3].item() == 1.0)
    return _GLOBAL_UNIFORM


def _reduce_diag_max(diag_max: Tensor) -> None:
    if _REG_GROUP is not None:
        import torch.distributed as dist
        dist.all_reduce(diag_max, op=dist.ReduceOp.MAX, group=None if _REG_GROUP is True else _REG_GROUP)


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


# ---- host-side facts about index / time tensors (one device read per tensor VERSION, cached by identity) ---------
class _IdCache:
    """tensor -> value, keyed by identity (tensors compare elementwise, so they cannot key a WeakKeyDictionary);
    entries die with their tensor."""

    def __init__(self):
        self._d = {}

    def get(self, t: Tensor):
        ent = self._d.get(id(t))
        return ent[1] if ent is not None and ent[0]() is t else None

    def put(self, t: Tensor, value) -> None:
        key = id(t)
        self._d[key] = (weakref.ref(t, lambda _r, k=key, d=self._d: d.pop(k, None)), value)


_PAIR_FACTS = _IdCache()
_TIME_FACTS = _IdCache()


def pairs_chained(pred_pairs: Tensor) -> bool:
    """pred_pairs[p][1] == pred_pairs[p+1][0] for every p (the fixed-interval selection, util_learning.py:107-150).
    The pairs are created on the host; a device copy is read back once (outside any graph capture)."""
    key = _PAIR_FACTS.get(pred_pairs)
    if key is not None and key[0] == pred_pairs._version:
        return key[1]
    if pred_pairs.is_cuda and torch.cuda.is_current_stream_capturing():
        return False                                     # cannot read back under capture: the safe, general layout
    pp = pred_pairs.detach().cpu()
    res = bool(pp.shape[0] >= 1 and (pp.shape[0] == 1 or bool((pp[:-1, 1] == pp[1:, 0]).all())))
    _PAIR_FACTS.put(pred_pairs, (pred_pairs._version, res))
    return res


_WARNED_CAPTURE = False


def times_uniform(init_time: Tensor, times: Tensor) -> bool:
    """Every episode has the same time grid (same init_time, same row of ``times``).  One device reduction + host read
    per tensor version; under graph capture an unknown tensor counts as non-uniform."""
    sig = (times._version, init_time.data_ptr(), init_time._version)
    key = _TIME_FACTS.get(times)
    if key is not None and key[0] == sig:
        return key[1]
    if times.is_cuda and torch.cuda.is_current_stream_capturing():
        global _WARNED_CAPTURE
        if not _WARNED_CAPTURE:                      # (a captured epoch keeps whatever path it was captured with)
            _WARNED_CAPTURE = True
            warnings.warn("tce_rl_b200: time grid of a dataset first seen during CUDA-graph capture -- the capture cannot "
                          "read the device, so the general-grid likelihood is recorded (slower than the common-grid "
                          "path); run one eager epoch on these tensors first or call ops_seglik.declare_uniform")
        return False
    res = bool(times.shape[0] >= 1 and bool(((times == times[:1]).all() & (init_time == init_time[:1]).all()).item()))
    _TIME_FACTS.put(times, (sig, res))
    return res


def declare_uniform(init_time: Tensor, times: Tensor, value: bool) -> None:
    """Record the answer of ``times_uniform`` for these tensors (e.g. decided on the host copy of a dataset)."""
    _TIME_FACTS.put(times, ((times._version, init_time.data_ptr(), init_time._version), bool(value)))


def shared_factor(L: Tensor, batch: int) -> Optional[Tensor]:
    """The ONE [1, n, n] matrix behind ``L`` if it is shared by the batch ([1, n, n], or a stride-0 expand of a
    [1, n, n] / [n, n] tensor), else None.  For an expand view the BASE tensor is returned so that autograd sends the
    (already batch-summed) gradient straight to it -- no [B, n, n] gradient is ever materialised."""
    n = L.shape[-1]
    if L.dim() == 2:
        return L.reshape(1, n, n)
    if L.dim() != 3:
        return None
    if L.shape[0] == 1:
        return L if L.is_contiguous() else L.contiguous()
    if L.stride(0) == 0 and L.stride(1) == n and L.stride(2) == 1:
        first = getattr(L, "_tce_first", None)
        if first is not None:
            return first
        base = L._base
        if base is not None and base.numel() == n * n and base.shape[-2:] == (n, n) and base.is_contiguous() \
                and base.data_ptr() == L.data_ptr():
            return base.reshape(1, n, n)
        return L[:1]
    return None


def compiled(tables: int) -> bool:
    """True for the five (num_dof, K1) shapes with specialised kernels (fused and uniform-grid paths), False for every
    other supported shape, which runs the staged kernels (``tce_seglik_compiled``: one host query, no launch; NOT
    cached by handle, see ``fused_config``).  Shapes outside the supported set fail in the kernels' entry points."""
    return _lib.load().tce_seglik_compiled(tables) == 1


def uniform_config(tables: int, B: int, P: int) -> dict:
    """Buffer sizes of the uniform-grid path; ``uni_parts`` = 0: its kernels do not take this P."""
    lib = _lib.load()
    nparts, apart = C.c_int32(), C.c_int64()
    rc = lib.tce_seglik_uniform_parts(tables, max(B, 1), P, C.byref(nparts), C.byref(apart))
    return {"ws_doubles": lib.tce_seglik_uniform_ws_doubles(tables, P),
            "uni_parts": nparts.value if rc == 0 else 0, "apart_doubles": apart.value if rc == 0 else 0}


def fused_config(tables: int, B: int, P: int, chained: bool) -> dict:
    """Launch geometry / buffer sizes of the fused path for these shapes (host integers; NOT cached by handle: a
    freed tables handle can be re-issued for another MP shape), and those of ``uniform_config``.  Raises
    ``TceError`` when the fused kernel does not take P (P > 256, or no episode group fits in shared memory)."""
    lib = _lib.load()
    E, grid, part, pre = C.c_int32(), C.c_int32(), C.c_int64(), C.c_int64()
    _lib.check(lib.tce_seglik_fused_config(tables, max(B, 1), P, int(chained), C.byref(E), C.byref(grid),
                                           C.byref(part), C.byref(pre)), "tce_seglik_fused_config")
    return {"E": E.value, "grid": grid.value, "part_floats": part.value, "pre_doubles": pre.value,
            **uniform_config(tables, B, P)}


@torch.library.custom_op("tce::seglik", mutates_args=())
def seglik(smp_traj: Tensor, mean: Tensor, L: Optional[Tensor], sigma: Optional[Tensor],
           sigma_scale: Optional[Tensor], times: Tensor, init_time: Tensor, init_pos: Tensor, init_vel: Tensor,
           pred_pairs: Tensor, tables: int, reg_rel: float, grad_mode: int, grad_logp: Optional[Tensor],
           logp_old: Optional[Tensor], advantage: Optional[Tensor], chained: bool, uniform: bool,
           want_grad_L: bool, want_grad_sigma: bool = False) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """The whole likelihood in one op.

    ``L``: [B, n, n] per-episode factors or [1, n, n] = one shared factor; ``sigma`` (+ optional ``sigma_scale`` [1]):
    the shared covariance itself as fp64 [n, n] (then ``L`` is only used for grad_L = 2 tril(dSigma L)).
    grad_mode 0: log-probs; 1: backward for ``grad_logp``; 2: fused surrogate with ``logp_old`` / ``advantage``.
    -> (logp [B,P], info [B,P] int32, acc [3] fp64 {regulariser seed max diag C, -mean(ratio adv), mean ratio},
        grad_mean [B,Dp] or empty, grad_L [B or 1, Dp, Dp] or empty,
        grad_sigma [Dp, Dp] fp64 = d loss / d (sigma_scale * sigma) (shared covariance, ``want_grad_sigma``) or empty)
    """
    smp_traj, mean, times = _chk(smp_traj, name="smp_traj"), _chk(mean, name="mean"), _chk(times, name="times")
    init_time, init_pos, init_vel = _chk(init_time), _chk(init_pos), _chk(init_vel)
    pairs = _chk(pred_pairs, torch.int64, "pred_pairs")
    B, T = times.shape
    P, Dp = pairs.shape[0], mean.shape[-1]
    dev = mean.device
    if L is None and sigma is None:
        raise TceError("either L or sigma is required")
    if L is not None:
        L = _chk(L, name="L")
        if L.dim() != 3 or L.shape[0] not in (1, B):
            raise TceError("L must be [B, n, n] or [1, n, n]")
    shared = sigma is not None or L.shape[0] == 1
    ldb = 0 if shared else Dp * Dp
    if sigma is not None:
        if sigma.dtype != torch.float64 or not sigma.is_cuda or not sigma.is_contiguous() or sigma.numel() != Dp * Dp:
            raise TceError("sigma must be a contiguous CUDA float64 [Dp, Dp] tensor")
    if uniform and not shared:
        raise TceError("the uniform path needs a shared covariance")
    logp = torch.empty(B, P, device=dev, dtype=torch.float32)
    info = torch.empty(B, P, device=dev, dtype=torch.int32)
    acc = torch.zeros(3, device=dev, dtype=torch.float64)       # {diag_max, loss, ratio}
    diag_max, stats = acc[:1], acc[1:]                          # (views for the kernels; the op returns acc)
    want = grad_mode != 0
    g_mean = torch.empty(B, Dp, device=dev, dtype=torch.float32) if want else mean.new_empty(0)
    need_L = want and want_grad_L
    need_S = want and want_grad_sigma
    if need_S and not shared:
        raise TceError("grad_sigma exists for a shared covariance only")
    g_L = mean.new_empty(0)
    g_S = mean.new_empty(0, dtype=torch.float64)
    if B == 0:
        if need_L:
            g_L = torch.zeros(1 if shared else 0, Dp, Dp, device=dev, dtype=torch.float32)
        if need_S:
            g_S = torch.zeros(Dp, Dp, device=dev, dtype=torch.float64)
        return logp, info, acc, g_mean, g_L, g_S
    if need_L and shared and L is None:
        raise TceError("grad_L of a shared covariance needs its factor L")
    cfg = None
    if compiled(tables):
        if uniform:
            cfg = uniform_config(tables, B, P)
            uniform = cfg["uni_parts"] > 0                   # P outside the uniform kernels: general path
        if not uniform:
            try:
                cfg = fused_config(tables, B, P, chained)
            except TceError:                                 # P outside the fused kernel: staged kernels
                cfg = None
    if cfg is None:
        g_L, g_S = _seglik_staged(smp_traj, mean, L, sigma, sigma_scale, times, init_time, init_pos, init_vel, pairs,
                                  tables, reg_rel, grad_mode, grad_logp, logp_old, advantage, shared, need_L, need_S,
                                  logp, info, acc, g_mean)
        return logp, info, acc, g_mean, g_L, g_S
    st = _stream()
    scale = 1.0 / (B * P)
    if uniform:
        ws = torch.empty(cfg["ws_doubles"], device=dev, dtype=torch.float64)
        Lp = None if sigma is not None else _p(L)
        if _REG_GROUP is None or (_GLOBAL_UNIFORM and shared):
            _lib.call("tce_seglik_uniform_prep", tables, Lp, _p(sigma), _p(sigma_scale), _p(times), _p(init_time),
                      _p(pairs), _p(ws), _p(diag_max), float(reg_rel), 3, P, st)
        else:
            _lib.call("tce_seglik_uniform_prep", tables, Lp, _p(sigma), _p(sigma_scale), _p(times), _p(init_time),
                      _p(pairs), _p(ws), _p(diag_max), float(reg_rel), 1, P, st)
            _reduce_diag_max(diag_max)
            _lib.call("tce_seglik_uniform_prep", tables, Lp, _p(sigma), _p(sigma_scale), _p(times), _p(init_time),
                      _p(pairs), _p(ws), _p(diag_max), float(reg_rel), 2, P, st)
        apart = torch.empty(cfg["apart_doubles"], device=dev, dtype=torch.float64) if (need_L or need_S) else None
        _lib.call("tce_seglik_uniform_main", tables, _p(ws), _p(smp_traj), _p(mean), _p(init_pos), _p(init_vel),
                  _p(pairs), int(grad_mode), _p(grad_logp), _p(logp_old), _p(advantage), scale, _p(stats), _p(logp),
                  _p(info), _p(g_mean) if want else None, _p(apart), B, T, P, st)
        if need_L or need_S:
            if need_L:
                g_L = torch.empty(1, Dp, Dp, device=dev, dtype=torch.float32)
            if need_S:
                g_S = torch.empty(Dp, Dp, device=dev, dtype=torch.float64)
            _lib.call("tce_seglik_uniform_finish", tables, _p(ws), _p(apart), cfg["uni_parts"],
                      _p(L) if need_L else None, None, _p(g_L) if need_L else None, _p(g_S) if need_S else None, P, st)
        return logp, info, acc, g_mean, g_L, g_S
    pre = torch.empty(B * cfg["pre_doubles"], device=dev, dtype=torch.float64)
    _lib.call("tce_seglik_prepass", tables, _p(smp_traj), _p(mean), None if sigma is not None else _p(L), ldb,
              _p(sigma), _p(sigma_scale), _p(times), _p(init_time), _p(init_pos), _p(init_vel), _p(pairs), _p(pre),
              _p(diag_max), int(chained), B, T, P, st)
    _reduce_diag_max(diag_max)
    part = None
    if need_L or need_S:
        if shared:
            part = torch.empty(cfg["part_floats"], device=dev, dtype=torch.float32)
        else:
            g_L = torch.empty(B, Dp, Dp, device=dev, dtype=torch.float32)
    _lib.call("tce_seglik_fused", tables, _p(pre), None if sigma is not None else _p(L), ldb, _p(sigma),
              _p(sigma_scale), _p(pairs), _p(diag_max), float(reg_rel), int(grad_mode), _p(grad_logp), _p(logp_old),
              _p(advantage), scale, _p(stats), _p(logp), _p(info), _p(g_mean) if want else None,
              _p(g_L) if (need_L and not shared) else None, _p(part), int(chained), B, P, st)
    if (need_L or need_S) and shared:
        if need_L:
            g_L = torch.empty(1, Dp, Dp, device=dev, dtype=torch.float32)
        if need_S:
            g_S = torch.empty(Dp, Dp, device=dev, dtype=torch.float64)
        _lib.call("tce_seglik_dsigma_reduce", tables, _p(part), cfg["grid"], _p(L) if need_L else None, None,
                  _p(g_L) if need_L else None, _p(g_S) if need_S else None, st)
    return logp, info, acc, g_mean, g_L, g_S


def _seglik_staged(smp_traj, mean, L, sigma, sigma_scale, times, init_time, init_pos, init_vel, pairs, tables, reg_rel,
                   grad_mode, grad_logp, logp_old, advantage, shared, need_L, need_S, logp, info, acc, g_mean):
    """``seglik`` on the staged kernels (shapes without fused / uniform-grid kernels, and segment counts that neither
    takes on the shapes with them, e.g. P > 256 segments): gram -> [all-reduce(MAX) of the
    regulariser seed] -> per-segment Cholesky (+ surrogate) -> backward.  A shared covariance sums its gradient over the
    batch in a fixed order (``tce_seglik_bwd_shared``).  Fills logp / info / acc / g_mean, returns (g_L, g_S)."""
    lib = _lib.load()
    B, T = times.shape
    P, Dp = pairs.shape[0], mean.shape[-1]
    dev = mean.device
    diag_max, stats = acc[:1], acc[1:]
    st = _stream()
    work = torch.empty(max(lib.tce_seglik_work_bytes(tables, B, P) // 8, 1), device=dev, dtype=torch.float64)
    if sigma is not None:
        _lib.call("tce_seglik_gram_sigma", tables, _p(smp_traj), _p(mean), _p(sigma), _p(sigma_scale), _p(times),
                  _p(init_time), _p(init_pos), _p(init_vel), _p(pairs), _p(work), _p(diag_max), B, T, P, st)
    else:
        _lib.call("tce_seglik_gram", tables, _p(smp_traj), _p(mean), _p(L), 0 if shared else Dp * Dp, _p(times),
                  _p(init_time), _p(init_pos), _p(init_vel), _p(pairs), _p(work), _p(diag_max), B, T, P, st)
    _reduce_diag_max(diag_max)
    want = grad_mode != 0
    _lib.call("tce_seglik_chol", tables, _p(work), _p(work) if want else None, _p(diag_max), float(reg_rel),
              _p(grad_logp) if grad_mode == 1 else None, _p(logp_old) if grad_mode == 2 else None,
              _p(advantage) if grad_mode == 2 else None, 1.0 / (B * P), _p(stats) if grad_mode == 2 else None,
              _p(logp), _p(info), B, P, st)
    g_L = mean.new_empty(0)
    g_S = mean.new_empty(0, dtype=torch.float64)
    if not want:
        return g_L, g_S
    if not shared:
        if need_L:
            g_L = torch.empty(B, Dp, Dp, device=dev, dtype=torch.float32)
        _lib.call("tce_seglik_bwd", tables, _p(work), _p(L), Dp * Dp, _p(times), _p(init_time), _p(pairs), None,
                  _p(g_mean), _p(g_L) if need_L else None, B, T, P, st)
        return g_L, g_S
    if need_L:
        g_L = torch.empty(1, Dp, Dp, device=dev, dtype=torch.float32)
    # the covariance gradient is formed even when only grad_mean is wanted: the shared backward needs a destination
    sig_out = torch.empty(Dp, Dp, device=dev, dtype=torch.float64) if (need_S or not need_L) else None
    part = torch.empty(lib.tce_seglik_shared_part_doubles(tables, B), device=dev, dtype=torch.float64)
    _lib.call("tce_seglik_bwd_shared", tables, _p(work), _p(L) if need_L else None, _p(times), _p(init_time),
              _p(pairs), None, _p(g_mean), _p(part), _p(g_L) if need_L else None, _p(sig_out), B, T, P, st)
    if need_S:
        g_S = sig_out
    return g_L, g_S


@seglik.register_fake
def _(smp_traj, mean, L, sigma, sigma_scale, times, init_time, init_pos, init_vel, pred_pairs, tables, reg_rel,
      grad_mode, grad_logp, logp_old, advantage, chained, uniform, want_grad_L, want_grad_sigma=False):
    B, P, Dp = times.shape[0], pred_pairs.shape[0], mean.shape[-1]
    shared = sigma is not None or L.shape[0] == 1
    want = grad_mode != 0
    return (mean.new_empty(B, P), mean.new_empty(B, P, dtype=torch.int32), mean.new_empty(3, dtype=torch.float64),
            mean.new_empty(B, Dp) if want else mean.new_empty(0),
            mean.new_empty(1 if shared else B, Dp, Dp) if (want and want_grad_L) else mean.new_empty(0),
            mean.new_empty(Dp, Dp, dtype=torch.float64) if (want and want_grad_sigma) else
            mean.new_empty(0, dtype=torch.float64))


def _resolve(L: Tensor, B: int, sigma):
    """-> (L as [B,n,n] or [1,n,n] connected to the autograd graph, shared?)"""
    first = shared_factor(L, B)
    if first is not None:
        return first, True
    if sigma is not None:
        raise TceError("sigma describes ONE covariance: pass the shared factor with it")
    return L, False


class _SegLogProb(torch.autograd.Function):
    """log-probs [B, P]; the backward re-runs the fused kernel with the upstream gradient (no saved workspace)."""

    @staticmethod
    def forward(ctx, smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs, tables, reg_rel, chained,
                uniform, sigma, sigma_scale):
        logp, info, acc, _, _, _ = seglik(smp_traj, mean, L, sigma, sigma_scale, times, init_time, init_pos, init_vel,
                                          pred_pairs, tables, reg_rel, 0, None, None, None, chained, uniform, False)
        diag_max = acc[:1]
        ctx.save_for_backward(smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs)
        ctx.sig = (sigma, sigma_scale)
        ctx.args = (tables, reg_rel, chained, uniform)
        ctx.mark_non_differentiable(info, diag_max)
        ctx.set_materialize_grads(False)
        return logp, info, diag_max

    @staticmethod
    def backward(ctx, g_logp, g_info, g_diag):
        if g_logp is None:
            return (None,) * 14
        smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs = ctx.saved_tensors
        tables, reg_rel, chained, uniform = ctx.args
        need_S = ctx.sig[0] is not None and ctx.needs_input_grad[12]      # the gradient flows through Sigma when it can
        need_L = ctx.needs_input_grad[2] and not need_S
        _, _, _, g_mean, g_L, g_S = seglik(smp_traj, mean, L, ctx.sig[0], ctx.sig[1], times, init_time, init_pos,
                                           init_vel, pred_pairs, tables, reg_rel, 1, g_logp.contiguous(), None, None,
                                           chained, uniform, need_L, need_S)
        return (None, g_mean if ctx.needs_input_grad[1] else None, g_L if need_L else None) + (None,) * 9 + (
            g_S.view_as(ctx.sig[0]) if need_S else None, None)


_UNIT = {}


def unit_seed(device, dtype) -> Tensor:
    """A cached 0-dim 1.0: pass it as the gradient of a loss term to ``torch.autograd.backward`` -- the likelihood
    ops recognise it (by identity) and skip the scaling kernels of their backward."""
    key = (str(device), dtype)
    if key not in _UNIT:
        _UNIT[key] = torch.ones((), device=device, dtype=dtype)
    return _UNIT[key]


class _SegSurrogate(torch.autograd.Function):
    """(surrogate loss, mean ratio, logp); the gradients w.r.t. mean / L are formed by the forward call."""

    @staticmethod
    def forward(ctx, smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs, logp_old, advantage, tables,
                reg_rel, chained, uniform, sigma, sigma_scale):
        need_S = sigma is not None and bool(ctx.needs_input_grad[14])     # the gradient flows through Sigma when it can
        need_L = bool(ctx.needs_input_grad[2]) and not need_S
        logp, info, acc, g_mean, g_L, g_S = seglik(smp_traj, mean, L, sigma, sigma_scale, times, init_time, init_pos,
                                                   init_vel, pred_pairs, tables, reg_rel, 2, None, logp_old, advantage,
                                                   chained, uniform, need_L, need_S)
        s32 = acc[1:].to(torch.float32)
        ctx.save_for_backward(g_mean, g_L, g_S.view_as(sigma) if need_S else g_S)
        ctx.need_L, ctx.need_S = need_L, need_S
        ctx.mark_non_differentiable(logp, info)
        ctx.set_materialize_grads(False)
        return s32[0], s32[1], logp, info

    @staticmethod
    def backward(ctx, g_loss, g_ratio, g_logp, g_info):
        if g_loss is None:
            return (None,) * 16
        g_mean, g_L, g_S = ctx.saved_tensors
        if g_loss is not unit_seed(g_loss.device, g_loss.dtype):
            g_mean = g_mean * g_loss
            g_L = g_L * g_loss if ctx.need_L else g_L
            g_S = g_S * g_loss if ctx.need_S else g_S
        return (None, g_mean if ctx.needs_input_grad[1] else None, g_L if ctx.need_L else None) + (None,) * 11 + (
            g_S if ctx.need_S else None, None)


def _facts(pred_pairs, init_time, times, shared, uniform):
    chained = pairs_chained(pred_pairs)
    if uniform is None:
        uniform = shared and times_uniform(init_time, times)
    return chained, bool(uniform and shared)


# Per-episode covariance factors (contextual layout): measured on B200 the staged kernels (4 CTAs per SM, fp64
# workspace in HBM) beat the one-CTA-per-SM fused kernel, whose register-resident design pays off only when the
# covariance -- and with a uniform time grid the factorisations -- are shared: B = 1024 x 24: 146 vs 248 us forward +
# backward, B = 16384: 1.60 vs 2.75 ms (scripts/perf_seglik.py).  False = fused kernel for every layout.
PER_EPISODE_STAGED = True


def seg_logprob(smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs, tables, reg_rel: float = 1e-4,
                return_info: bool = False, uniform: Optional[bool] = None, sigma=None):
    """Segment-wise log-likelihood [B, P], differentiable w.r.t. ``mean`` and ``L``.  ``uniform``: None = decide from
    the data (one cached device read), True / False = the caller knows.  ``sigma`` = (Sigma0 [n,n] fp64, scale [1])."""
    Lr, shared = _resolve(L, times.shape[0], sigma)
    if not shared and PER_EPISODE_STAGED and times.shape[0] > 0:
        from . import ops
        return ops.seg_logprob_staged(smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs, tables,
                                      reg_rel, return_info)
    chained, uni = _facts(pred_pairs, init_time, times, shared, uniform)
    logp, info, diag_max = _SegLogProb.apply(smp_traj, mean, Lr, times, init_time, init_pos, init_vel, pred_pairs,
                                             tables.handle, float(reg_rel), chained, uni,
                                             None if sigma is None else sigma[0], None if sigma is None else sigma[1])
    return (logp, info, diag_max) if return_info else logp


def diag_strides(L: Tensor, name: str = "L") -> Tuple[int, int]:
    """(ldb, inc) of the diagonals of a [B, n, n] float32 CUDA factor as a strided vector: element i of episode b is
    at ``data_ptr + b * ldb + i * inc`` (any strides; a single matrix or a stride-0 batch expand gives ldb = 0)."""
    if not L.is_cuda or L.dtype != torch.float32 or L.dim() != 3 or L.shape[-1] != L.shape[-2]:
        raise TceError(f"{name} must be a CUDA float32 [B, n, n] tensor")
    return (0 if L.shape[0] == 1 else L.stride(0)), L.stride(1) + L.stride(2)


def _dense_diag_grad(L: Tensor) -> Tuple[Tensor, int, int]:
    """Zero [B, n, n] gradient buffer whose diagonal a kernel writes (ldb = n^2, inc = n + 1)."""
    n = L.shape[-1]
    return torch.zeros(L.shape[0], n, n, device=L.device, dtype=torch.float32), n * n, n + 1


@torch.library.custom_op("tce::seglik_diag_fwd", mutates_args=())
def seglik_diag_fwd(smp_traj: Tensor, mean: Tensor, L: Tensor, times: Tensor, init_time: Tensor, init_pos: Tensor,
                    init_vel: Tensor, pred_pairs: Tensor, tables: int, reg_rel: float) -> Tuple[Tensor, Tensor, Tensor]:
    """Diagonal per-episode factors L [B, Dp, Dp] (only the diagonal is read) -> (logp [B, P], diag_max [1] fp64,
    info [B, P] int32)."""
    smp_traj, mean, times = _chk(smp_traj, name="smp_traj"), _chk(mean, name="mean"), _chk(times, name="times")
    init_time, init_pos, init_vel = _chk(init_time), _chk(init_pos), _chk(init_vel)
    pairs = _chk(pred_pairs, torch.int64, "pred_pairs")
    ldb, inc = diag_strides(L)
    B, T = times.shape
    P = pairs.shape[0]
    dev = mean.device
    diag_max = torch.zeros(1, device=dev, dtype=torch.float64)
    logp = torch.empty(B, P, device=dev, dtype=torch.float32)
    info = torch.empty(B, P, device=dev, dtype=torch.int32)
    if B == 0:
        return logp, diag_max, info
    st = _stream()
    _lib.call("tce_seglik_diag_max", tables, _p(L), ldb, inc, _p(times), _p(init_time), _p(pairs), _p(diag_max), B, T,
              P, st)
    _reduce_diag_max(diag_max)
    _lib.call("tce_seglik_diag_fwd", tables, _p(smp_traj), _p(mean), _p(L), ldb, inc, _p(times), _p(init_time),
              _p(init_pos), _p(init_vel), _p(pairs), _p(diag_max), float(reg_rel), _p(logp), _p(info), B, T, P, st)
    return logp, diag_max, info


@seglik_diag_fwd.register_fake
def _(smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs, tables, reg_rel):
    B, P = times.shape[0], pred_pairs.shape[0]
    return mean.new_empty(B, P), mean.new_empty(1, dtype=torch.float64), mean.new_empty(B, P, dtype=torch.int32)


@torch.library.custom_op("tce::seglik_diag_bwd", mutates_args=())
def seglik_diag_bwd(grad_logp: Tensor, smp_traj: Tensor, mean: Tensor, L: Tensor, times: Tensor, init_time: Tensor,
                    init_pos: Tensor, init_vel: Tensor, pred_pairs: Tensor, diag_max: Tensor, tables: int,
                    reg_rel: float) -> Tuple[Tensor, Tensor]:
    """-> (grad_mean [B, Dp], grad_L [B, Dp, Dp], non-zero on the diagonal only)."""
    grad_logp = _chk(grad_logp, name="grad_logp")
    smp_traj, mean, times = _chk(smp_traj), _chk(mean), _chk(times)
    init_time, init_pos, init_vel = _chk(init_time), _chk(init_pos), _chk(init_vel)
    pairs = _chk(pred_pairs, torch.int64, "pred_pairs")
    ldb, inc = diag_strides(L)
    B, T = times.shape
    g_mean = torch.empty(B, mean.shape[-1], device=mean.device, dtype=torch.float32)
    g_L, ldb_g, inc_g = _dense_diag_grad(L)
    if B == 0:
        return g_mean, g_L
    _lib.call("tce_seglik_diag_bwd", tables, _p(smp_traj), _p(mean), _p(L), ldb, inc, _p(times), _p(init_time),
              _p(init_pos), _p(init_vel), _p(pairs), _p(diag_max), float(reg_rel), _p(grad_logp), _p(g_mean), _p(g_L),
              ldb_g, inc_g, B, T, pairs.shape[0], _stream())
    return g_mean, g_L


@seglik_diag_bwd.register_fake
def _(grad_logp, smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs, diag_max, tables, reg_rel):
    return mean.new_empty(mean.shape), L.new_empty(L.shape)


def _seglik_diag_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs[:8], output[1])
    ctx.tables, ctx.reg_rel = inputs[8], inputs[9]
    ctx.set_materialize_grads(False)


def _seglik_diag_backward(ctx, g_logp, g_diag, g_info):
    if g_logp is None:
        return (None,) * 10
    smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs, diag_max = ctx.saved_tensors
    g_mean, g_L = seglik_diag_bwd(g_logp.contiguous(), smp_traj, mean, L, times, init_time, init_pos, init_vel,
                                  pred_pairs, diag_max, ctx.tables, ctx.reg_rel)
    return (None, g_mean if ctx.needs_input_grad[1] else None, g_L if ctx.needs_input_grad[2] else None) + (None,) * 7


seglik_diag_fwd.register_autograd(_seglik_diag_backward, setup_context=_seglik_diag_setup)


def seg_logprob_diag(smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs, tables, reg_rel: float = 1e-4,
                     return_info: bool = False):
    """Segment-wise log-likelihood [B, P] of a diagonal covariance (std_only policy) with per-episode factors
    L [B, Dp, Dp]: only the diagonal of L is read, C is block diagonal per DoF (2 x 2 blocks), O(Dp) per segment.
    Differentiable w.r.t. ``mean`` and ``L`` (the gradient w.r.t. L is zero off the diagonal)."""
    logp, diag_max, info = seglik_diag_fwd(smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs,
                                           tables.handle, float(reg_rel))
    return (logp, info, diag_max) if return_info else logp


def seg_surrogate(smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs, logp_old, advantage, tables,
                  reg_rel: float = 1e-4, uniform: Optional[bool] = None, sigma=None):
    """-> (surrogate loss = -mean(exp(lp - lp_old) * adv) [fp32 scalar, differentiable], mean ratio, logp).
    ``sigma`` = (Sigma0 [n,n] or [1,n,n] fp64, scale [1] fp64 or None): the shared covariance scale * Sigma0 itself; when
    Sigma0 requires grad the gradient is returned w.r.t. the covariance (d loss / d (scale * Sigma0)) and not w.r.t. ``L``
    (contract with the KL projection layer, whose backward consumes it: ops._ProjKLEntropy)."""
    if sigma is None:
        sigma = getattr(L, "_tce_sigma", None)
        if sigma is not None:
            sigma = sigma[:2]
    Lr, shared = _resolve(L, times.shape[0], sigma)
    if not shared:
        sigma = None
        if PER_EPISODE_STAGED and times.shape[0] > 0:
            from . import ops
            return ops.seg_surrogate_staged(smp_traj, mean, L, times, init_time, init_pos, init_vel, pred_pairs,
                                            _chk(logp_old, name="logp_old"), _chk(advantage, name="advantage"),
                                            tables, reg_rel)
    chained, uni = _facts(pred_pairs, init_time, times, shared, uniform)
    loss, ratio, logp, _ = _SegSurrogate.apply(smp_traj, mean, Lr, times, init_time, init_pos, init_vel, pred_pairs,
                                               _chk(logp_old, name="logp_old"), _chk(advantage, name="advantage"),
                                               tables.handle, float(reg_rel), chained, uni,
                                               None if sigma is None else sigma[0],
                                               None if sigma is None else sigma[1])
    return loss, ratio.detach(), logp

"""ctypes binding of libtce_b200.so (the C ABI declared in include/tce_b200.h).

There is no CPU fallback: importing this module without the built library raises, and every
wrapper raises ``TceError`` on a non-zero status.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libtce_b200.so")


class TceError(RuntimeError):
    pass


class MpCfg(C.Structure):
    """Mirror of ``tce_mp_cfg``."""
    _fields_ = [("num_dof", C.c_int32), ("num_basis", C.c_int32), ("num_basis_outside", C.c_int32),
                ("pre_compute_length_factor", C.c_int32), ("auto_scale_basis", C.c_int32),
                ("relative_goal", C.c_int32), ("relative_goal_scaled", C.c_int32), ("reserved", C.c_int32),
                ("tau", C.c_double), ("delay", C.c_double), ("dt", C.c_double), ("alpha", C.c_double),
                ("alpha_phase", C.c_double), ("basis_bandwidth_factor", C.c_double),
                ("weights_scale", C.c_double), ("goal_scale", C.c_double)]


_P, _I64, _I32, _U64, _F, _D = C.c_void_p, C.c_int64, C.c_int, C.c_uint64, C.c_float, C.c_double

# name -> (restype, argtypes); the single source of truth for tests/test_abi.py
SIGNATURES = {
    "tce_version": (C.c_int, []),
    "tce_strerror": (C.c_char_p, [C.c_int]),
    "tce_last_cuda_error": (C.c_char_p, []),
    "tce_prodmp_tables_create": (C.c_int, [C.POINTER(MpCfg), _P, C.POINTER(_P)]),
    "tce_prodmp_tables_destroy": (None, [_P]),
    "tce_prodmp_tables_num_pc": (C.c_int, [_P]),
    "tce_prodmp_tables_export": (C.c_int, [_P] * 8),
    "tce_prodmp_traj_fwd": (C.c_int, [_P] * 7 + [_I64, _I64, _P]),
    "tce_prodmp_traj_fwd_uniform": (C.c_int, [_P] * 8 + [_I64, _I64, _P]),
    "tce_prodmp_traj_bwd": (C.c_int, [_P] * 7 + [_I64, _I64, _P]),
    "tce_mvn_rsample": (C.c_int, [_P, _P, _I64, _P, _U64, _U64, _P, _I64, _I32, _P]),
    "tce_chol_fwd": (C.c_int, [_P, _P, _P, _I64, _I32, _P]),
    "tce_chol_bwd": (C.c_int, [_P, _P, _P, _I64, _I32, _P]),
    "tce_policy_head_fwd": (C.c_int, [_P, _I64, _F, _P, _I64, _I32, _P]),
    "tce_policy_head_bwd": (C.c_int, [_P, _I64, _P, _P, _I64, _I32, _P]),
    "tce_policy_head_diag_fwd": (C.c_int, [_P, _I64, _F, _P, _I64, _I32, _P]),
    "tce_policy_head_diag_bwd": (C.c_int, [_P, _I64, _P, _P, _I64, _I32, _P]),
    "tce_proj_kl_diag_fwd": (C.c_int, [_P, _I64, _I64, _P, _I64, _I64, _D, _P, _I64, _I32, _P, _I64, _I64, _P, _P, _I64,
                                       _I32, _P]),
    "tce_proj_kl_diag_bwd": (C.c_int, [_P, _I64, _I64, _P, _I64, _I64, _P, _P, _I64, _I64, _P, _I64, _I64, _I64, _I32,
                                       _P]),
    "tce_seglik_diag_max": (C.c_int, [_P, _P, _I64, _I64, _P, _P, _P, _P, _I64, _I64, _I64, _P]),
    "tce_seglik_diag_fwd": (C.c_int, [_P, _P, _P, _P, _I64, _I64, _P, _P, _P, _P, _P, _P, _D, _P, _P, _I64, _I64, _I64,
                                      _P]),
    "tce_seglik_diag_bwd": (C.c_int, [_P, _P, _P, _P, _I64, _I64, _P, _P, _P, _P, _P, _P, _D, _P, _P, _P, _I64, _I64,
                                      _I64, _I64, _I64, _P]),
    "tce_gauss_stats": (C.c_int, [_P, _P, _I64, _P, _P, _I64, _P, _I64, _I32, _P]),
    "tce_gauss_stats_bwd": (C.c_int, [_P, _P, _I64, _P, _P, _I64, _P, _P, _P, _I64, _I32, _P]),
    "tce_gauss_maha": (C.c_int, [_P, _P, _P, _I64, _P, _P, _P, _I64, _I32, _P]),
    "tce_gauss_maha_bwd_full": (C.c_int, [_P, _P, _P, _I64, _P, _P, _P, _I64, _I32, _P]),
    "tce_tri_inverse": (C.c_int, [_P, _I64, _P, _I64, _I32, _P]),
    "tce_gauss_maha_shared": (C.c_int, [_P, _P, _P, _P, _P, _P, _I64, _I32, _P]),
    "tce_proj_mean_fwd": (C.c_int, [_P, _P, _P, _D, _P, _I64, _I32, _P]),
    "tce_proj_mean_bwd": (C.c_int, [_P, _P, _P, _D, _P, _P, _P, _I64, _I32, _P]),
    "tce_proj_entropy_fwd": (C.c_int, [_P, _P, _I64, _I32, _P, _P, _I64, _I32, _P]),
    "tce_proj_entropy_bwd": (C.c_int, [_P, _P, _I64, _I32, _P, _P, _I64, _I32, _P]),
    "tce_proj_kl_save_doubles": (C.c_size_t, [_I64, _I32]),
    "tce_proj_kl_cov_fwd": (C.c_int, [_P, _P, _D, _P, _P, _P, _I32, _I64, _I32, _P]),
    "tce_proj_kl_cov_bwd": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I32, _P]),
    "tce_proj_kl_entropy_fwd": (C.c_int, [_P, _P, _D, _P, _I64, _I32, _P, _P, _P, _P, _I32, _I64, _I32, _P]),
    "tce_proj_kl_entropy_bwd": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I32, _P]),
    "tce_proj_kl_entropy_bwd_tr": (C.c_int, [_P, _P, _P, _P, _D, _P, _I64, _I32, _P]),
    "tce_proj_kl_bwd_sigma": (C.c_int, [_P, _P, _P, _I32, _D, _P, _I64, _I32, _P]),
    "tce_proj_kl_bwd_sigma_k": (C.c_int, [_P, _P, _P, _I32, _D, _P, _I64, _I32, _P]),
    "tce_proj_kl_bwd_prep": (C.c_int, [_P, _I64, _I32, _P]),
    "tce_proj_kl_entropy_fwd_sigma_vec": (C.c_int, [_P, _I64, _F, _P, _P, _D, _P, _I64, _I32, _P, _P, _P, _P, _I32, _I64,
                                                    _I32, _P]),
    "tce_proj_kl_bwd_sigma_k_vec": (C.c_int, [_P, _P, _I64, _P, _P, _I32, _D, _P, _I64, _I32, _P]),
    "tce_proj_kl_entropy_bwd_inv": (C.c_int, [_P, _P, _P, _P, _P, _P, _I64, _I32, _P]),
    "tce_proj_kl_entropy_fwd_sigma": (C.c_int, [_P, _P, _D, _P, _I64, _I32, _P, _P, _P, _P, _I32, _I64, _I32, _P]),
    "tce_proj_kl_entropy_fwd_chol": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I32, _P]),
    "tce_grad_sumsq": (C.c_int, [_P, _I64, _P, _P]),
    "tce_adam_step": (C.c_int, [_I32, _P, _P, _P, _P, _P, _P, _D, _D, _D, _D, _D, _D, _P]),
    "tce_proj_frob_cov_fwd": (C.c_int, [_P, _P, _I64, _D, _P, _P, _P, _I64, _I32, _P]),
    "tce_proj_frob_cov_bwd": (C.c_int, [_P, _P, _I64, _D, _P, _P, _P, _P, _I64, _I32, _P]),
    "tce_proj_w2_cov_fwd": (C.c_int, [_P, _P, _I64, _D, _I32, _P, _P, _I64, _I32, _P]),
    "tce_proj_w2_cov_bwd": (C.c_int, [_P, _P, _I64, _D, _I32, _P, _P, _I64, _I32, _P]),
    "tce_cov_distance": (C.c_int, [_I32, _P, _P, _I64, _I32, _P, _P, _P, _I64, _I32, _P]),
    "tce_seglik_work_bytes": (C.c_size_t, [_P, _I64, _I64]),
    "tce_seglik_gram": (C.c_int, [_P, _P, _P, _P, _I64, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _P]),
    "tce_seglik_chol": (C.c_int, [_P, _P, _P, _P, _D, _P, _P, _P, _D, _P, _P, _P, _I64, _I64, _P]),
    "tce_seglik_bwd": (C.c_int, [_P, _P, _P, _I64, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _P]),
    "tce_seglik_compiled": (C.c_int, [_P]),
    "tce_seglik_gram_sigma": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _P]),
    "tce_seglik_shared_part_doubles": (C.c_size_t, [_P, _I64]),
    "tce_seglik_bwd_shared": (C.c_int, [_P] * 11 + [_I64, _I64, _I64, _P]),
    "tce_seglik_fused_config": (C.c_int, [_P, _I64, _I64, _I32, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                          C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "tce_seglik_prepass": (C.c_int, [_P] * 4 + [_I64] + [_P] * 9 + [_I32, _I64, _I64, _I64, _P]),
    "tce_seglik_fused": (C.c_int, [_P, _P, _P, _I64, _P, _P, _P, _P, _D, _I32, _P, _P, _P, _D, _P, _P, _P, _P, _P, _P,
                                   _I32, _I64, _I64, _P]),
    "tce_seglik_dsigma_reduce": (C.c_int, [_P, _P, _I32, _P, _P, _P, _P, _P]),
    "tce_seglik_uniform_ws_doubles": (C.c_size_t, [_P, _I64]),
    "tce_seglik_uniform_parts": (C.c_int, [_P, _I64, _I64, C.POINTER(C.c_int32), C.POINTER(C.c_int64)]),
    "tce_seglik_uniform_prep": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _D, _I32, _I64, _P]),
    "tce_seglik_uniform_main": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I32, _P, _P, _P, _D, _P, _P, _P, _P, _P, _I64,
                                          _I64, _I64, _P]),
    "tce_seglik_uniform_finish": (C.c_int, [_P, _P, _P, _I32, _P, _P, _P, _P, _I64, _P]),
    "tce_p2p_allreduce_sumsq": (C.c_int, [_I32, _I32, _P, _P, _I64, _P, _P, _P, _P]),
    "tce_p2p_allreduce_sumsq_range": (C.c_int, [_I32, _I32, _P, _P, _I64, _I64, _I32, _I32, _P, _P, _P, _P]),
    "tce_p2p_push_xchg_bytes": (C.c_size_t, [_I32, _I64]),
    "tce_p2p_push_allreduce_sumsq": (C.c_int, [_I32, _I32, _P, _P, _I64, _I64, _I64, _I32, _I32, _P, _P, _P, _P]),
    "tce_epoch_mean_fwd": (C.c_int, [_P, _P, _P, _D, _P, _P, _P, _P, _I64, _I32, _P]),
    "tce_epoch_tr_mean": (C.c_int, [_P, _P, _P, _P, _P, _P, _D, _D, _P, _P, _I64, _I32, _P]),
    "tce_epoch_mean_combine": (C.c_int, [_P, _P, _P, _P, _P, _P, _D, _P, _I64, _I32, _P]),
    "tce_epoch_metrics": (C.c_int, [_P, _P, _P, _P, _I64, _D, _I32, _D, _P, _P]),
    "tce_gae": (C.c_int, [_P, _P, _P, _P, _F, _F, _I32, _P, _P, _I64, _I64, _P]),
    "tce_segment_advantage_raw": (C.c_int, [_I32, _P, _P, _P, _P, _F, _P, _P, _I64, _I64, _I64, _P]),
    "tce_sum_stats": (C.c_int, [_P, _P, _I64, _P]),
    "tce_normalize_by_stats": (C.c_int, [_P, _P, _I64, _P]),
    "tce_debug_kl_phase_cycles": (C.c_int, [_P]),
    "tce_debug_seglik_phase_cycles": (C.c_int, [_P]),
    "tce_bench_fma": (C.c_int, [_I32, _I32, _P, C.POINTER(C.c_double), _P]),
}

_lib = None


def load() -> C.CDLL:
    """Load the shared library (raises if it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise TceError(f"{LIB_PATH} is missing: run `python -m tce_rl_b200._build` "
                           "(or __graft_entry__.build()); there is no CPU fallback")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(status: int, what: str = "") -> None:
    if status != 0:
        lib = load()
        msg = lib.tce_strerror(status).decode()
        if status == -3:
            msg += " -- " + lib.tce_last_cuda_error().decode()
        raise TceError(f"{what}: {msg} (status {status})")


LAUNCHES = 0          # kernel launches issued through the C ABI (bench.py reports them as gpu_launches)
_NO_KERNEL = {"tce_seglik_fused_config", "tce_seglik_compiled", "tce_seglik_shared_part_doubles", "tce_seglik_uniform_parts", "tce_prodmp_tables_export", "tce_prodmp_tables_create", "tce_debug_kl_phase_cycles", "tce_debug_seglik_phase_cycles"}


# Optional per-launch timing (bench.py's roofline report): when TIMING is a list, every kernel-launching ABI call is
# bracketed by CUDA events on ITS launching stream (the `stream` argument, always the last one) and
# (name, start_event, stop_event) is appended.  None = off (the default: no overhead on the product path).
TIMING = None


def call(name: str, *args) -> None:
    global LAUNCHES
    if TIMING is not None and name not in _NO_KERNEL:
        import torch
        st = torch.cuda.ExternalStream(args[-1]) if args[-1] else torch.cuda.default_stream()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        check(getattr(load(), name)(*args), name)
        b.record(st)
        TIMING.append((name, a, b))
        LAUNCHES += 1
        return
    check(getattr(load(), name)(*args), name)
    if name not in _NO_KERNEL:
        LAUNCHES += 1

"""ProDMP with the (stateful) method surface of ``mp_pytorch.mp.ProDMP`` on top of the stateless kernels.

Reference construction: ``get_mp`` (mprl/util/util_mp.py:11-46); reference call sites:
mprl/rl/policy/temporal_correlated_policy.py:76-92,188-192.  Everything is evaluated by the CUDA
kernels (``tce::prodmp_traj``, ``tce::mvn_rsample``, ``tce::traj_pos_cov``, ``tce::traj_pos_std``).
"""
from __future__ import annotations

import torch

from . import ops, ops_seglik


class ProDMP:
    def __init__(self, tables: ops.Tables):
        self.tables = tables
        self.num_dof = tables.num_dof
        self.num_basis_g = tables.num_basis_g
        self.reset()

    # ---- mp_pytorch keeps the last inputs -----------------------------------------------------------
    def reset(self):
        self.times = self.params = self.params_L = None
        self.init_time = self.init_pos = self.init_vel = None
        self._traj = None

    def update_inputs(self, times=None, params=None, params_L=None, init_time=None, init_pos=None, init_vel=None):
        for name, val in (("times", times), ("params", params), ("params_L", params_L), ("init_time", init_time),
                          ("init_pos", init_pos), ("init_vel", init_vel)):
            if val is not None:
                setattr(self, name, val)
                self._traj = None
                if name == "times":
                    self._check_range(val)

    strict_range = True      # raise like mp_pytorch as soon as a time lies beyond the pre-computed range

    def _check_range(self, times):
        """mp_pytorch raises ``RuntimeError`` when a scaled time exceeds the pre-computed range (``factor`` = 5
        periods, util_mp.py:33).  The kernels clamp the table index (no device-side exception), so the shim keeps a
        lazy device flag ``range_flag`` (1 = some time was out of range since the last ``check_range()``) and, with
        ``strict_range`` (default), reads it right away -- one host synchronisation, as in the reference; under CUDA-
        graph capture or with ``strict_range = False`` call ``check_range()`` when convenient."""
        if times is None or times.numel() == 0:
            return
        over = ((times.detach().amax() - self.tables.delay) / self.tables.tau > self.tables.factor).to(torch.int32)
        self.range_flag = over if getattr(self, "range_flag", None) is None else torch.maximum(self.range_flag, over)
        if self.strict_range and not (times.is_cuda and torch.cuda.is_current_stream_capturing()):
            self.check_range()

    def check_range(self):
        flag = getattr(self, "range_flag", None)
        self.range_flag = None
        if flag is not None and bool(flag.item()):
            raise RuntimeError("Time is beyond the pre-computation range.")

    def _flat(self, t, trailing):
        lead = t.shape[:t.ndim - trailing]
        return t.reshape(-1, *t.shape[t.ndim - trailing:]), lead

    def _trajectory(self):
        if self._traj is None:
            times, lead = self._flat(self.times, 1)
            params, _ = self._flat(self.params, 1)
            it, _ = self._flat(self.init_time, 0)
            ip, _ = self._flat(self.init_pos, 1)
            iv, _ = self._flat(self.init_vel, 1)
            traj = ops.prodmp_traj(params.contiguous(), times.contiguous(), it.contiguous(), ip.contiguous(),
                                   iv.contiguous(), self.tables.handle, self.num_dof)
            self._traj = traj.reshape(*lead, traj.shape[-2], traj.shape[-1])
        return self._traj

    def get_traj_pos(self, times=None, params=None, init_time=None, init_pos=None, init_vel=None, flat_shape=False):
        self.update_inputs(times, params, None, init_time, init_pos, init_vel)
        pos = self._trajectory()[..., :self.num_dof]                  # [*a, T, D]
        return pos.transpose(-1, -2).reshape(*pos.shape[:-2], -1) if flat_shape else pos

    def get_traj_vel(self, times=None, params=None, init_time=None, init_pos=None, init_vel=None, flat_shape=False):
        self.update_inputs(times, params, None, init_time, init_pos, init_vel)
        vel = self._trajectory()[..., self.num_dof:]
        return vel.transpose(-1, -2).reshape(*vel.shape[:-2], -1) if flat_shape else vel

    def sample_trajectories(self, times=None, params=None, params_L=None, init_time=None, init_pos=None,
                            init_vel=None, num_smp=1, flat_shape=False, eps=None, seed=None, offset=0):
        """theta ~ N(params, L L^T), then pos / vel: [*a, num_smp, T, D] each (sample axis after the batch axes)."""
        old = (self.times, self.params, self.params_L, self.init_time, self.init_pos, self.init_vel)
        lead = params.shape[:-1]
        mean2, _ = self._flat(params, 1)
        L3 = params_L.reshape(-1, *params_L.shape[-2:]) if params_L.dim() != 3 else params_L
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, [], device="cpu").item())   # host generator -> reproducible
        smp = []
        for s in range(num_smp):
            e = None if eps is None else eps[s].reshape(mean2.shape)
            smp.append(ops.mvn_rsample(mean2.contiguous(), L3, e, seed, offset + s))
        theta = torch.stack(smp, 1).reshape(*lead, num_smp, -1)
        ex = lambda v, trailing: v.unsqueeze(v.ndim - trailing).expand(*v.shape[:v.ndim - trailing], num_smp,
                                                                       *v.shape[v.ndim - trailing:])
        self.reset()
        self.update_inputs(ex(times, 1), theta, None, ex(init_time, 0), ex(init_pos, 1), ex(init_vel, 1))
        pos, vel = self.get_traj_pos(flat_shape=flat_shape), self.get_traj_vel(flat_shape=flat_shape)
        self.reset()
        self.update_inputs(*old)
        return pos, vel

    def _pos_cov_inputs(self):
        """times [n, T], init_time [n] and params_L as [n, Dp, Dp], or as the ONE [1, Dp, Dp] matrix behind a
        broadcast (stride-0) factor, so that a shared factor is neither copied nor given a per-episode gradient."""
        times, lead = self._flat(self.times, 1)
        n, Dp = times.shape[0], self.num_dof * self.num_basis_g
        L = self.params_L
        if L.dim() > 2 and tuple(L.shape[:-2]) != tuple(lead):
            L = L.expand(*lead, Dp, Dp)
        if L.dim() > 3:
            L = L.reshape(-1, Dp, Dp)
        shared = ops_seglik.shared_factor(L, n)
        if shared is not None:
            L = shared
        elif L.dim() != 3 or L.shape[0] != n:
            raise ValueError(f"params_L must broadcast to [*a, {Dp}, {Dp}] over times [*a, T], got {list(L.shape)}")
        return times, self.init_time.reshape(-1), L, lead

    def get_traj_pos_cov(self, times=None, params_L=None, init_time=None, init_pos=None, init_vel=None,
                         reg: float = 1e-4):
        """[*a, D*T, D*T] covariance of the positions at the times [*a, T] (rows DoF-major, time-minor) under the
        parameter distribution N(., L L^T): H (L L^T) H^T + reg * max diag over the whole call * I.  Any time grid
        (TCE passes pairs, [*a] = [B, P]); differentiable w.r.t. params_L.  One factor may be broadcast over the
        batch (stride-0 expand): it is read once and its gradient is summed over the batch."""
        self.update_inputs(times, None, params_L, init_time, init_pos, init_vel)
        times2, it, L, lead = self._pos_cov_inputs()
        cov = ops.traj_pos_cov(L, times2, it, self.tables.handle, self.num_dof, float(reg))
        return cov.reshape(*lead, *cov.shape[-2:])

    def get_traj_pos_std(self, times=None, params_L=None, init_time=None, init_pos=None, init_vel=None,
                         flat_shape=False, reg: float = 1e-4):
        """Standard deviations of the positions, sqrt(diag(get_traj_pos_cov)) with the same regulariser, without
        forming the covariance: [*a, T, D], or [*a, D*T] DoF-major with ``flat_shape``.  Differentiable w.r.t.
        params_L."""
        self.update_inputs(times, None, params_L, init_time, init_pos, init_vel)
        times2, it, L, lead = self._pos_cov_inputs()
        std = ops.traj_pos_std(L, times2, it, self.tables.handle, self.num_dof, float(reg))
        std = std.reshape(*lead, *std.shape[-2:])
        return std.transpose(-1, -2).reshape(*lead, -1) if flat_shape else std


def get_mp(**kwargs) -> ProDMP:
    """Mirror of ``mprl.util.util_mp.get_mp`` (util_mp.py:11-46): {"type": "prodmp", "args": {...}}."""
    assert kwargs["type"] == "prodmp"
    args = dict(kwargs["args"])
    args.pop("dtype", None)
    args.pop("device", None)
    for unsupported in ("learn_tau", "learn_delay", "learn_alpha_phase", "disable_weights", "disable_goal"):
        if args.pop(unsupported, False):
            raise NotImplementedError(f"{unsupported}=True is not used by any TCE config and is not built")
    return ProDMP(ops.Tables(**args))

"""The first stage of the policy, forward and backward: reparameterised sampling (``tce::mvn_rsample`` and the policy and
ProDMP entry points on top of it) and trajectory synthesis (``tce::prodmp_traj``), against the fp64 oracle with torch
autograd for the reference gradients.  Inputs are fp32 values; the oracle evaluates the same values in fp64.

Every case states which kernel and which regime it reaches.  Where the choice is made in Python (uniform or general
trajectory kernel, a regenerating backward launch) the launch counter asserts it; where the C entry point chooses
(bulk-copy or row-wise rsample, episodes per CTA, grid-stride loops, store paths) the case gives the arithmetic, and the
mirror ``ops.traj_uniform_layout`` of the uniform launch is checked against it on a 148-SM device.

Outputs are allocated into blocks just filled with NaN, so a store a kernel skips shows up as NaN rather than as a
stale value of an earlier call."""
import math

import pytest
import torch

from oracle import policy as opol
from oracle import util as ou
from oracle.gen_golden import MP_CONFIGS, NUM_TIMES
from oracle.prodmp import get_mp as oracle_get_mp

pytestmark = pytest.mark.gpu
if torch.cuda.is_available():
    from tce_rl_b200 import ops
    from tce_rl_b200.mp import ProDMP
    from tce_rl_b200.rl import policy_factory

DEV = "cuda:0"
RSAMPLE_TOL = 2e-5       # relative to the largest reference value, as the rsample and Mahalanobis tests
TRAJ_TOL = 1e-5          # trajectories and their gradients: the backward sums the T terms serially in fp32
UNIFORM_VS_GENERAL = 2e-6
B200_SMS = 148           # the regime arithmetic below is for this SM count
# the five compiled (num_dof, K1) shapes and the task settings they run with, and (4, 16): Dp = 64, not compiled
SHAPES = {(2, 3): "metaworld", (7, 4): "table_tennis", (4, 9): "metaworld", (7, 9): "box", (4, 16): "box"}
COMPILED = [(7, 9), (4, 9), (7, 4), (3, 4), (2, 3)]
COMPILED_TASK = {(7, 9): "box", (4, 9): "metaworld", (7, 4): "table_tennis", (3, 4): "table_tennis",
                 (2, 3): "metaworld"}


def f64(t):
    return t.detach().double().cpu()


def gen(seed):
    return torch.Generator().manual_seed(seed)


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def assert_close(got, want, tol, what):
    """max |got - want| <= tol * max |want|, want in fp64 on the CPU; NaN fails."""
    got, want = f64(got), want.detach().double()
    assert got.shape == want.shape, what
    err = (got - want).abs().max().item() / want.abs().max().item()
    assert err <= tol, f"{what}: relative error {err:.3g} > {tol:.3g}"


_COUNTS = {}


def _lib_launch_count(name):
    """Launches of one ABI entry so far (a counting wrapper installed on first use)."""
    from tce_rl_b200 import _lib
    if "installed" not in _COUNTS:
        orig = _lib.call

        def counting(n, *a):
            _COUNTS[n] = _COUNTS.get(n, 0) + 1
            return orig(n, *a)
        _lib.call = counting
        _COUNTS["installed"] = True
    return _COUNTS.get(name, 0)


class Launches:
    """Launch counts of the given ABI entries inside a ``with`` block: ``.delta`` -> {entry: count}."""

    def __init__(self, *names):
        self.names = names

    def __enter__(self):
        self.start = {n: _lib_launch_count(n) for n in self.names}
        return self

    def __exit__(self, *exc):
        self.delta = {n: _lib_launch_count(n) - self.start[n] for n in self.names}


def poison(shape):
    """Fill a block of the caching allocator with NaN and free it: the next allocation of this size gets it."""
    junk = torch.full(shape, float("nan"), device=DEV)
    del junk


def factor(n, B, g, upper=True):
    """Well-conditioned lower-triangular factors (diagonal in [0.5, 1.5]); ``upper`` fills the strict upper triangle
    with values the kernels must never read."""
    L = torch.tril(0.3 / math.sqrt(n) * torch.randn(B, n, n, generator=g), -1) + \
        torch.diag_embed(0.5 + torch.rand(B, n, generator=g))
    return L + torch.triu(torch.randn(B, n, n, generator=g), 1) if upper else L


def shared_vector(n, g):
    """Covariance vector of a non-contextual policy: softplus(diagonal) + 1e-4 in [0.5, 1.5], small strict lower part."""
    d = 0.5 + torch.rand(n, generator=g, dtype=torch.float64) - 1e-4
    return torch.cat([torch.log(torch.expm1(d)), 0.3 / math.sqrt(n) * torch.randn(n * (n - 1) // 2, generator=g,
                                                                                    dtype=torch.float64)]).float()


def solve_eps(L64, z, mean):
    """The standard-normal draw behind z = mean + tril(L) eps, solved in fp64."""
    return torch.linalg.solve_triangular(torch.tril(L64), (f64(z) - f64(mean))[..., None], upper=False)[..., 0]


def host_seed(k):
    """The seed a policy's ``sample`` draws after ``torch.manual_seed(k)`` (its host generator)."""
    torch.manual_seed(k)
    return int(torch.randint(0, 2 ** 62, [], device="cpu").item())


_POLICIES = {}


def tce_policy(typ, n, cfg=None):
    """A non-contextual policy of the package (its covariance vector is set by the caller)."""
    key = (typ, n, None if cfg is None else tuple(sorted(cfg.items())))
    if key not in _POLICIES:
        kw = dict(dim_in=4, dim_out=n, mean_net_args=dict(avg_neuron=8, num_hidden=1, shape=0.0),
                  variance_net_args=dict(std_only=False, contextual=False), init_method="orthogonal",
                  out_layer_gain=0.01, act_func_hidden="leaky_relu", act_func_last=None, dtype="float32", device=DEV,
                  min_std=1e-4)
        if cfg is not None:
            kw["mp"] = dict(type="prodmp", args=dict(cfg))
        _POLICIES[key] = policy_factory(typ, **kw)
    return _POLICIES[key]


def oracle_traj(cfg, params, times, init_time, init_pos, init_vel):
    omp = oracle_get_mp(type="prodmp", args=dict(cfg, dtype=torch.float64))
    omp.update_inputs(times, params, None, init_time, init_pos, init_vel)
    return torch.cat([omp.get_traj_pos(), omp.get_traj_vel()], -1)


# ---- A. reparameterised-sample gradients ---------------------------------------------------------------------------
# tce_mvn_rsample takes the bulk-copy kernel for contiguous, 16-byte aligned per-episode factors of odd n <= 64 and
# B >= 32 (here n = 63 at B = 32, 33, 2051), on floor(B / 4) groups of four episodes -- 512 groups at B = 2051, more
# than its 3 x 148 CTAs, so the group loop strides -- and runs the B % 4 tail (1 at B = 33, 3 at B = 2051) through the
# row-wise kernel.  Everything else is row-wise: even n, n = 100, B < 32, stride-0 shared factors and misaligned views.
RS_N = [6, 28, 36, 63, 64, 100]
RS_B = [1, 31, 32, 33, 2051]
RS_CASES = [(n, B, noise, fac) for n in RS_N for B in RS_B for noise in ("injected", "philox")
            for fac in ("episode", "shared")] + \
           [(63, B, noise, "misaligned") for B in (32, 33, 2051) for noise in ("injected", "philox")]


def rsample_kernel(n, B, fac):
    if fac == "episode" and n % 2 == 1 and n <= 64 and B >= 32:
        return "bulk" + ("+rows" if B % 4 else "")
    return "rows"


@pytest.mark.parametrize("n,B,noise,fac", RS_CASES)
def test_rsample_gradients(n, B, noise, fac):
    """BlackBoxPolicy.sample(True, ...) = mean + tril(L) eps: gradients w.r.t. the mean, the factor (per episode, a
    misaligned view, or the policy's stride-0 shared factor through the head's backward to its covariance vector) and
    the injected eps, against autograd of the oracle.  In-kernel draws: the reference eps is solved from the sample."""
    kernel = rsample_kernel(n, B, fac)
    g = gen(n * 7919 + B)
    mean, eps, w = torch.randn(B, n, generator=g), torch.randn(B, n, generator=g), torch.randn(B, n, generator=g)
    pol = tce_policy("BlackBoxPolicy", n)
    m = mean.to(DEV).requires_grad_(True)
    e = eps.to(DEV).requires_grad_(fac != "shared") if noise == "injected" else None
    if fac == "shared":
        vec = shared_vector(n, g)
        with torch.no_grad():
            pol.variance_net.variable.copy_(vec.to(DEV))
        pol.variance_net.variable.grad = None
        L = pol.shared_params_L(B)
        assert B == 1 or L.stride(0) == 0
    else:
        L_host = factor(n, B, g)
        if fac == "misaligned":
            buf = torch.zeros(B * n * n + 1, device=DEV)
            buf[1:] = L_host.reshape(-1).to(DEV)
            buf.requires_grad_(True)
            L = buf[1:].view(B, n, n)
            assert L.is_contiguous() and L.data_ptr() % 16 != 0
        else:
            L = L_host.to(DEV).requires_grad_(True)
    with Launches("tce_mvn_rsample") as fwd:
        torch.manual_seed(0)                            # the policy's host generator picks the Philox seed
        poison((B, n))
        z = pol.sample(True, m, L, eps=e, use_mean=False)
    assert fwd.delta["tce_mvn_rsample"] == 1 and z.requires_grad
    # reference
    m64 = mean.double().requires_grad_(True)
    if fac == "shared":
        vec64 = vec.double().requires_grad_(True)
        opolicy = opol.BlackBoxPolicy(n, cov_vector=vec64, contextual=False, min_std=1e-4)
        L64 = opolicy.vector_to_cholesky(ou.add_expand_dim(vec64, [0], [B]))
        wrt = [m64, vec64]
    else:
        L64 = L_host.double().requires_grad_(True)
        wrt = [m64, L64]
    if noise == "injected":
        e64 = eps.double().requires_grad_(e is not None and e.requires_grad)
        if e64.requires_grad:
            wrt.append(e64)
    else:
        e64 = solve_eps(L64.detach(), z, mean)
        # the draws are those of the identity factor at stride 0 (what the backward regenerates), whatever the factor
        torch.manual_seed(0)
        zs = pol.sample(False, torch.zeros(B, n, device=DEV), torch.eye(n, device=DEV).expand(B, n, n))
        assert (f64(zs) - e64).abs().max().item() <= 1e-4 * e64.abs().max().item()
        if B * n >= 1000:
            assert abs(e64.std().item() - 1.0) < 0.1
    z64 = m64 + torch.einsum('bij,bj->bi', torch.tril(L64), e64)
    if noise == "injected":
        assert_close(z, z64, RSAMPLE_TOL, f"sample ({kernel})")
    refs = torch.autograd.grad((z64 * w.double()).sum(), wrt)
    with Launches("tce_mvn_rsample") as bwd:
        z.backward(w.to(DEV))
    # in-kernel draws: one launch regenerates them for d/dL; injected eps: no launch
    assert bwd.delta["tce_mvn_rsample"] == (1 if noise == "philox" else 0)
    assert torch.equal(m.grad.cpu(), w)                                           # d/dmean = g exactly
    if fac == "shared":
        assert_close(pol.variance_net.variable.grad, refs[1], RSAMPLE_TOL, "d/d covariance vector")
    else:
        gL = buf.grad[1:].view(B, n, n) if fac == "misaligned" else L.grad
        if fac == "misaligned":
            assert buf.grad[0].item() == 0.0
        assert_close(gL, refs[1], RSAMPLE_TOL, f"d/dL ({kernel})")
        assert gL.triu(1).abs().max().item() == 0.0
    if len(refs) == 3:
        assert_close(e.grad, refs[2], RSAMPLE_TOL, "d/deps")
    elif e is not None:
        assert e.grad is None


def test_sample_without_grad_records_nothing():
    """``sample(False, ...)`` on inputs that require grad: one launch per op, no tensor saved for a backward, a result
    without history; the op itself on inputs without grad saves nothing either."""
    n, B = 28, 40
    g = gen(3)
    cfg = dict(MP_CONFIGS["table_tennis"])
    T = NUM_TIMES["table_tennis"]
    m = torch.randn(B, n, generator=g).to(DEV).requires_grad_(True)
    L = factor(n, B, g, upper=False).to(DEV).requires_grad_(True)
    times = ou.get_times(torch.zeros(B, dtype=torch.float64), T, cfg["dt"]).float().to(DEV)
    z0, it = torch.zeros(B, 7, device=DEV), torch.zeros(B, device=DEV)
    saved = []

    def pack(t):
        saved.append(t)
        return t
    for typ in ("BlackBoxPolicy", "TemporalCorrelatedPolicy"):
        pol = tce_policy(typ, n, cfg if typ != "BlackBoxPolicy" else None)
        args = (times, it, z0, z0) if typ != "BlackBoxPolicy" else ()
        for eps in (None, torch.randn(B, n, device=DEV, requires_grad=True)):
            with Launches("tce_mvn_rsample", "tce_prodmp_traj_fwd") as n_l, \
                    torch.autograd.graph.saved_tensors_hooks(pack, lambda t: t):
                out = pol.sample(False, m, L, *args, eps=eps)
            assert out.grad_fn is None and not out.requires_grad and saved == []
            assert n_l.delta == {"tce_mvn_rsample": 1, "tce_prodmp_traj_fwd": int(typ != "BlackBoxPolicy")}
    with torch.autograd.graph.saved_tensors_hooks(pack, lambda t: t):
        out = ops.mvn_rsample(m.detach(), L.detach(), None, 1, 0)
    assert out.grad_fn is None and saved == []


@pytest.mark.parametrize("D,K1", list(SHAPES))
@pytest.mark.parametrize("B", [1, 33, 2051])
@pytest.mark.parametrize("noise", ["injected", "philox"])
@pytest.mark.parametrize("fac", ["episode", "shared"])
def test_trajectory_sample_gradients(D, K1, B, noise, fac):
    """TemporalCorrelatedPolicy.sample(True, ...): rsample then trajectory, gradients w.r.t. the mean, the factor (or
    the covariance vector behind the shared factor) and the injected eps.  Time grid common to the batch, starting at
    0: B = 2051 synthesises on the uniform kernel (4 episodes per CTA, see part E), B = 1 and 33 on the general kernel.
    rsample as in test_rsample_gradients (bulk copy plus a row-wise tail at n = 63, B >= 33)."""
    task = SHAPES[(D, K1)]
    cfg, T = dict(MP_CONFIGS[task], num_dof=D, num_basis=K1 - 1), NUM_TIMES[task]
    n = D * K1
    g = gen(1000 * n + B)
    mean, eps = 0.5 * torch.randn(B, n, generator=g), torch.randn(B, n, generator=g)
    init_pos, init_vel = torch.rand(B, D, generator=g) * 2 - 1, 0.1 * torch.randn(B, D, generator=g)
    init_time = torch.zeros(B)
    times = ou.get_times(init_time.double(), T, cfg["dt"]).float()
    w = torch.randn(B, T, 2 * D, generator=g)
    pol = tce_policy("TemporalCorrelatedPolicy", n, cfg)
    m = mean.to(DEV).requires_grad_(True)
    e = eps.to(DEV).requires_grad_(True) if noise == "injected" else None
    if fac == "shared":
        vec = shared_vector(n, g)
        with torch.no_grad():
            pol.variance_net.variable.copy_(vec.to(DEV))
        pol.variance_net.variable.grad = None
        L = pol.shared_params_L(B)
    else:
        L_host = factor(n, B, g)
        L = L_host.to(DEV).requires_grad_(True)
    c = lambda t: t.to(DEV)
    entry = "tce_prodmp_traj_fwd_uniform" if B >= 64 else "tce_prodmp_traj_fwd"
    with Launches("tce_mvn_rsample", entry) as fwd:
        torch.manual_seed(11)
        poison((B, T, 2 * D))
        traj = pol.sample(True, m, L, c(times), c(init_time), c(init_pos), c(init_vel), eps=e)
    assert fwd.delta == {"tce_mvn_rsample": 1, entry: 1}
    m64 = mean.double().requires_grad_(True)
    if fac == "shared":
        vec64 = vec.double().requires_grad_(True)
        opolicy = opol.TemporalCorrelatedPolicy(n, mp=dict(type="prodmp", args=dict(cfg, dtype=torch.float64)),
                                                cov_vector=vec64, contextual=False, min_std=1e-4)
        L64 = opolicy.vector_to_cholesky(ou.add_expand_dim(vec64, [0], [B]))
        wrt = [m64, vec64]
    else:
        opolicy = opol.TemporalCorrelatedPolicy(n, mp=dict(type="prodmp", args=dict(cfg, dtype=torch.float64)),
                                                contextual=True, min_std=1e-4)
        L64 = L_host.double().requires_grad_(True)
        wrt = [m64, L64]
    if noise == "injected":
        e64 = eps.double().requires_grad_(True)
        wrt.append(e64)
    else:
        theta = ops.mvn_rsample(m.detach(), L.detach(), None, host_seed(11), 0)
        e64 = solve_eps(L64.detach(), theta, mean)
    ref = opolicy.sample(True, m64, torch.tril(L64), times.double(), init_time.double(), init_pos.double(),
                         init_vel.double(), eps=e64)
    assert_close(traj, ref, TRAJ_TOL, "trajectory")
    refs = torch.autograd.grad((ref * w.double()).sum(), wrt)
    with Launches("tce_mvn_rsample", "tce_prodmp_traj_bwd") as bwd:
        traj.backward(c(w))
    assert bwd.delta == {"tce_mvn_rsample": int(noise == "philox"), "tce_prodmp_traj_bwd": 1}
    assert_close(m.grad, refs[0], RSAMPLE_TOL, "d/dmean")
    if fac == "shared":
        assert_close(pol.variance_net.variable.grad, refs[1], RSAMPLE_TOL, "d/d covariance vector")
    else:
        assert_close(L.grad, refs[1], RSAMPLE_TOL, "d/dL")
        assert L.grad.triu(1).abs().max().item() == 0.0
    if noise == "injected":
        assert_close(e.grad, refs[2], RSAMPLE_TOL, "d/deps")


@pytest.mark.parametrize("D,K1", list(SHAPES))
@pytest.mark.parametrize("noise", ["injected", "philox"])
def test_sample_trajectories_gradients(D, K1, noise):
    """ProDMP.sample_trajectories with two samples per episode: the second sample's draws come from offset + 1, and
    the backward regenerates each sample's own draws.  B = 33 per-episode factors (bulk + 1 tail at n = 63); the 66
    flattened episodes share one grid and synthesise on the uniform kernel."""
    task = SHAPES[(D, K1)]
    cfg, T = dict(MP_CONFIGS[task], num_dof=D, num_basis=K1 - 1), NUM_TIMES[task]
    n, B, S, seed, offset = D * K1, 33, 2, 77, 3
    g = gen(n)
    mean, eps = 0.5 * torch.randn(B, n, generator=g), torch.randn(S, B, n, generator=g)
    L_host = factor(n, B, g)
    init_pos, init_vel = torch.rand(B, D, generator=g) * 2 - 1, 0.1 * torch.randn(B, D, generator=g)
    init_time = torch.zeros(B)
    times = ou.get_times(init_time.double(), T, cfg["dt"]).float()
    wp, wv = torch.randn(B, S, T, D, generator=g), torch.randn(B, S, T, D, generator=g)
    c = lambda t: t.to(DEV)
    m, L = c(mean).requires_grad_(True), c(L_host).requires_grad_(True)
    e = c(eps).requires_grad_(True) if noise == "injected" else None
    shim = ProDMP(ops.Tables(**cfg))
    with Launches("tce_mvn_rsample", "tce_prodmp_traj_fwd_uniform") as fwd:
        pos, vel = shim.sample_trajectories(times=c(times), params=m, params_L=L, init_time=c(init_time),
                                            init_pos=c(init_pos), init_vel=c(init_vel), num_smp=S, eps=e, seed=seed,
                                            offset=offset)
    assert fwd.delta == {"tce_mvn_rsample": S, "tce_prodmp_traj_fwd_uniform": 1}
    m64, L64 = mean.double().requires_grad_(True), L_host.double().requires_grad_(True)
    wrt = [m64, L64]
    if noise == "injected":
        e64 = eps.double().requires_grad_(True)
        wrt.append(e64)
    else:
        e64 = torch.stack([solve_eps(L_host.double(), ops.mvn_rsample(c(mean), c(L_host), None, seed, offset + s), mean)
                           for s in range(S)])
        assert (e64[0] - e64[1]).abs().max().item() > 0.1
    omp = oracle_get_mp(type="prodmp", args=dict(cfg, dtype=torch.float64))
    pos64, vel64 = omp.sample_trajectories(times=times.double(), params=m64, params_L=torch.tril(L64),
                                           init_time=init_time.double(), init_pos=init_pos.double(),
                                           init_vel=init_vel.double(), num_smp=S, eps=e64)
    assert_close(pos, pos64, TRAJ_TOL, "pos")
    assert_close(vel, vel64, TRAJ_TOL, "vel")
    refs = torch.autograd.grad((pos64 * wp.double()).sum() + (vel64 * wv.double()).sum(), wrt)
    with Launches("tce_mvn_rsample") as bwd:
        ((pos * c(wp)).sum() + (vel * c(wv)).sum()).backward()
    assert bwd.delta["tce_mvn_rsample"] == (S if noise == "philox" else 0)
    assert_close(m.grad, refs[0], RSAMPLE_TOL, "d/dmean")
    assert_close(L.grad, refs[1], RSAMPLE_TOL, "d/dL")
    assert L.grad.triu(1).abs().max().item() == 0.0
    if noise == "injected":
        assert_close(e.grad, refs[2], RSAMPLE_TOL, "d/deps")


# ---- C. trajectory gradients w.r.t. every input --------------------------------------------------------------------
# Table tennis's settings (0.3 s delay, tau 0.75, T = 350) with the shape and goal handling of each case.  Per-episode
# start times spread over [0, 0.6] s, so about half the episodes start before the delay (s clamped to 0, as in the
# oracle); the common grid starts at 0.2 s for all 64 episodes (B >= 64: the uniform forward kernel).
TRAJ_SHAPES = [(3, k) for k in range(2, 17)] + [(d, k) for d in (1, 7, 8) for k in (2, 4, 9, 16)]
GOALS = {"absolute": dict(relative_goal=False, relative_goal_scaled=False),
         "relative": dict(relative_goal=True, relative_goal_scaled=False),
         "relative_scaled": dict(relative_goal=True, relative_goal_scaled=True)}


def traj_case(D, K1, B, seed, init_time, **mp):
    cfg = dict(MP_CONFIGS["table_tennis"], num_dof=D, num_basis=K1 - 1, **mp)
    g = gen(seed)
    params = 0.5 * torch.randn(B, D * K1, generator=g)
    init_pos, init_vel = torch.rand(B, D, generator=g) * 2 - 1, 0.1 * torch.randn(B, D, generator=g)
    if init_time is None:
        init_time = torch.rand(B, generator=g) * 0.6
        init_time[:2] = torch.tensor([0.0, 0.3])
    else:
        init_time = torch.full((B,), float(init_time))
    return cfg, params, init_time, init_pos, init_vel


@pytest.mark.parametrize("auto_scale", [True, False])
@pytest.mark.parametrize("goal", list(GOALS))
@pytest.mark.parametrize("D,K1", TRAJ_SHAPES)
def test_trajectory_gradients_match_oracle(D, K1, goal, auto_scale):
    """prodmp_traj forward and d/dparams, d/dinit_pos, d/dinit_vel (traj_bwd_kernel, including its relative-goal
    branch) against autograd of the oracle, on per-episode start times (general kernel) and a common grid (uniform)."""
    T = NUM_TIMES["table_tennis"]
    for grid, B, start in (("episode", 24, None), ("common", 64, 0.2)):
        cfg, params, init_time, init_pos, init_vel = traj_case(D, K1, B, 100 * D + K1, start, auto_scale_basis=auto_scale,
                                                               **GOALS[goal])
        times = ou.get_times(init_time.double(), T, cfg["dt"]).float()
        w = torch.randn(B, T, 2 * D, generator=gen(K1))
        tabs = ops.Tables(**cfg)
        p, ip, iv = (t.to(DEV).requires_grad_(True) for t in (params, init_pos, init_vel))
        entry = "tce_prodmp_traj_fwd_uniform" if grid == "common" else "tce_prodmp_traj_fwd"
        with Launches(entry, "tce_prodmp_traj_bwd") as n_l:
            poison((B, T, 2 * D))
            traj = ops.prodmp_traj(p, times.to(DEV), init_time.to(DEV), ip, iv, tabs.handle, D)
            traj.backward(w.to(DEV))
        assert n_l.delta == {entry: 1, "tce_prodmp_traj_bwd": 1}
        p64, ip64, iv64 = (t.double().requires_grad_(True) for t in (params, init_pos, init_vel))
        ref = oracle_traj(cfg, p64, times.double(), init_time.double(), ip64, iv64)
        assert_close(traj, ref, TRAJ_TOL, f"{grid}: trajectory")
        gp, gy, gv = torch.autograd.grad((ref * w.double()).sum(), [p64, ip64, iv64])
        assert_close(p.grad, gp, TRAJ_TOL, f"{grid}: d/dparams")
        assert_close(ip.grad, gy, TRAJ_TOL, f"{grid}: d/dinit_pos")
        assert_close(iv.grad, gv, TRAJ_TOL, f"{grid}: d/dinit_vel")


# ---- D. store paths and tails --------------------------------------------------------------------------------------
# General kernel (a warp per 32-step slab): 128-bit stores when the slab's nt * 2D floats and its offset (b T + t0) 2D
# are multiples of 4, scalar stores otherwise.  Even D: always 128-bit.  Odd D: scalar for an odd tail slab (T = 1, 31,
# 33, 101: nt = 1, 31, 1, 5) and, at odd T, for every slab of an odd episode; T = 32 is all 128-bit.
# Uniform kernel (20-step tiles): 128-bit when nt * 2D, (b0 T + t0) 2D and T * 2D are multiples of 4.  Even D: always.
# Odd D: scalar at odd T (1, 31, 33, 101); T = 32 (tiles of 20 and 12 steps, epc even) is 128-bit.  Tiles: T = 1 one
# step; 31 = 20 + 11, 32 = 20 + 12, 33 = 20 + 13, 101 = 5 x 20 + 1.  B = 67 at epc 4: 17 groups, the last of 3.
@pytest.mark.parametrize("T", [1, 31, 32, 33, 101])
@pytest.mark.parametrize("D,K1", [(7, 4), (1, 5), (4, 9), (8, 3)])
def test_trajectory_store_paths_and_tails(D, K1, T):
    B = 67
    results = {}
    for name, start, uniform in (("general", None, False), ("general_common", 0.1, False), ("uniform", 0.1, True)):
        cfg, params, init_time, init_pos, init_vel = traj_case(D, K1, B, 7 * T + D, start)
        times = ou.get_times(init_time.double(), T, cfg["dt"]).float()
        tabs = ops.Tables(**cfg)
        entry = "tce_prodmp_traj_fwd_uniform" if uniform else "tce_prodmp_traj_fwd"
        ops.UNIFORM_TRAJ = uniform
        try:
            with Launches(entry) as n_l:
                poison((B, T, 2 * D))
                traj = ops.prodmp_traj(*(t.to(DEV) for t in (params, times, init_time, init_pos, init_vel)),
                                       tabs.handle, D)
        finally:
            ops.UNIFORM_TRAJ = True
        assert n_l.delta == {entry: 1}
        ref = oracle_traj(cfg, params.double(), times.double(), init_time.double(), init_pos.double(),
                          init_vel.double())
        assert_close(traj, ref, TRAJ_TOL, name)
        results[name] = traj
    assert_close(results["uniform"], f64(results["general_common"]), UNIFORM_VS_GENERAL, "uniform vs general")


# ---- E. large batches ----------------------------------------------------------------------------------------------
# Uniform kernel on 148 SMs: epc = 16, halved while ceil(B / epc) < 2 x 148 = 296 and epc > 4:
#   B = 64, 2360 -> 4;  2361 (296 groups of 8), 4720 (590 of 8) -> 8;  4721 (296 of 16) -> 16;
#   20001 -> 16 with 1251 groups > 8 x 148 = 1184 CTAs: the group loop strides, and its last group holds one episode.
UNIFORM_EPC = {64: 4, 2360: 4, 2361: 8, 4720: 8, 4721: 16, 20001: 16}


def oracle_subset(B, epc, seed):
    """First and last 64 episodes, the last group, and 64 random ones."""
    last = (B - 1) // epc * epc
    idx = set(range(min(64, B))) | set(range(max(0, B - 64), B)) | set(range(last, B))
    idx |= set(torch.randint(0, B, (64,), generator=gen(seed)).tolist())
    return torch.tensor(sorted(idx))


@pytest.mark.parametrize("B", list(UNIFORM_EPC))
@pytest.mark.parametrize("name", ["box", "metaworld", "table_tennis"])
def test_uniform_kernel_batch_regimes(name, B):
    cfg, T = MP_CONFIGS[name], NUM_TIMES[name]
    D, K1 = cfg["num_dof"], cfg["num_basis"] + 1
    epc, _ = ops.traj_uniform_layout(B, T, D, K1, sms())
    if sms() == B200_SMS:
        assert epc == UNIFORM_EPC[B] and (-(-B // epc) > 8 * B200_SMS) == (B == 20001)
    g = gen(B)
    params = 0.5 * torch.randn(B, D * K1, generator=g)
    init_pos, init_vel = torch.rand(B, D, generator=g) * 2 - 1, 0.1 * torch.randn(B, D, generator=g)
    init_time = torch.zeros(B)
    times = ou.get_times(init_time.double(), T, cfg["dt"]).float()
    tabs = ops.Tables(**cfg)                            # owns the device tables: alive until the kernels have run
    args = [t.to(DEV) for t in (params, times, init_time, init_pos, init_vel)] + [tabs.handle, D]
    with Launches("tce_prodmp_traj_fwd_uniform") as n_l:
        poison((B, T, 2 * D))
        fast = ops.prodmp_traj(*args)
    assert n_l.delta["tce_prodmp_traj_fwd_uniform"] == 1
    ops.UNIFORM_TRAJ = False
    try:
        poison((B, T, 2 * D))
        general = ops.prodmp_traj(*args)
    finally:
        ops.UNIFORM_TRAJ = True
    assert bool(torch.isfinite(fast).all()) and bool(torch.isfinite(general).all())
    scale = general.abs().max().item()
    assert (fast - general).abs().max().item() <= UNIFORM_VS_GENERAL * scale
    idx = oracle_subset(B, epc, B)
    ref = oracle_traj(cfg, params[idx].double(), times[idx].double(), init_time[idx].double(),
                      init_pos[idx].double(), init_vel[idx].double())
    assert_close(fast[idx.to(DEV)], ref, TRAJ_TOL, "uniform vs oracle")


# General kernel: one warp per (episode, 32-step slab), 8 warps per CTA, at most 8 x 148 CTAs = 9472 warps: box at
# B = 3001 (T = 100: 12004 slabs) and metaworld at B = 700 (T = 500: 11200 slabs) run the slab loop twice.
@pytest.mark.parametrize("name,B", [("box", 3001), ("metaworld", 700)])
def test_general_kernel_grid_stride(name, B):
    cfg, T = MP_CONFIGS[name], NUM_TIMES[name]
    D, K1 = cfg["num_dof"], cfg["num_basis"] + 1
    assert B * -(-T // 32) > 8 * 8 * B200_SMS
    g = gen(B)
    params = 0.5 * torch.randn(B, D * K1, generator=g)
    init_pos, init_vel = torch.rand(B, D, generator=g) * 2 - 1, 0.1 * torch.randn(B, D, generator=g)
    init_time = torch.rand(B, generator=g) * 0.5
    times = ou.get_times(init_time.double(), T, cfg["dt"]).float()
    tabs = ops.Tables(**cfg)
    with Launches("tce_prodmp_traj_fwd") as n_l:
        poison((B, T, 2 * D))
        traj = ops.prodmp_traj(*(t.to(DEV) for t in (params, times, init_time, init_pos, init_vel)), tabs.handle, D)
    assert n_l.delta["tce_prodmp_traj_fwd"] == 1
    ref = oracle_traj(cfg, params.double(), times.double(), init_time.double(), init_pos.double(), init_vel.double())
    assert_close(traj, ref, TRAJ_TOL, "general vs oracle")


# ---- F. long horizons on one common grid ---------------------------------------------------------------------------
# D = 4, K1 = 16: 36 floats (144 B) of basis rows per step, plus an output tile of epc x 168 floats.  On 148 SMs the
# uniform kernel's 200 KB hold 144 T + 2688 B at B = 64 (epc 4): T <= 1403, and 144 T + 10752 B at B = 4721 (epc 16):
# T <= 1347.  Past that the general kernel serves the common grid.  dt = 0.005 s, tau = 2 s: the tables cover
# 5 tau = 10 s, T = 1500 steps 7.5 s.
LONG = dict(MP_CONFIGS["box"], num_dof=4, num_basis=15, tau=2.0, dt=0.005)


@pytest.mark.parametrize("B,T", [(64, 1403), (64, 1404), (64, 1500), (4721, 1347), (4721, 1348)])
def test_long_horizon_common_grid(B, T):
    D, K1 = 4, 16
    epc, smem = ops.traj_uniform_layout(B, T, D, K1, sms())
    uniform = smem <= ops.TRAJ_UNIFORM_SMEM
    if sms() == B200_SMS:
        assert uniform == (T in (1403, 1347))
    g = gen(T)
    params = 0.5 * torch.randn(B, D * K1, generator=g)
    init_pos, init_vel = torch.rand(B, D, generator=g) * 2 - 1, 0.1 * torch.randn(B, D, generator=g)
    init_time = torch.zeros(B)
    times = ou.get_times(init_time.double(), T, LONG["dt"]).float()
    tabs = ops.Tables(**LONG)
    assert (T - 1) * LONG["dt"] <= tabs.max_time()
    entry = "tce_prodmp_traj_fwd_uniform" if uniform else "tce_prodmp_traj_fwd"
    with Launches("tce_prodmp_traj_fwd_uniform", "tce_prodmp_traj_fwd") as n_l:
        poison((B, T, 2 * D))
        traj = ops.prodmp_traj(*(t.to(DEV) for t in (params, times, init_time, init_pos, init_vel)), tabs.handle, D)
    assert n_l.delta == {"tce_prodmp_traj_fwd_uniform": int(uniform), "tce_prodmp_traj_fwd": int(not uniform)}
    idx = oracle_subset(B, epc, T) if B > 64 else torch.arange(B)
    ref = oracle_traj(LONG, params[idx].double(), times[idx].double(), init_time[idx].double(),
                      init_pos[idx].double(), init_vel[idx].double())
    assert_close(traj[idx.to(DEV)], ref, TRAJ_TOL, entry)


@pytest.mark.parametrize("D,K1", COMPILED)
def test_compiled_shapes_keep_the_uniform_kernel(D, K1):
    """The five compiled shapes at their task's T take the uniform kernel on a common grid, at the smallest (epc 4)
    and the largest (epc 16) tile."""
    task = COMPILED_TASK[(D, K1)]
    cfg, T = dict(MP_CONFIGS[task], num_dof=D, num_basis=K1 - 1), NUM_TIMES[task]
    tabs = ops.Tables(**cfg)
    assert tabs.compiled
    for B in (64, 4721):
        assert ops.traj_uniform_layout(B, T, D, K1, sms())[1] <= ops.TRAJ_UNIFORM_SMEM
        times = ou.get_times(torch.zeros(B, dtype=torch.float64), T, cfg["dt"]).float().to(DEV)
        z = torch.zeros(B, D, device=DEV)
        with Launches("tce_prodmp_traj_fwd_uniform", "tce_prodmp_traj_fwd") as n_l:
            traj = ops.prodmp_traj(torch.randn(B, D * K1, device=DEV), times, torch.zeros(B, device=DEV), z, z,
                                   tabs.handle, D)
        assert n_l.delta == {"tce_prodmp_traj_fwd_uniform": 1, "tce_prodmp_traj_fwd": 0}
        assert bool(torch.isfinite(traj).all())

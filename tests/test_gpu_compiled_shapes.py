"""The five (num_dof, K1) shapes with specialised likelihood kernels, on every device route that accepts a case,
against the fp64 oracle (``TemporalCorrelatedPolicy.log_prob`` + autograd, ``oracle.agent.surrogate_loss``).

Routes of ``ops_seglik`` for these shapes:
* staged   : ``tce_seglik_gram`` / ``_chol`` / ``_bwd`` (per-episode factors, the default) and the shared-covariance
             staged kernels when the fused kernel refuses the segment count;
* fused    : ``tce_seglik_prepass`` + ``tce_seglik_fused`` (+ ``tce_seglik_dsigma_reduce`` for a shared covariance);
* uniform  : shared covariance on one time grid, ``tce_seglik_uniform_*``, for P (NT + 1) <= 12 * 256.

The segment counts sit on both sides of every limit that depends on P, the batch sizes on the batch edges of the
fused and the uniform launches, and which route ran is asserted by counting launches, so that a silent fallback
cannot pass as coverage.  Mode 1 also runs with one-hot upstream gradients (the first and the last segment): a
single segment's adjoints then determine the whole gradient, so a lost or misindexed adjoint cannot average out.

Tolerances (north star): log-probs <= 1e-4 absolute, gradients <= 2e-4 of their largest entry."""
import pytest
import torch

from oracle import agent as oa
from oracle import policy as opol
from oracle import util as ou
from oracle.gen_golden import MP_CONFIGS, NUM_TIMES
from test_gpu_any_shape import f64, inputs
from test_gpu_kernels import _lib_launch_count

pytestmark = pytest.mark.gpu
if torch.cuda.is_available():
    from tce_rl_b200 import ops, ops_seglik
    from tce_rl_b200._lib import TceError

DEV = "cuda:0"
# (num_dof, K1) -> the task whose MP settings it runs with: the three shipped configs, (3, 4) with table tennis's
# relative goal, delay and T = 350, (2, 3) with metaworld's T = 500 (room for P past the uniform and fused limits)
TASK = {(7, 9): "box", (4, 9): "metaworld", (7, 4): "table_tennis", (3, 4): "table_tennis", (2, 3): "metaworld"}
SHAPES = list(TASK)
FUSED_MAX_P = 256                                        # threads of the fused kernel: one segment slot per thread
UNIFORM_SLOTS = 12 * 256                                 # the uniform kernels take P * (NT + 1) <= this
ENTRIES = {"staged": ("tce_seglik_gram", "tce_seglik_gram_sigma"), "fused": ("tce_seglik_fused",),
           "uniform": ("tce_seglik_uniform_main",)}


def tri(n):
    return n * (n + 1) // 2


def mp_cfg(D, K1):
    task = TASK[(D, K1)]
    return dict(MP_CONFIGS[task], num_dof=D, num_basis=K1 - 1), NUM_TIMES[task]


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def chained_pairs(T, P):
    torch.manual_seed(P)
    pairs = ou.get_time_pairs(T, dict(num_select=P + 1, fixed_interval=True))[:P]
    assert pairs.shape == (P, 2)
    return pairs


def ragged_pairs(T):
    """Seven non-chained pairs with repeats: the first and last time point, a long and a one-step segment."""
    return torch.tensor([[0, 1], [0, T - 1], [5, 50], [T - 2, T - 1], [10, 11], [11, 12], [40, 80]])


def test_the_five_shapes_are_compiled():
    for D, K1 in SHAPES:
        cfg, _ = mp_cfg(D, K1)
        assert ops.Tables(**cfg).compiled, (D, K1)
    for name in ("box", "metaworld", "table_tennis"):
        D, K1 = MP_CONFIGS[name]["num_dof"], MP_CONFIGS[name]["num_basis"] + 1
        assert TASK[(D, K1)] == name and mp_cfg(D, K1)[0] == MP_CONFIGS[name]


@pytest.mark.parametrize("D,K1", SHAPES)
def test_route_limits(D, K1):
    """The uniform kernels accept every P with P (NT + 1) <= 12 * 256 at every batch size, on both sides of the
    switch from 8 to 32 episodes per CTA; the fused kernel refuses P > 256."""
    cfg, T = mp_cfg(D, K1)
    tabs = ops.Tables(**cfg)
    pmax = UNIFORM_SLOTS // (tri(2 * D) + 1)
    for B in (1, 8 * sms(), 8 * sms() + 1):
        for P in (1, pmax):
            assert ops_seglik.uniform_config(tabs.handle, B, P)["uni_parts"] > 0, (B, P)
        assert ops_seglik.uniform_config(tabs.handle, B, pmax + 1)["uni_parts"] == 0
    with pytest.raises(TceError):
        ops_seglik.fused_config(tabs.handle, 4, FUSED_MAX_P + 1, True)


# ---- oracle ---------------------------------------------------------------------------------------------------------
class Case:
    """One shape, batch and pair set on one kind of time grid: inputs, sample and the oracle's answers for every
    covariance layout asked for."""

    def __init__(self, D, K1, B, pairs, one_grid, one_hot, seed=5):
        self.D, self.K1, self.B, self.Dp = D, K1, B, D * K1
        self.cfg, self.T = mp_cfg(D, K1)
        self.inp = inp = inputs(D, K1, B, seed=seed)
        if one_grid:
            inp["init_time"] = inp["init_time"][:1].expand(B).contiguous()
        self.times = ou.get_times(inp["init_time"].double(), self.T, self.cfg["dt"]).float()
        self.pairs, self.P = pairs, pairs.shape[0]
        self.pol = opol.TemporalCorrelatedPolicy(self.Dp, mp=dict(type="prodmp", args=dict(self.cfg,
                                                                                             dtype=torch.float64)),
                                                 contextual=True)
        d = lambda k: inp[k].double()
        self.args64 = (self.times.double(), d("init_time"), d("init_pos"), d("init_vel"))
        self.smp = self.pol.sample(False, d("mean"), d("L"), *self.args64, eps=d("eps")).float()
        self.S = inp["L"][0].double() @ inp["L"][0].double().T
        P = self.P
        # upstreams and advantages are fp32 values: the kernels and the oracle see the same numbers
        self.upstreams = {"w": torch.linspace(0.5, 1.5, B * P).reshape(B, P).double()}
        if one_hot:
            for p in sorted({0, P - 1}):
                e = torch.zeros(B, P, dtype=torch.float64)
                e[:, p] = 1.0
                self.upstreams[f"e{p}"] = e
        self.adv = torch.randn(B, P, generator=torch.Generator().manual_seed(2)).double()

    def oracle(self, cov):
        """-> dict: lp, reg, grads[upstream] = (d/d mean, d/d cov), surrogate (loss, ratio, d/d mean, d/d cov),
        lp_old.  ``cov``: episode (per-episode L), shared_L (one L) or shared_sigma (one Sigma)."""
        B, inp = self.B, self.inp
        mean64 = inp["mean"].double().requires_grad_(True)
        if cov == "episode":
            wrt = inp["L"].double().requires_grad_(True)
            Lo = wrt
        elif cov == "shared_L":
            wrt = inp["L"][:1].double().requires_grad_(True)
            Lo = wrt.expand(B, -1, -1)
        else:
            wrt = self.S.clone().requires_grad_(True)
            Lo = torch.linalg.cholesky(0.5 * (wrt + wrt.T)).expand(B, -1, -1)
        lp, _, _, reg = self.pol.log_prob(self.smp.double(), mean64, Lo, *self.args64, pred_pairs=self.pairs,
                                          return_parts=True)
        # a factor's free entries are its lower triangle: the kernels return tril(d lp / d L)
        free = (lambda g: g) if cov == "shared_sigma" else torch.tril
        out = dict(lp=lp.detach(), reg=reg, grads={})
        for k, g in self.upstreams.items():
            gm, gc = torch.autograd.grad((lp * g).sum(), [mean64, wrt], retain_graph=True)
            out["grads"][k] = (gm, free(gc))
        lp_old = (lp.detach() + 0.1 * torch.randn(lp.shape, generator=torch.Generator().manual_seed(1),
                                                  dtype=torch.float64)).float().double()
        loss, parts = oa.surrogate_loss(self.adv, lp, lp_old)
        gm, gc = torch.autograd.grad(loss, [mean64, wrt])
        out["surrogate"] = (loss.item(), parts["imp_smp_ratio"].item(), gm, free(gc))
        out["lp_old"] = lp_old
        return out


# ---- device -------------------------------------------------------------------------------------------------------
class Routed:
    """Counts the launches of every route's entry points over a block; ``ran`` is the set of routes that launched."""

    def __enter__(self):
        self.n0 = {r: sum(_lib_launch_count(e) for e in es) for r, es in ENTRIES.items()}
        return self

    def __exit__(self, *exc):
        self.ran = {r for r, es in ENTRIES.items() if sum(_lib_launch_count(e) for e in es) > self.n0[r]}


def expected_route(case, cov, per_episode_staged, one_grid, tabs):
    shared = cov != "episode" or case.B == 1               # one per-episode factor is one shared factor
    if not shared and per_episode_staged:
        return "staged"
    if shared and one_grid and case.P * (tri(2 * case.D) + 1) <= UNIFORM_SLOTS:
        return "uniform"
    try:
        ops_seglik.fused_config(tabs.handle, case.B, case.P, ops_seglik.pairs_chained(case.pairs))
    except TceError:
        return "staged"
    return "fused"


def run_device(case, cov, tabs, one_grid, lp_old):
    """The public likelihood entry points on one covariance layout: log-probs (mode 0), their backward for every
    upstream (mode 1), the fused surrogate and its gradients (mode 2).  Asserts one route per call."""
    c = lambda t: t.to(DEV)
    inp, B = case.inp, case.B
    targs = (c(case.times), c(inp["init_time"]), c(inp["init_pos"]), c(inp["init_vel"]), c(case.pairs), tabs)
    uniform = one_grid and cov != "episode"

    def leaves():
        mean = c(inp["mean"]).requires_grad_(True)
        if cov == "episode":
            cv = c(inp["L"]).requires_grad_(True)
            return mean, cv, cv, None
        if cov == "shared_L":
            cv = c(inp["L"][:1]).requires_grad_(True)
            return mean, cv, cv, None
        cv = c(case.S / 2.0).requires_grad_(True)              # Sigma = 2 * (S / 2): d / d Sigma comes back
        return mean, cv, c(inp["L"][:1]), (cv, torch.full((1,), 2.0, device=DEV, dtype=torch.float64))

    out, ran = {"grads": {}}, set()
    mean, cv, L, sigma = leaves()
    with torch.no_grad(), Routed() as r:
        lp, info, dmax = ops_seglik.seg_logprob(c(case.smp), mean, L, *targs, return_info=True, uniform=uniform,
                                                sigma=sigma)
    ran |= r.ran
    out.update(lp=f64(lp), info=info, dmax=dmax.reshape(-1)[0].item())
    for k, g in case.upstreams.items():
        mean, cv, L, sigma = leaves()
        with Routed() as r:
            lp = ops_seglik.seg_logprob(c(case.smp), mean, L, *targs, uniform=uniform, sigma=sigma)
            (lp * c(g.float())).sum().backward()
        ran |= r.ran
        out["grads"][k] = (f64(mean.grad), f64(cv.grad))
        if cov != "shared_sigma":
            assert float(cv.grad.triu(1).abs().max()) == 0.0
    mean, cv, L, sigma = leaves()
    with Routed() as r:
        loss, ratio, lp2 = ops_seglik.seg_surrogate(c(case.smp), mean, L, *targs[:5], c(lp_old.float()),
                                                    c(case.adv.float()), tabs, uniform=uniform, sigma=sigma)
        loss.backward()
    ran |= r.ran
    out["surrogate"] = (loss.item(), ratio.item(), f64(mean.grad), f64(cv.grad))
    out["lp2"] = f64(lp2)
    out["ran"] = ran
    return out


def close(got, want, rel):
    return (got - want).abs().max().item() <= rel * want.abs().max().item()


def check_against_oracle(got, ref, cov):
    assert int(got["info"].abs().max()) == 0
    assert (got["lp"] - ref["lp"]).abs().max() <= 1e-4
    assert (got["lp2"] - ref["lp"]).abs().max() <= 1e-4
    # the regulariser: 1e-4 x the batch-global max of the un-regularised diagonal of C
    assert abs(1e-4 * got["dmax"] - ref["reg"]) <= 1e-6 * ref["reg"]
    for k, (gm_ref, gc_ref) in ref["grads"].items():
        gm, gc = got["grads"][k]
        assert close(gm, gm_ref, 2e-4), (cov, k, "grad_mean")
        gc = gc.reshape(gc_ref.shape)
        err = (gc - gc_ref).abs()
        assert err.max().item() <= 2e-4 * gc_ref.abs().max().item(), \
            (cov, k, "grad_cov", err.max().item(), gc_ref.abs().max().item(), (err.amax(-1) > 2e-4 *
                                                                                 gc_ref.abs().max()).nonzero()[:8])
    loss_ref, ratio_ref, gm_ref, gc_ref = ref["surrogate"]
    loss, ratio, gm, gc = got["surrogate"]
    assert abs(loss - loss_ref) <= 1e-4 * max(1.0, abs(loss_ref))
    assert abs(ratio - ratio_ref) <= 1e-4
    assert close(gm, gm_ref, 2e-4), (cov, "surrogate grad_mean")
    assert close(gc.reshape(gc_ref.shape), gc_ref, 2e-4), (cov, "surrogate grad_cov")


def run_case(D, K1, B, P, routes=("episode", "shared_L", "shared_sigma"), grids=(False, True)):
    """P: a segment count (chained pairs) or "ragged".  Every covariance layout in ``routes`` on every grid in
    ``grids`` (False: per-episode start times, True: one time grid); per-episode factors run on the staged and on
    the fused kernels and the two are also compared with each other.  Small batches also take the one-hot upstreams
    (the oracle's graph grows with B P Dp^2 and is kept for every upstream)."""
    cfg, T = mp_cfg(D, K1)
    tabs = ops.Tables(**cfg)
    pairs = ragged_pairs(T) if P == "ragged" else chained_pairs(T, P)
    for one_grid in grids:
        case = Case(D, K1, B, pairs, one_grid, one_hot=B <= 64)
        for cov in routes:
            if cov == "episode" and one_grid:
                continue
            ref = case.oracle(cov)
            outs = []
            for staged in ((True, False) if cov == "episode" else (ops_seglik.PER_EPISODE_STAGED,)):
                old = ops_seglik.PER_EPISODE_STAGED
                ops_seglik.PER_EPISODE_STAGED = staged
                try:
                    got = run_device(case, cov, tabs, one_grid, ref["lp_old"])
                finally:
                    ops_seglik.PER_EPISODE_STAGED = old
                assert got["ran"] == {expected_route(case, cov, staged, one_grid, tabs)}, (cov, staged, got["ran"])
                check_against_oracle(got, ref, cov)
                outs.append(got)
            if len(outs) == 2:
                # staged == fused on the weighted batch gradient, at test_fused_equals_staged's bounds.  A one-hot
                # gradient is one segment's, whose C is far worse conditioned at large P: each path stays within the
                # oracle's bound there, but they round differently by more than these.
                a, b = outs
                assert (a["lp"] - b["lp"]).abs().max() <= 2e-5
                assert close(b["grads"]["w"][0], a["grads"]["w"][0], 2e-5)
                assert close(b["grads"]["w"][1], a["grads"]["w"][1], 5e-5)


COMMON = [(1, 1), (3, 2), (36, 24), (37, 25), (3, "ragged")]
EDGES = {
    (7, 9): [(5, 37), (4, 38), (3, 39), (4, 28), (5, 29), (3, 99)],
    (7, 4): [(5, 7), (4, 8), (3, 9), (4, 28), (5, 29), (3, 256), (3, 257), (3, 349)],
    (3, 4): [(5, 6), (3, 7), (4, 139), (5, 140), (4, 256), (3, 257)],
    (4, 9): [(3, 83), (4, 84), (4, 256), (3, 257)],
    (2, 3): [(4, 256), (3, 257), (5, 279), (4, 280)],
}
CASES = [(D, K1, B, P) for D, K1 in SHAPES for B, P in COMMON + EDGES[(D, K1)]]


@pytest.mark.parametrize("D,K1,B,P", CASES, ids=[f"{D}x{K1}-B{B}-P{P}" for D, K1, B, P in CASES])
def test_routes_match_oracle(D, K1, B, P):
    run_case(D, K1, B, P)


@pytest.mark.parametrize("D,K1", SHAPES)
def test_fused_batch_edge(D, K1):
    """B = E * grid + 1 on the fused kernel: every CTA loops over its episode groups and the last group holds one
    episode (per-episode factors on the fused kernel, a shared factor and a shared Sigma on per-episode grids)."""
    cfg, T = mp_cfg(D, K1)
    tabs = ops.Tables(**cfg)
    P = 25
    fc = ops_seglik.fused_config(tabs.handle, 1 << 20, P, True)
    assert fc["grid"] == sms()
    B = fc["E"] * fc["grid"] + 1
    assert ops_seglik.fused_config(tabs.handle, B, P, True)["grid"] == sms()
    run_case(D, K1, B, P, grids=(False,))


@pytest.mark.parametrize("D,K1", SHAPES)
@pytest.mark.parametrize("extra", [0, 1])
@pytest.mark.parametrize("at", ["P25", "uniform_limit"])
def test_uniform_batch_edge(D, K1, extra, at):
    """B = 8 SMs and 8 SMs + 1 on the uniform kernels, where they switch from 8 to 32 episodes per CTA, at P = 25
    and at the largest P they accept."""
    P = 25 if at == "P25" else UNIFORM_SLOTS // (tri(2 * D) + 1)
    run_case(D, K1, 8 * sms() + extra, P, routes=("shared_L", "shared_sigma"), grids=(True,))


@pytest.mark.parametrize("D,K1", [(3, 4), (2, 3)])
@pytest.mark.parametrize("B,P", [(5, 24), (3, 25), (1, 1), (4, "ragged")])
def test_diagonal_covariance(D, K1, B, P):
    """seg_logprob_diag (std_only policies): forward and backward against the oracle on diagonal factors."""
    cfg, T = mp_cfg(D, K1)
    Dp = D * K1
    tabs = ops.Tables(**cfg)
    pairs = ragged_pairs(T) if P == "ragged" else chained_pairs(T, P)
    inp = inputs(D, K1, B, seed=11)
    s = torch.exp(0.3 * torch.randn(B, Dp, generator=torch.Generator().manual_seed(3)))
    inp["L"] = torch.diag_embed(s).float()
    times = ou.get_times(inp["init_time"].double(), T, cfg["dt"]).float()
    pol = opol.TemporalCorrelatedPolicy(Dp, mp=dict(type="prodmp", args=dict(cfg, dtype=torch.float64)),
                                        contextual=True, std_only=True, min_std=1e-4)
    d = lambda k: inp[k].double()
    args64 = (times.double(), d("init_time"), d("init_pos"), d("init_vel"))
    smp = pol.sample(False, d("mean"), d("L"), *args64, eps=d("eps")).float()
    mean64, L64 = d("mean").requires_grad_(True), d("L").requires_grad_(True)
    lp = pol.log_prob(smp.double(), mean64, L64, *args64, pred_pairs=pairs)
    c = lambda t: t.to(DEV)
    args = (c(times), c(inp["init_time"]), c(inp["init_pos"]), c(inp["init_vel"]), c(pairs), tabs)
    n = lp.shape[1]
    ups = [torch.linspace(0.5, 1.5, lp.numel(), dtype=torch.float64).reshape(lp.shape)]
    for p in sorted({0, n - 1}):
        e = torch.zeros(lp.shape, dtype=torch.float64)
        e[:, p] = 1.0
        ups.append(e)
    for i, w in enumerate(ups):
        gm_ref, gL_ref = torch.autograd.grad((lp * w).sum(), [mean64, L64], retain_graph=True)
        gL_ref = gL_ref.diagonal(dim1=-2, dim2=-1)
        mean_g, L_g = c(inp["mean"]).requires_grad_(True), c(inp["L"]).requires_grad_(True)
        got, info, _ = ops_seglik.seg_logprob_diag(c(smp), mean_g, L_g, *args, return_info=True)
        if i == 0:
            assert got.shape == lp.shape and int(info.abs().max()) == 0
            assert (f64(got) - lp.detach()).abs().max() <= 1e-4
        (got * c(w.float())).sum().backward()
        assert close(f64(mean_g.grad), gm_ref, 2e-4), i
        gd = f64(L_g.grad)
        assert close(gd.diagonal(dim1=-2, dim2=-1), gL_ref, 2e-4), i
        assert float((gd - torch.diag_embed(gd.diagonal(dim1=-2, dim2=-1))).abs().max()) == 0.0

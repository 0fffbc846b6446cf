"""Generate the golden fixtures under ``tests/golden`` by running the REAL reference code.

TEST INFRASTRUCTURE ONLY.  Run in the build container (``/root/reference`` present):

    python -m oracle.gen_golden

What is produced (all tiny, float64 unless the reference's own test uses float32):
* ``ref_util.pt``   -- outputs of the reference's ``mprl.util`` helpers on the inputs of its own
                       known-answer tests (mprl/test/util_test/util_matrix_test.py:7-105,
                       util_numerical_test.py:19-36) plus ``select_pred_pairs`` for seeds 0..4 and
                       T in {100, 350, 360, 500} (bit-exact integer goldens).
* ``ref_agent.pt``  -- ``TemporalCorrelatedAgent.get_advantage_return`` / ``get_segment_advantage``
                       (all three modes) / ``surrogate_loss`` / ``value_loss`` on seeded inputs.
* ``ref_policy.pt`` -- the reference's ``TemporalCorrelatedPolicy`` (built by ``policy_factory`` with
                       the box-pushing config; its ``mp`` is the oracle ProDMP through the shim in
                       ``oracle/ref_loader.py``) : policy(), Gaussian helpers, sample(use_mean),
                       log_prob -- pins the tensor plumbing of the oracle policy.
* ``oracle_path.pt`` -- oracle-generated (PARITY UNPINNED) ProDMP tables for three MP shapes.
"""
from __future__ import annotations

import os
import sys

import torch

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")

MP_CONFIGS = {
    # mprl/config/box_push_random_init/tcp/entire/shared.yaml:53-70
    "box": dict(num_dof=7, tau=2.0, alpha_phase=3, num_basis=8, basis_bandwidth_factor=3, num_basis_outside=0,
                alpha=10, relative_goal=False, auto_scale_basis=True, weights_scale=0.3, goal_scale=0.3,
                dt=0.02),
    # mprl/config/metaworld/tcp/entire/shared.yaml:53-70
    "metaworld": dict(num_dof=4, tau=5.0, alpha_phase=3, num_basis=8, basis_bandwidth_factor=5,
                      num_basis_outside=0, alpha=10, relative_goal=True, auto_scale_basis=True,
                      weights_scale=0.1, goal_scale=0.1, dt=0.0125),
    # mprl/config/table_tennis_4d/tcp/entire/shared.yaml:53-73
    "table_tennis": dict(num_dof=7, tau=0.75, delay=0.3, alpha_phase=3, num_basis=3, basis_bandwidth_factor=3,
                         num_basis_outside=0, alpha=25, relative_goal=True, auto_scale_basis=True,
                         weights_scale=0.7, goal_scale=0.1, dt=0.008),
}
NUM_TIMES = {"box": 100, "metaworld": 500, "table_tennis": 350}


def synthetic_inputs(name: str, B: int, seed: int = 1234, dtype=torch.float64):
    """Synthetic tensors of SURVEY 8(d) (same draw order for every consumer)."""
    cfg = MP_CONFIGS[name]
    D, K1 = cfg["num_dof"], cfg["num_basis"] + 1
    Dp, T = D * K1, NUM_TIMES[name]
    g = torch.Generator().manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    mean = 0.5 * rn(B, Dp)
    L = torch.tril(0.05 * rn(B, Dp, Dp), -1) + torch.diag_embed(torch.nn.functional.softplus(rn(B, Dp)) + 1e-4)
    mean_old = mean + 0.05 * rn(B, Dp)
    L_old = 1.05 * L + torch.tril(0.01 * rn(B, Dp, Dp), -1)
    init_time = torch.zeros(B, dtype=torch.float64)
    init_pos = torch.rand(B, D, generator=g, dtype=torch.float64) * 2 - 1
    init_vel = 0.1 * rn(B, D)
    eps = rn(B, Dp)
    rewards, values = rn(B, T), rn(B, T + 1)
    dones = torch.zeros(B, T, dtype=torch.bool)
    dones[:, -1] = True
    out = dict(mean=mean, L=L, mean_old=mean_old, L_old=L_old, init_time=init_time, init_pos=init_pos,
               init_vel=init_vel, eps=eps, rewards=rewards, values=values, dones=dones,
               time_limit_dones=torch.zeros(B, T, dtype=torch.bool))
    return {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in out.items()}


def gen_ref_util(util):
    g = {}
    diag = torch.ones(6) * 0.5
    off = torch.arange(1, 16, dtype=torch.float32)
    L = util.build_lower_matrix(diag, off)
    g["build_lower_matrix"] = dict(diag=diag, off=off, L=L)
    d2, o2 = util.reverse_build_matrix(L, True)
    g["reverse_build_matrix"] = dict(diag=d2, off=o2)
    x = torch.arange(24, dtype=torch.float64).reshape(2, 3, 4)
    g["add_expand_dim"] = dict(x=x, a=util.add_expand_dim(x, [1, 3, 5], [2, 3, 5]).contiguous(),
                               b=util.add_expand_dim(x, [1, -3, -1], [2, 3, 5]).contiguous(),
                               c=util.add_expand_dim(x, [-2], [7]).contiguous())
    end = torch.arange(0, 11, dtype=torch.float64)
    g["tensor_linspace"] = dict(end=end, out=util.tensor_linspace(0, end.clone(), 11))
    data = torch.arange(10, dtype=torch.float64)[:, None].expand(10, 2).contiguous()
    idx = torch.tensor([[0.5, 1.5, 2.5, 3.5, 4.5]] * 3, dtype=torch.float64)
    g["indexing_interpolate"] = dict(data=data, idx=idx, out=util.indexing_interpolate(data, idx))
    idx2 = torch.tensor([-0.3, 0.0, 8.2, 9.0, 9.7], dtype=torch.float64)
    g["indexing_interpolate_edge"] = dict(data=data, idx=idx2, out=util.indexing_interpolate(data, idx2))
    z = torch.tensor([0.0, -3.0, 2.5], dtype=torch.float64)
    g["softplus"] = dict(x=z, none=util.to_softplus_space(z, None), two=util.to_softplus_space(z, 2.0),
                         inv=util.reverse_from_softplus_space(util.to_softplus_space(z, None), None))
    pp = {}
    for T in (100, 350, 360, 500):
        for seed in range(5):
            torch.manual_seed(seed)
            pp[(T, seed)] = util.select_pred_pairs(num_all=T, num_select=25, fixed_interval=True).to(torch.long)
    torch.manual_seed(7)
    pp[("random", 7)] = util.select_pred_pairs(num_all=100, num_select=10, fixed_interval=False).to(torch.long)
    g["select_pred_pairs"] = pp
    init_time = torch.tensor([0.0, 0.3, 1.0], dtype=torch.float64)
    g["get_times"] = dict(init_time=init_time, dt=0.02, T=100,
                          out=util.tensor_linspace(init_time + 0.02, init_time + 100 * 0.02, 100).T.contiguous())
    return g


def gen_ref_agent(mprl):
    from types import SimpleNamespace
    from mprl.rl.agent.temporal_correlated_agent import TemporalCorrelatedAgent as A
    out = {}
    for tag, gamma, B, T in (("g1", 1.0, 6, 100), ("g099", 0.99, 5, 37)):
        g = torch.Generator().manual_seed(11)
        rewards = torch.randn(B, T, generator=g, dtype=torch.float64)
        values = torch.randn(B, T + 1, generator=g, dtype=torch.float64)
        dones = torch.zeros(B, T, dtype=torch.bool)
        dones[:, -1] = True
        dones[1, T // 2] = True
        tl = torch.zeros(B, T, dtype=torch.bool)
        tl[2, T // 3] = True
        torch.manual_seed(0)
        import mprl.util as util
        pairs = util.select_pred_pairs(num_all=T, num_select=min(25, T // 3), fixed_interval=True).to(torch.long)
        rec = dict(rewards=rewards, values=values, dones=dones, time_limit_dones=tl, pred_pairs=pairs,
                   gamma=gamma, lam=0.95)
        for use_gae in (True, False):
            me = SimpleNamespace(discount_factor=torch.tensor(gamma, dtype=torch.float64), use_gae=use_gae,
                                 gae_scaling=0.95)
            adv, ret = A.get_advantage_return(me, rewards, values, dones, tl)
            rec[f"adv_gae{int(use_gae)}"], rec[f"ret_gae{int(use_gae)}"] = adv, ret
        adv = rec["adv_gae1"]
        for mode in ("accumulate", "value_subtraction", "accumulated_rewards"):
            for norm in (True, False):
                me = SimpleNamespace(discount_factor=torch.tensor(gamma, dtype=torch.float64),
                                     segment_advantage=mode, norm_advantages=norm, clip_advantages=0.0,
                                     dtype=torch.float64, device=torch.device("cpu"))
                rec[f"seg_{mode}_norm{int(norm)}"] = A.get_segment_advantage(me, rewards, values, adv, pairs)
        lp_new = torch.randn(B, pairs.shape[0], generator=g, dtype=torch.float64)
        lp_old = lp_new + 0.1 * torch.randn(B, pairs.shape[0], generator=g, dtype=torch.float64)
        rec["lp_new"], rec["lp_old"] = lp_new, lp_old
        rec["surrogate"] = A.surrogate_loss(rec["seg_value_subtraction_norm1"], lp_new, lp_old)[0]
        vnew = values[:, :-1] + 0.3 * torch.randn(B, T, generator=g, dtype=torch.float64)
        rec["values_new"] = vnew
        for clip in (0.0, 0.2):
            me = SimpleNamespace(clip_critic=clip)
            rec[f"value_loss_clip{clip}"] = A.value_loss(me, vnew, rec["ret_gae1"], values[:, :-1])
        out[tag] = rec
    return out


def gen_ref_policy(mprl):
    from mprl.rl.policy import policy_factory
    out = {}
    for name in ("box", "table_tennis"):
        cfg = MP_CONFIGS[name]
        D, K1, T = cfg["num_dof"], cfg["num_basis"] + 1, NUM_TIMES[name]
        Dp = D * K1
        torch.manual_seed(3)
        pol = policy_factory("TemporalCorrelatedPolicy", dim_in=5, dim_out=Dp,
                             mean_net_args=dict(avg_neuron=16, num_hidden=2, shape=0.0),
                             variance_net_args=dict(std_only=False, contextual=False),
                             init_method="orthogonal", out_layer_gain=0.01, act_func_hidden="leaky_relu",
                             act_func_last=None, dtype="float64", device="cpu", min_std=1e-4,
                             mp=dict(type="prodmp", args=dict(cfg, dtype="float64", device="cpu")))
        B = 3
        inp = synthetic_inputs(name, B, seed=5)
        obs = torch.randn(B, 5, dtype=torch.float64)
        with torch.no_grad():
            pol.variance_net.variable.add_(0.05 * torch.randn_like(pol.variance_net.variable))
            mean, L = pol.policy(obs)
        rec = dict(cov_vector=pol.variance_net.variable.detach().clone(), obs=obs,
                   mean_net_state={k: v.clone() for k, v in pol.mean_net.state_dict().items()},
                   mean=mean, L=L)
        rec["entropy"] = pol.entropy([mean, L]).detach()
        rec["covariance"] = pol.covariance(L).detach()
        rec["log_determinant"] = pol.log_determinant(L).detach()
        rec["precision"] = pol.precision(L).detach()
        rec["maha"] = pol.maha(inp["mean"], inp["mean_old"], inp["L_old"]).detach()
        rec["bb_log_prob"] = super(type(pol), pol).log_prob(inp["mean_old"], inp["mean"], inp["L"]).detach()
        init_time = torch.tensor([0.0, 0.1, 0.0], dtype=torch.float64)
        times = util_times(init_time, T, cfg["dt"])
        traj = pol.sample(False, inp["mean"], inp["L"], times, init_time, inp["init_pos"], inp["init_vel"],
                          use_mean=True)
        torch.manual_seed(0)
        import mprl.util as util
        pairs = util.select_pred_pairs(num_all=T, num_select=25, fixed_interval=True).to(torch.long)
        # a "sampled" trajectory: synthesised from theta = mean + L eps through the mean path
        theta = inp["mean"] + torch.einsum('bij,bj->bi', inp["L"], inp["eps"])
        smp = pol.sample(False, theta, inp["L"], times, init_time, inp["init_pos"], inp["init_vel"],
                         use_mean=True)
        lp = pol.log_prob(smp, inp["mean"], inp["L"], times, init_time, inp["init_pos"], inp["init_vel"],
                          pred_pairs=pairs)
        rec.update(inputs=inp, init_time=init_time, times=times, traj_mean=traj, smp_traj=smp,
                   pred_pairs=pairs, log_prob=lp.detach())
        out[name] = rec
    return out


def util_times(init_time, T, dt):
    import mprl.util as util
    return util.tensor_linspace(init_time + dt, init_time + T * dt, T).T.contiguous()


def gen_oracle_path():
    """PARITY UNPINNED ProDMP tables straight from the oracle (regression fixtures for the CUDA tables).  Only what a
    test reads is stored: every fixture file stays under 1 MB."""
    from . import policy as opol
    out = {}
    for name in ("box", "metaworld", "table_tennis"):
        cfg = MP_CONFIGS[name]
        Dp = cfg["num_dof"] * (cfg["num_basis"] + 1)
        pol = opol.TemporalCorrelatedPolicy(Dp, mp=dict(type="prodmp", args=dict(cfg, dtype=torch.float64)),
                                            contextual=True, min_std=1e-4)
        tb = pol.mp.tables
        out[name] = dict(tables=dict(y1=tb.y1, y2=tb.y2, dy1=tb.dy1, dy2=tb.dy2, pos_basis=tb.pos_basis,
                                     vel_basis=tb.vel_basis, scale=pol.mp.weights_goal_scale))
    return out


def gen_ref_glue(mprl):
    """Rollout-side glue and agent pieces from the REAL reference: RunningMeanStd, make_mdp_reward, checkpoint paths and
    file contents of ``MLP.save`` / ``TrainableVariable.save``, ``generate_minibatches`` (numpy global generator),
    ``BlackBoxAgent.process_dataset`` and ``TemporalCorrelatedAgent.update_critic`` (run unbound on a stand-in self)."""
    import tempfile
    import types
    import numpy as np
    import mprl.util as util
    from mprl.rl.agent.black_box_agent import BlackBoxAgent
    from mprl.rl.agent.temporal_correlated_agent import TemporalCorrelatedAgent
    g = {}
    gen = torch.Generator().manual_seed(11)
    # ---- RunningMeanStd ------------------------------------------------------------------------------------------------
    rms = util.RunningMeanStd(name="obs", shape=(5,), dtype="torch.float64", device="cpu")
    batches = [torch.randn(n, 5, generator=gen, dtype=torch.float64) * (i + 1) + i for i, n in enumerate((7, 1000, 3))]
    hist = []
    for b in batches[:2]:
        rms.update(b)
        hist.append(dict(mean=rms.mean.clone(), var=rms.var.clone(), count=float(rms.count)))
    other = util.RunningMeanStd(shape=(5,), dtype="torch.float64", device="cpu")
    other.update(batches[2])
    rms.combine(other)
    hist.append(dict(mean=rms.mean.clone(), var=rms.var.clone(), count=float(rms.count)))
    g["rms"] = dict(batches=batches, hist=hist)
    # ---- make_mdp_reward -----------------------------------------------------------------------------------------------
    E, T = 6, 9
    rewards = torch.randn(E, T, generator=gen, dtype=torch.float64)
    first = [4, 0, 8, 1, -1, 3]                       # -1: never; 0: event from the very first step (argmax 0 -> "not happened")
    event = np.zeros((E, T), dtype=bool)
    for e, f in enumerate(first):
        if f >= 0:
            event[e, f:] = True
    infos_hit = [{"hit_ball": event[e].tolist(), "has_left_floor": event[e][::-1].tolist()} for e in range(E)]
    g["mdp"] = dict(rewards=rewards.clone(), event=torch.as_tensor(event),
                    table_tennis=util.make_mdp_reward("TableTennis4D-v0", rewards.clone(), infos_hit, torch.float64, "cpu"),
                    hopper=util.make_mdp_reward("HopperJumpSparse", rewards.clone(), infos_hit, torch.float64, "cpu"),
                    other=util.make_mdp_reward("BoxPushingDense", rewards.clone(), infos_hit, torch.float64, "cpu"))
    # ---- checkpoint paths and file contents --------------------------------------------------------------------------
    g["paths"] = dict(nn=util.get_nn_save_paths("/log", "policy_mean_mlp", 12), nn_none=util.get_nn_save_paths("/log", "x", None),
                      state=util.get_training_state_save_path("/log", "policy_optimizer", 3),
                      state_none=util.get_training_state_save_path("/log", "obs", None))
    torch.manual_seed(3)
    mlp = util.MLP(name="critic_net", dim_in=4, dim_out=1, hidden_layers=[8, 6], init_method="orthogonal",
                   out_layer_gain=1.0, act_func_hidden="leaky_relu", act_func_last=None, dtype=torch.float64,
                   device=torch.device("cpu"))
    var = util.TrainableVariable("cov", torch.arange(5, dtype=torch.float64))
    with tempfile.TemporaryDirectory() as d:
        mlp.save(d, 7)
        var.save(d, 7)
        files = sorted(os.listdir(d))
        import pickle as pkl
        with open(os.path.join(d, "critic_net_mlp_parameters.pkl"), "rb") as f:
            structure = pkl.load(f)
        weights = torch.load(os.path.join(d, "critic_net_mlp_weights_7"), weights_only=False)
        with open(os.path.join(d, "cov_variable_parameters.pkl"), "rb") as f:
            var_structure = pkl.load(f)
        var_saved = torch.load(os.path.join(d, "cov_variable_weights_7"), weights_only=False)
    x = torch.randn(3, 4, generator=gen, dtype=torch.float64)
    g["ckpt"] = dict(files=files, structure={k: (str(v) if k in ("dtype", "device") else v) for k, v in structure.items()},
                     weights={k: v.clone() for k, v in weights.items()}, x=x, y=mlp(x).detach(),
                     var_structure={k: (str(v) if k in ("dtype", "device") else (tuple(v) if k == "variable_shape" else v))
                                    for k, v in var_structure.items()}, var_saved=var_saved.detach().clone())
    # ---- generate_minibatches ------------------------------------------------------------------------------------------
    np.random.seed(7)
    g["minibatches"] = [[torch.as_tensor(s) for s in util.generate_minibatches(23, 4)] for _ in range(2)]
    # ---- BlackBoxAgent.process_dataset -------------------------------------------------------------------------------
    for n in (9, 1):
        fake = types.SimpleNamespace(norm_advantages=True, clip_advantages=1.5)
        ds = dict(segment_reward=torch.randn(n, generator=gen, dtype=torch.float64) * 3,
                  segment_value=torch.randn(n, generator=gen, dtype=torch.float64))
        out = BlackBoxAgent.process_dataset(fake, {k: v.clone() for k, v in ds.items()})
        g[f"bbrl_process_{n}"] = dict(inputs=ds, advantage=out["segment_advantage"].clone())
    # ---- TemporalCorrelatedAgent.update_critic -----------------------------------------------------------------------
    torch.manual_seed(5)
    critic_net = util.MLP(name="ValueFunction", dim_in=6, dim_out=1, hidden_layers=[16, 16], init_method="orthogonal",
                          out_layer_gain=1.0, act_func_hidden="leaky_relu", act_func_last=None, dtype=torch.float64,
                          device=torch.device("cpu"))
    w0 = {k: v.clone() for k, v in critic_net.state_dict().items()}
    D = 2
    ds = dict(step_states=torch.randn(5, 12, 6 + 2 * D, generator=gen, dtype=torch.float64),
              step_values=torch.randn(5, 13, generator=gen, dtype=torch.float64),
              step_returns=torch.randn(5, 12, generator=gen, dtype=torch.float64))
    for clip_critic, clip_norm in ((0.0, 0.0), (0.2, 0.5)):
        critic_net.load_state_dict(w0)
        opt = torch.optim.Adam(critic_net.parameters(), lr=1e-3, weight_decay=5e-5)
        fake = types.SimpleNamespace(epochs_critic=3, num_minibatchs=4, clip_grad_norm=clip_norm, clip_critic=clip_critic,
                                     critic=types.SimpleNamespace(critic=critic_net), policy=types.SimpleNamespace(num_dof=D),
                                     critic_optimizer=opt, critic_net_params=list(critic_net.parameters()))
        fake.value_loss = types.MethodType(TemporalCorrelatedAgent.value_loss, fake)
        np.random.seed(99)
        stats = TemporalCorrelatedAgent.update_critic(fake, ds)
        g[f"update_critic_{clip_critic}_{clip_norm}"] = dict(
            stats={k: float(v) for k, v in stats.items()},
            weights={k: v.clone() for k, v in critic_net.state_dict().items()})
    g["update_critic_inputs"] = dict(dataset=ds, w0=w0, num_dof=D)
    return g


def main():
    from . import ref_loader
    os.makedirs(OUT, exist_ok=True)
    mprl = ref_loader.load()
    import mprl.util as util
    torch.save(gen_ref_util(util), os.path.join(OUT, "ref_util.pt"))
    torch.save(gen_ref_agent(mprl), os.path.join(OUT, "ref_agent.pt"))
    torch.save(gen_ref_policy(mprl), os.path.join(OUT, "ref_policy.pt"))
    torch.save(gen_oracle_path(), os.path.join(OUT, "oracle_path.pt"))
    torch.save(gen_ref_glue(mprl), os.path.join(OUT, "ref_glue.pt"))
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()

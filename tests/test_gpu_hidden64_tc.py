"""hidden_units = 64 (the reference class default, ``w_nl.py:71``: GRU width 32, MLP width 64) on the tcgen05 encoder and
rollout kernels: forward against the fp64 oracle in every prediction-time form, plans against the oracle's MPPI step in both
rollout forms, the ping-pong form against the one-tile form beyond one wave, the kernel names a forward and a plan launch,
and the batched / sharded planners.

Weights: seeded hidden-64 models with the phi bias shifted into the trained operating range (the recipe of
``test_gpu_parity.py::test_hidden_units_64_class_default``).  Bounds (``_util.relerr``): ``tc_split3`` 1e-4, ``tc_fp16``
5e-2, the stated bounds of the two modes."""
import numpy as np
import pytest
import torch

from _util import DT, START_STATE, action_relerr, injected_noise, relerr
from test_gpu_multi_time import ENV_SHAPE, _inputs, _model, _oracle, _state_dict

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

H = 64
ENVS = list(ENV_SHAPE)
MODE_TOL = {"tc_split3": 1e-4, "tc_fp16": 5e-2}


def _nlc():
    import neurallaplacecontrol_b200 as nlc

    return nlc


def _ts_form(ts, form):
    """ts_pred as passed to the model (one time for all samples, one per sample, or (K, n_t)) and the (K, n_t) times of
    the oracle."""
    K = ts.shape[0]
    if form == "fixed":
        t = ts[0, 0].clone()
        return t, t.expand(K, 1)
    if form == "per_sample":
        return ts[:, :1].clone(), ts[:, :1]
    return ts, ts


def _check_forward(env, S, K, mode, B=4, eot=False, forms=("fixed", "per_sample", "Knt")):
    sd = _state_dict(env, H, S, calibrated=True, eot=eot)
    m = _model(env, sd, H, S, eot, math_mode=mode)
    for form in forms:
        obs, act, ts = _inputs(env, K, 3 if form == "Knt" else 1, B, seed=K + S, eot=eot)
        ts_pred, ts_ref = _ts_form(ts, form)
        ref = _oracle(sd, obs, act, ts_ref, torch.float64)
        out = m(obs.cuda(), act.cuda(), ts_pred.cuda())
        e = relerr(ref, out)
        print(f"hidden 64 {env} S={S} K={K} B={B} eot={eot} {mode} {form}: {e:.2e}")
        assert e < MODE_TOL[mode], (env, S, K, B, eot, mode, form, e)


@pytest.mark.parametrize("mode", list(MODE_TOL))
@pytest.mark.parametrize("K", [1, 333, 20011])
@pytest.mark.parametrize("S", [17, 33])
@pytest.mark.parametrize("env", ENVS)
def test_forward_matches_fp64_oracle(env, S, K, mode):
    """One prediction time, per-sample times and (K, n_t) times."""
    _check_forward(env, S, K, mode)


@pytest.mark.parametrize("case", [("oderl-cartpole", 4, True), ("oderl-pendulum", 2, False), ("oderl-cartpole", 2, False),
                                  ("oderl-acrobot", 2, False), ("oderl-pendulum", 8, False), ("oderl-cartpole", 8, False)],
                         ids=["eot", "B2-pendulum", "B2-cartpole", "B2-acrobot", "B8-pendulum", "B8-cartpole"])
def test_forward_window_variants(case):
    """encode_obs_time (GRU input width 2) and window lengths 2 and 8, every case with B * input width <= 8 (the tensor-core
    encoder's [x | 1] block).  The oracle broadcasts action_mean over the time channel only for one action, as the reference."""
    env, B, eot = case
    for mode in MODE_TOL:
        _check_forward(env, 17, 333, mode, B=B, eot=eot, forms=("fixed", "per_sample"))


def _planner(env, m, K, T, mode, U0, **kw):
    from oracle import costs

    nlc = _nlc()
    nx, nu = ENV_SHAPE[env]
    ah = float(costs.ENV_ACT_HIGH[env])
    return nlc.MPPIDelay(nlc.NLDynamics(m, DT), nlc.EnvRunningCost(env), nx, nlc.noise_sigma_for(nu), num_samples=K, horizon=T,
                         device="cuda:0", lambda_=1.0, u_min=torch.tensor(-ah), u_max=torch.tensor(ah), u_scale=ah,
                         U_init=U0.clone(), math_mode=mode, **kw)


def _plan(env, S, K, T, mode, seed=13, sd=None):
    """One control step of a hidden-64 planner with injected noise; returns (planner, action, noise, state dict)."""
    nx, nu = ENV_SHAPE[env]
    sd = sd if sd is not None else _state_dict(env, H, S, calibrated=True)
    m = _model(env, sd, H, S, math_mode=mode)
    noise = injected_noise(K, T, nu, seed=seed)
    p = _planner(env, m, K, T, mode, torch.zeros(T, nu, dtype=torch.float64))
    p.noise_dist.sample = lambda shape: noise
    action = p.command(np.array(START_STATE[env]), torch.zeros(4, nu, dtype=torch.float64))
    torch.cuda.synchronize()
    return p, action, noise, sd


@pytest.mark.parametrize("form", ["1", "3"])
@pytest.mark.parametrize("S", [17, 33])
@pytest.mark.parametrize("env", ENVS)
def test_plan_matches_oracle(env, S, form, monkeypatch):
    """Costs, trajectories, U and the action of one tc_split3 control step against ``oracle.mppi.command`` (fp64), with the
    one-tile (1) and the ping-pong (3) rollout forced; shapes without a ping-pong form (2 nx S > 256) run the one-tile form."""
    from oracle import costs, mppi

    monkeypatch.setenv("NLC_ROLLOUT_TILES", form)
    K, T = 1000, 8
    nx, nu = ENV_SHAPE[env]
    ah = float(costs.ENV_ACT_HIGH[env])
    p, action, noise, sd = _plan(env, S, K, T, "tc_split3")
    ref = mppi.command(torch.zeros(T, nu, dtype=torch.float64), torch.tensor(START_STATE[env]), torch.zeros(4, nu, dtype=torch.float64),
                       noise, mppi.make_nl_dynamics(sd, DT), costs.running_cost(env), noise_sigma=mppi.noise_sigma_for(nu), u_scale=ah,
                       u_min=-ah, u_max=ah)
    errs = {"cost": relerr(ref["cost_total"], p.cost_total), "states": relerr(ref["states"], p.states), "U": relerr(ref["U"], p.U),
            "action": action_relerr(ref["action"], action, ref["U"], ah)}
    print(f"hidden 64 plan {env} S={S} form {form}: " + "  ".join(f"{k}={v:.2e}" for k, v in errs.items()))
    for k, v in errs.items():
        assert v < 1e-4, (k, errs)


@pytest.mark.parametrize("env", ["oderl-cartpole", "oderl-acrobot"])
def test_forms_beyond_one_wave_agree(env, monkeypatch):
    """K = 20011 (157 tiles, more than one wave): the ping-pong and one-tile forms give the same costs to 2e-6, and both
    match the fp32 CUDA-core anchor to 1e-4."""
    K, T, S = 20011, 8, 17
    sd = _state_dict(env, H, S, calibrated=True)
    costs_by = {}
    for mode, form in (("tc_split3", "3"), ("tc_split3", "1"), ("fp32", "1")):
        monkeypatch.setenv("NLC_ROLLOUT_TILES", form)
        p, _, _, _ = _plan(env, S, K, T, mode, seed=29, sd=sd)
        costs_by[(mode, form)] = p.cost_total.double().cpu()
    pp, one, anchor = costs_by[("tc_split3", "3")], costs_by[("tc_split3", "1")], costs_by[("fp32", "1")]
    e_forms, e_pp, e_one = relerr(one, pp), relerr(anchor, pp), relerr(anchor, one)
    print(f"hidden 64 {env} K={K}: ping-pong vs one-tile {e_forms:.2e}, vs fp32 anchor {e_pp:.2e} / {e_one:.2e}")
    assert e_forms < 2e-6 and e_pp < 1e-4 and e_one < 1e-4, (e_forms, e_pp, e_one)


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type.name == "CUDA"]


def test_forward_and_plan_run_the_tensor_core_kernels():
    """Under torch.profiler: a hidden-64 forward and a hidden-64 plan beyond one wave launch the width-32 tcgen05 encoder and
    the width-64 tcgen05 rollout (ping-pong for the plan), and neither fp32 CUDA-core kernel."""
    env, S = "oderl-cartpole", 17
    sd = _state_dict(env, H, S, calibrated=True)
    m = _model(env, sd, H, S, math_mode="tc_split3")
    obs, act, ts = _inputs(env, 333, 1, seed=3)
    m(obs.cuda(), act.cuda(), ts[:, :1].cuda())  # warm-up: module load and buffer allocation outside the profiled region
    fwd = _kernel_names(lambda: m(obs.cuda(), act.cuda(), torch.tensor(DT, dtype=torch.float64).cuda()))
    nx, nu = ENV_SHAPE[env]
    K, T = 20011, 8
    p = _planner(env, m, K, T, "tc_split3", torch.zeros(T, nu, dtype=torch.float64))
    state, buf = np.array(START_STATE[env]), torch.zeros(4, nu, dtype=torch.float64)
    p.command(state, buf)
    plan = _kernel_names(lambda: p.command(state, buf))
    for what, names, rollout in (("forward", fwd, ("rollout_tc2_kernel<64",)), ("plan", plan, ("rollout_pp_kernel<64",))):
        assert any("encode_tc2_kernel<32" in n for n in names), (what, sorted(set(names)))
        assert any(r in n for n in names for r in rollout), (what, sorted(set(names)))
        assert not any("encode_gru_kernel" in n or "rollout_nl_kernel" in n for n in names), (what, sorted(set(names)))


def test_batched_planner_reproduces_standalone_planners(monkeypatch):
    """Instance i of a hidden-64 BatchedMPPIDelay == MPPIDelay(seed=i) on the same state / buffer / U: bit-identical samples,
    costs, U and actions over two control steps."""
    from oracle import costs

    monkeypatch.setenv("NLC_ROLLOUT_TILES", "1")  # both sides on the same rollout form regardless of I * K
    nlc = _nlc()
    env, S, I, K, T = "oderl-acrobot", 17, 3, 512, 6
    nx, nu = ENV_SHAPE[env]
    ah = float(costs.ENV_ACT_HIGH[env])
    m = _model(env, _state_dict(env, H, S, calibrated=True), H, S, math_mode="tc_split3")
    common = dict(num_samples=K, horizon=T, device="cuda:0", lambda_=1.0, u_min=torch.tensor(-ah), u_max=torch.tensor(ah), u_scale=ah,
                  math_mode="tc_split3")
    gen = torch.Generator().manual_seed(5)
    U0 = torch.randn(I, T, nu, generator=gen, dtype=torch.float64) * 0.3
    states = torch.tensor([START_STATE[env]] * I, dtype=torch.float64) + 0.05 * torch.randn(I, nx, generator=gen, dtype=torch.float64)
    bufs = (torch.rand(I, 4, nu, generator=gen, dtype=torch.float64) * 2 - 1) * ah
    seeds = list(range(I))
    batch = nlc.BatchedMPPIDelay(nlc.NLDynamics(m, DT), nlc.EnvRunningCost(env), nx, nlc.noise_sigma_for(nu), I, seeds=seeds, U_init=U0,
                                 **common)
    singles = [nlc.MPPIDelay(nlc.NLDynamics(m, DT), nlc.EnvRunningCost(env), nx, nlc.noise_sigma_for(nu), U_init=U0[i], seed=seeds[i],
                             keep_states=False, **common) for i in range(I)]
    for call in range(2):
        act_b = batch.command(states, bufs)
        torch.cuda.synchronize()
        for i, p in enumerate(singles):
            a = p.command(states[i].cuda(), bufs[i].cuda())
            torch.cuda.synchronize()
            assert torch.equal(p.noise, batch.noise[i]), (call, i)
            assert torch.equal(p.cost_total, batch.cost_total[i]), (call, i)
            assert torch.equal(a.float(), act_b[i].float()), (call, i)
            assert torch.equal(p.U.float(), batch.U[i]), (call, i)


@pytest.mark.parametrize("form", ["1", "3"])
def test_sharded_step_equals_unsharded(form, monkeypatch):
    """shard=(r, 4) in one process, merged through the shard triples: the concatenated shard costs are bit-identical to the
    unsharded plan's in the same rollout form, and every shard's U is the unsharded U to 1e-5."""
    monkeypatch.setenv("NLC_ROLLOUT_TILES", form)
    env, S, K, T, G = "oderl-cartpole", 17, 4096, 8, 4
    nx, nu = ENV_SHAPE[env]
    m = _model(env, _state_dict(env, H, S, calibrated=True), H, S, math_mode="tc_split3")
    noise = injected_noise(K, T, nu, seed=31)
    state, buf = np.array(START_STATE[env]), torch.zeros(4, nu, dtype=torch.float64)
    U0 = torch.zeros(T, nu, dtype=torch.float64)
    whole = _planner(env, m, K, T, "tc_split3", U0)
    whole.noise_dist.sample = lambda shape: noise
    whole.command(state, buf)
    planners = [_planner(env, m, K, T, "tc_split3", U0, shard=(r, G)) for r in range(G)]
    for p in planners:
        p.noise_dist.sample = lambda shape: noise
        assert p._begin(state, buf) is None
    triples = torch.stack([p.shard_triple.clone() for p in planners])
    for p in planners:
        p.all_triples.copy_(triples)
        p._finish()
    torch.cuda.synchronize()
    assert torch.equal(torch.cat([p.cost_total for p in planners]), whole.cost_total)
    for p in planners:
        assert relerr(whole.U, p.U) < 1e-5, relerr(whole.U, p.U)

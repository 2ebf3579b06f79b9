"""``MPPIDelay(..., math_mode="fp64")``: the fp64 planner (``nlc_planner_f64_*``) against the reference's own fp64 plans
(``tests/golden/plan_*.npz``), the fp64 oracle, and the composition a user can write without it (the reference's control step
around ``NeuralLaplaceModel(math_mode="fp64")``, ``tools/bench_plan_fp64.py:composition``).

Bounds (``_util.relerr``: max |ref - got| / max |ref| per tensor; ``relerr_per_channel`` for trajectories) are budgets sized
from the fp64 model's measured 6e-15 .. 2.7e-13 against the reference: stage-1 tensors bit-identical for a single call
(a second call perturbs the U the first call planned: 1e-12 against the golden, bit-identical to the reference's chain on
the planner's own U), states and costs 1e-10 (analytic dynamics 1e-11), the softmax
outputs 1e-10 on calibrated weights and 1e-6 on raw ones (lambda = 1 turns a cost of ~1e8 at fp64 precision into ~1e-6 of
weight), 1e-13 against the composition on the same GPU (its exponential weights 1e-12)."""
import ctypes as C
import importlib.util
import os

import numpy as np
import pytest
import torch

from _util import DT, ENVS, FULL_SIZE, S_TERMS, START_STATE, injected_noise, load, relerr, relerr_per_channel, short
from test_gpu_parity import PLAN_KEYS, _run_plan, make_model, make_planner
from test_plan_fp64_cpu import f64_noise

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STAGE1 = ("noise", "perturbed_action", "actions")


def _bench():
    spec = importlib.util.spec_from_file_location("bench_plan_fp64", os.path.join(ROOT, "tools", "bench_plan_fp64.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _nlc():
    import neurallaplacecontrol_b200 as nlc

    return nlc


def _check_stage1_chain(env, U_prev, noise, out):
    """Stage 1 of a control step from U_prev: the reference's fp64 chain (oracle.mppi.perturb, mppi_delay.py:319-340)
    reproduced bit for bit."""
    from oracle import costs, mppi

    nu = noise.shape[-1]
    ah = float(np.float32(costs.ENV_ACT_HIGH[env]))
    U = torch.roll(U_prev.double(), -1, dims=0)
    U[-1] = 0
    pert, nb, _ = mppi.perturb(U, noise.clone(), torch.inverse(mppi.noise_sigma_for(nu)), 1.0, ah, torch.tensor(-ah, dtype=torch.float64),
                               torch.tensor(ah, dtype=torch.float64))
    assert torch.equal(pert, out["perturbed_action"].cpu()) and torch.equal(nb, out["noise"].cpu())
    assert torch.equal((ah * pert) / ah, out["actions"].cpu())


@pytest.mark.parametrize("env", ENVS)
@pytest.mark.parametrize("case", ["raw", "cal_calls1", "cal_calls2", "cal_stateK"])
def test_plan_matches_reference_fp64(env, case):
    name = f"plan_raw_{short(env)}" if case == "raw" else f"plan_{case.replace('cal_', 'cal_' + short(env) + '_')}"
    g = load(name)
    planner, out = _run_plan(env, g, calibrated=case != "raw", n_calls=2 if case.endswith("calls2") else 1, math_mode="fp64")
    assert out["action"].dtype == torch.float64 and out["noise"].dtype == torch.float64
    errs = {k: relerr(g[k], out[k]) for k in PLAN_KEYS}
    print(f"\n{env} {case}: " + "  ".join(f"{k}={v:.1e}" for k, v in errs.items()))
    if case.endswith("calls2"):
        # the second call perturbs the U the first call planned, which carries that call's softmax error (U within 1e-10,
        # measured ~6e-13 relative): against the golden the stage-1 tensors inherit it (1e-12; measured 1.0e-13 .. 1.2e-13)
        # and are bit-identical to the reference's chain applied to the planner's own U
        for k in STAGE1:
            assert errs[k] <= 1e-12, (k, errs)
        _, first = _run_plan(env, g, calibrated=True, n_calls=1, math_mode="fp64")
        _check_stage1_chain(env, first["U"].cpu(), torch.from_numpy(g["in_noise"][1]), out)
    else:
        for k in STAGE1:
            assert torch.equal(torch.from_numpy(g[k]), out[k].cpu()), (k, errs[k])
    for k in ("states", "cost_total"):
        assert errs[k] <= 1e-10, (k, errs)
    for k in ("cost_total_non_zero", "omega", "U", "action"):
        assert errs[k] <= (1e-6 if case == "raw" else 1e-10), (k, errs)
    assert abs(float(out["omega"].sum()) - 1.0) < 1e-12


def test_cfg1_pendulum_K1000_H20_fp64():
    from oracle.gen_golden import injected_noise as gen_noise

    env = "oderl-pendulum"
    g = load("plan_cfg1_pendulum_K1000_H20")
    K, T, nu = 1000, 20, 1
    gg = {"in_U": np.zeros((T, nu)), "in_buffer": np.zeros((4, nu)), "in_state": np.array(START_STATE[env]),
          "in_noise": gen_noise(K, T, nu, seed=int(g["noise_seed"])).numpy()}
    planner, out = _run_plan(env, gg, calibrated=True, math_mode="fp64")
    assert relerr(g["cost_total"], out["cost_total"]) <= 1e-10
    assert relerr(g["states_first16"], out["states"][:16]) <= 1e-10
    assert relerr(g["states_last"], out["states"][:, -1]) <= 1e-10
    for k in ("omega", "U", "action"):
        assert relerr(g[k], out[k]) <= 1e-10, k


@pytest.mark.parametrize("env", ENVS)
@pytest.mark.parametrize("delay", [0, 1, 3])
def test_analytic_dynamics_plan_fp64(env, delay):
    g = load(f"plan_oracledyn_{short(env)}_d{delay}")
    dyn = _nlc().AnalyticDelayDynamics(env, delay, DT)
    noise = torch.from_numpy(g["in_noise"])
    planner = make_planner(env, None, noise.shape[0], noise.shape[1], g["in_U"], dynamics=dyn, math_mode="fp64")
    planner.noise_dist.sample = lambda shape: noise.clone()
    action = planner.command(np.asarray(g["in_state"]), torch.from_numpy(g["in_buffer"]))
    for k in STAGE1:
        assert torch.equal(torch.from_numpy(g[k]), getattr(planner, k).cpu()), k
    for k in ("states", "cost_total"):
        assert relerr(g[k], getattr(planner, k)) <= 1e-11, k
    for k in ("omega", "U"):
        assert relerr(g[k], getattr(planner, k)) <= 1e-10, k
    assert relerr(g["action"], action) <= 1e-10


def _full_size(cfg, family):
    from oracle import costs

    nlc = _nlc()
    env, K, T, name = FULL_SIZE[cfg]
    nx, nu = costs.ENV_DIMS[env]
    ah = np.float32(costs.ENV_ACT_HIGH[env])
    m = make_model(env, calibrated=family == "cal", math_mode="tc_split3")  # the planner works whatever the model's own mode
    p = nlc.MPPIDelay(nlc.NLDynamics(m, DT), nlc.EnvRunningCost(env), nx, nlc.noise_sigma_for(nu), num_samples=K, horizon=T,
                      device="cuda:0", lambda_=1.0, u_min=torch.tensor(-ah), u_max=torch.tensor(ah), u_scale=ah,
                      U_init=torch.zeros(T, nu, dtype=torch.float64), math_mode="fp64")
    g = load(f"{name}_{family}")
    noise = injected_noise(K, T, nu, seed=int(g["noise_seed"]))
    p.noise_dist.sample = lambda shape: noise
    action = p.command(np.array(START_STATE[env]), torch.zeros(4, nu, dtype=torch.float64))
    return env, g, p, action


@pytest.mark.parametrize("cfg", ["cfg3", "cfg4"])
def test_full_size_plan_fp64_calibrated(cfg):
    env, g, p, action = _full_size(cfg, "cal")
    idx = torch.from_numpy(g["spread_idx"]).cuda()
    errs = {
        "cost_total": relerr(g["cost_total"], p.cost_total),
        "states_spread": relerr_per_channel(g["states_spread"], p.states[idx]),
        "states_last": relerr_per_channel(g["states_last"], p.states[:, -1]),
        "omega_top": relerr(g["omega_top"], p.omega[torch.from_numpy(g["omega_top_idx"]).cuda()]),
        "U": relerr(g["U"], p.U),
        "action": relerr(g["action"], action),
    }
    print(f"\n{cfg} fp64 vs reference fp64: " + "  ".join(f"{k}={v:.2e}" for k, v in errs.items()))
    for k in ("cost_total", "states_spread", "U", "action"):
        assert errs[k] <= 1e-10, (k, errs)
    assert errs["omega_top"] <= 1e-9, errs
    assert errs["states_last"] <= 1e-6, errs  # that golden is stored in float32


@pytest.mark.parametrize("cfg", ["cfg3", "cfg4"])
def test_full_size_plan_fp64_raw_first_steps(cfg):
    """Raw init is chaotic (a perturbation grows ~6x per step even between two fp64 runs): steps 0-5 per channel."""
    env, g, p, action = _full_size(cfg, "raw")
    idx = torch.from_numpy(g["spread_idx"]).cuda()
    curve = [relerr_per_channel(g["states_spread"][:, t], p.states[idx][:, t]) for t in range(g["states_spread"].shape[1])]
    print(f"\n{cfg} raw fp64 per-step error: " + " ".join(f"{e:.1e}" for e in curve[:12]))
    assert max(curve[:6]) <= 1e-9, curve[:6]


@pytest.mark.parametrize("env", ["oderl-cartpole", "oderl-acrobot"])
def test_equals_composition_with_fp64_model(env):
    """Against the reference's control step around NeuralLaplaceModel(math_mode="fp64") on the same GPU, K = 1000, T = 20."""
    bench = _bench()
    K, T = 1000, 20
    p, noise, state, ah = bench.build(env, K, T, "fp64", seed=3)
    m, noise_d, _, _ = bench.build(env, K, T, "composition", seed=3)
    p.noise_dist.sample = lambda shape: noise
    nu = noise.shape[-1]
    buf = torch.tensor([[0.3] * nu, [-0.2] * nu, [0.1] * nu, [0.5] * nu], dtype=torch.float64)
    action = p.command(state, buf)
    lo, hi = torch.tensor(-float(ah), dtype=torch.float64), torch.tensor(float(ah), dtype=torch.float64)
    ref = bench.composition(m, env, torch.zeros(T, nu, dtype=torch.float64, device="cuda"), torch.from_numpy(state).cuda(), buf.cuda(),
                            noise_d, float(ah), DT, bounds=(lo, hi))
    errs = {k: relerr(ref[k], getattr(p, k)) for k in bench.KEYS}
    errs["action"] = relerr(ref["action"], action)
    print(f"\n{env} fp64 planner vs composition: " + "  ".join(f"{k}={v:.1e}" for k, v in errs.items()))
    # lambda = 1 turns the absolute cost difference (~1e-13 at costs of ~1e2: the fused running cost against torch's
    # separate operations) into that relative difference of the exponential weights (measured 1.2e-13 .. 1.4e-13)
    for k, v in errs.items():
        assert v <= (1e-12 if k in ("cost_total_non_zero", "omega") else 1e-13), (k, errs)


def _oracle_plan(env, sd, U0, state, buf, noise, u_scale, lo, hi, encode_obs_time=False, **opts):
    from oracle import costs, mppi

    return mppi.command(U0.clone(), torch.as_tensor(state), buf, noise, mppi.make_nl_dynamics(sd, DT, encode_obs_time),
                        costs.running_cost(env, **opts), noise_sigma=mppi.noise_sigma_for(noise.shape[-1]), u_scale=u_scale,
                        u_min=lo, u_max=hi)


OPTIONS = ["null_action", "abs_cost", "dim_bounds", "u_per_command", "B1", "B8", "eot", "hidden64", "S33", "goal_m2",
           "goal_p2_constraint", "two_commands"]


@pytest.mark.parametrize("opt", OPTIONS)
def test_options_match_fp64_oracle(opt):
    from oracle import costs, mppi

    nlc = _nlc()
    env = {"null_action": "oderl-acrobot", "abs_cost": "oderl-acrobot", "dim_bounds": "oderl-acrobot", "eot": "oderl-pendulum"}.get(
        opt, "oderl-cartpole")
    nx, nu = costs.ENV_DIMS[env]
    K, T, B = 96, 6, {"B1": 1, "B8": 8}.get(opt, 4)
    H, S = (64 if opt == "hidden64" else 128), (33 if opt == "S33" else S_TERMS)
    ah = float(costs.ENV_ACT_HIGH[env])
    lo, hi = (torch.tensor([-1.0, -0.25]), torch.tensor([0.5, 2.0])) if opt == "dim_bounds" else (torch.tensor(-ah), torch.tensor(ah))
    torch.manual_seed(5)
    eot = opt == "eot"
    m = nlc.NeuralLaplaceModel(nx, nu, nx, hidden_units=H, s_recon_terms=S, encode_obs_time=eot, state_mean=np.zeros(nx),
                               state_std=np.ones(nx), action_mean=np.zeros(nu), action_std=np.array([1.5]), normalize=True,
                               normalize_time=True, dt=DT, device="cuda:0").double()
    if eot:
        m.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in load("weights_eot_" + short(env)).items()})
    else:
        with torch.no_grad():
            m.laplace_rep_func.linear_tanh_stack[4].bias[nx * S:].sub_(4.0)
    sd = {k: v.detach().cpu().double() for k, v in m.state_dict().items()}
    cost_opts = {"goal_m2": {"change_goal": True}, "goal_p2_constraint": {"change_goal": True, "change_goal_flipped": True,
                                                                         "state_constraint": True}}.get(opt, {})
    kw = {"sample_null_action": opt == "null_action", "noise_abs_cost": opt == "abs_cost", "u_per_command": 3 if opt == "u_per_command" else 1}
    g = torch.Generator().manual_seed(11)
    U0 = torch.randn(T, nu, generator=g, dtype=torch.float64) * 0.2
    state = np.array(START_STATE[env]) + 0.01
    buf = (torch.rand(B, nu, generator=g, dtype=torch.float64) * 2 - 1) * ah
    p = nlc.MPPIDelay(nlc.NLDynamics(m, DT), nlc.EnvRunningCost(env, **cost_opts), nx, nlc.noise_sigma_for(nu), num_samples=K, horizon=T,
                      device="cuda:0", u_min=lo, u_max=hi, u_scale=ah, U_init=U0.clone(), math_mode="fp64", **kw)
    U_ref = U0.clone()
    for c in range(2 if opt == "two_commands" else 1):
        noise = injected_noise(K, T, nu, seed=20 + c)
        p.noise_dist.sample = lambda shape, noise=noise: noise
        a = p.command(state, buf)
        if kw["sample_null_action"] or kw["noise_abs_cost"]:
            Ur = torch.roll(U_ref, -1, dims=0)
            Ur[-1] = 0
            pert, nb, pc = mppi.perturb(Ur, noise.clone(), torch.inverse(mppi.noise_sigma_for(nu)), 1.0, ah, lo.double(), hi.double(),
                                        sample_null_action=kw["sample_null_action"], noise_abs_cost=kw["noise_abs_cost"])
            cost, states, _ = mppi.rollout_costs(mppi.make_nl_dynamics(sd, DT), costs.running_cost(env), torch.from_numpy(state), pert,
                                                 buf, ah)
            Un, w, omega = mppi.softmax_update(Ur, cost + pc, nb, 1.0)
            ref = {"perturbed_action": pert, "noise": nb, "cost_total": cost + pc, "states": states, "U": Un, "omega": omega}
        else:
            ref = _oracle_plan(env, sd, U_ref, state, buf, noise, ah, lo.double(), hi.double(), eot, **cost_opts)
        U_ref = ref["U"]
        errs = {k: relerr(ref[k], getattr(p, k)) for k in ("perturbed_action", "noise", "cost_total", "states", "U", "omega")}
        if opt == "u_per_command":
            assert a.shape == (3, nu)
            errs["action"] = relerr(ref["U"][:3] * ah, a)
        assert max(errs.values()) <= 1e-10, (opt, c, errs)
        buf, _ = mppi.get_action(buf, p.U[0].cpu() * ah, min(1, B - 1))
    if opt == "null_action":
        assert float(p.perturbed_action[-1].abs().max()) == 0.0


def test_planner_level_encode_obs_time_analytic_fp64():
    g = load("plan_oracledyn_pendulum_d1")
    noise = torch.from_numpy(g["in_noise"])
    dyn = _nlc().AnalyticDelayDynamics("oderl-pendulum", 1, DT)
    p = make_planner("oderl-pendulum", None, noise.shape[0], noise.shape[1], g["in_U"], dynamics=dyn, encode_obs_time=True,
                     math_mode="fp64")
    p.noise_dist.sample = lambda shape: noise.clone()
    buf = torch.cat((torch.from_numpy(g["in_buffer"]), torch.arange(4, dtype=torch.float64).view(4, 1) * DT), dim=1)
    a = p.command(np.asarray(g["in_state"]), buf)
    assert relerr(g["cost_total"], p.cost_total) <= 1e-11 and relerr(g["action"], a) <= 1e-10


def _sampler_planner(env, K, T, seed, **kw):
    m = make_model(env, calibrated=True)
    return make_planner(env, m, K, T, np.zeros((T, 2 if env == "oderl-acrobot" else 1)), seed=seed, math_mode="fp64", **kw)


@pytest.mark.parametrize("seed", [0, 77])
def test_on_device_sampler_matches_statement(seed):
    from oracle import mppi

    env, K, T, nu = "oderl-acrobot", 512, 12, 2
    p = _sampler_planner(env, K, T, seed)
    chol = torch.linalg.cholesky(mppi.noise_sigma_for(nu)).numpy()
    state, buf = np.array(START_STATE[env]), torch.zeros(4, nu, dtype=torch.float64)
    prev = None
    for call in range(2):
        p.command(state, buf)
        raw = f64_noise(K, T, nu, seed, call, chol, np.zeros(nu))
        # perturbed - rolled U is the raw draw (up to the rounding of U + raw) wherever the bounds did not clamp
        Ur = torch.roll(torch.from_numpy(np.zeros((T, nu))) if call == 0 else prev_U, -1, dims=0)
        Ur[-1] = 0
        got = (p.perturbed_action.cpu() - Ur).numpy()
        inside = np.abs(p.perturbed_action.cpu().numpy()) < 0.999
        assert inside.mean() > 0.3
        assert np.abs(got - raw)[inside].max() <= 1e-14 * max(1.0, np.abs(raw).max())
        if prev is not None:
            assert not np.array_equal(prev, raw)
        prev, prev_U = raw, p.U.cpu().clone()
    z = raw.reshape(-1, nu)
    assert np.abs(z.mean(0)).max() < 0.05
    assert np.abs(np.cov(z.T) - mppi.noise_sigma_for(nu).numpy()).max() < 0.05


def test_deterministic_and_fresh_noise_per_command():
    env = "oderl-cartpole"
    outs = []
    for _ in range(2):
        p = _sampler_planner(env, 700, 9, seed=4)
        a = p.command(np.array(START_STATE[env]), torch.zeros(4, 1, dtype=torch.float64))
        outs.append([a] + [getattr(p, k).clone() for k in PLAN_KEYS if k != "action"])
        n0 = p.noise.clone()
        p.command(np.array(START_STATE[env]), torch.zeros(4, 1, dtype=torch.float64))
        assert not torch.equal(n0, p.noise)
    for x, y in zip(*outs):
        assert torch.equal(x, y)


def test_host_and_device_inputs_agree():
    env = "oderl-cartpole"
    res = []
    for dev in (False, True):
        p = _sampler_planner(env, 300, 8, seed=9)
        state, buf = torch.tensor(START_STATE[env], dtype=torch.float64) + 0.01, torch.full((4, 1), 0.2, dtype=torch.float64)
        acts = [p.command(state.cuda() if dev else state, buf.cuda() if dev else buf) for _ in range(2)]
        res.append((torch.stack(acts), p.U.clone(), p.cost_total.clone()))
    for x, y in zip(*res):
        assert torch.equal(x, y)


def test_weights_follow_an_optimizer_step():
    from oracle import costs

    env = "oderl-cartpole"
    nx, nu = costs.ENV_DIMS[env]
    K, T = 256, 8
    noise = injected_noise(K, T, nu, seed=8)
    state, buf = np.array(START_STATE[env]), torch.zeros(4, nu, dtype=torch.float64)
    m = make_model(env, calibrated=True, math_mode="fp64").cuda()
    p = make_planner(env, m, K, T, np.zeros((T, nu)), math_mode="fp64")
    p.noise_dist.sample = lambda shape: noise
    p.command(state, buf)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    with torch.enable_grad():
        obs = torch.randn(32, nx, dtype=torch.float64, device="cuda")
        act = torch.randn(32, 4, nu, dtype=torch.float64, device="cuda")
        loss = m(obs, act, torch.full((32, 1), DT, dtype=torch.float64, device="cuda")).pow(2).sum()
        loss.backward()
    opt.step()
    p.U = torch.zeros(T, nu, dtype=torch.float64)
    a1 = p.command(state, buf)
    m2 = make_model(env, calibrated=True, math_mode="fp64")
    m2.load_state_dict(m.state_dict())
    p2 = make_planner(env, m2, K, T, np.zeros((T, nu)), math_mode="fp64")
    p2.noise_dist.sample = lambda shape: noise
    a2 = p2.command(state, buf)
    assert torch.equal(a1, a2) and torch.equal(p.cost_total, p2.cost_total) and torch.equal(p.U, p2.U)


def test_rejections():
    from neurallaplacecontrol_b200 import _lib
    from neurallaplacecontrol_b200.episode import BatchedMPPIDelay

    nlc = _nlc()
    env = "oderl-pendulum"
    m = make_model(env, calibrated=True)
    args = (nlc.NLDynamics(m, DT), nlc.EnvRunningCost(env), 3, nlc.noise_sigma_for(1))
    with pytest.raises(NotImplementedError):
        nlc.MPPIDelay(*args, device="cuda:0", math_mode="fp64", shard=(0, 2))
    with pytest.raises(NotImplementedError):
        nlc.MPPIDelay(*args, device="cuda:0", math_mode="fp64", process_group=object())
    with pytest.raises(NotImplementedError):
        BatchedMPPIDelay(*args, n_instances=2, num_samples=64, horizon=5, device="cuda:0", math_mode="fp64")
    p = nlc.MPPIDelay(*args, num_samples=64, horizon=5, device="cuda:0", math_mode="fp64")
    for call in (lambda: p.get_rollouts(np.zeros(3)), lambda: p.set_inputs(np.zeros(3), torch.zeros(4, 1)), p.step):
        with pytest.raises(NotImplementedError):
            call()
    lib = _lib.load()
    d = _lib.PlannerF64Desc()
    d.base.mppi.K, d.base.mppi.T, d.base.mppi.nu, d.base.mppi.B, d.base.nx, d.base.n_shards = 64, 5, 1, 4, 3, 2
    d.base.rollout.dynamics, d.lambda_, d.u_scale, d.dt = 1, 1.0, 1.0, DT
    h = C.c_void_p()
    assert lib.nlc_planner_f64_create(C.byref(h), None, C.byref(d), 0) == -5  # NLC_ERR_UNSUPPORTED
    d.base.n_shards = 1
    assert lib.nlc_planner_f64_create(C.byref(h), None, C.byref(d), 0) == 0
    assert lib.nlc_planner_f64_destroy(h) == 0

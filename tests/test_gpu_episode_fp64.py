"""The closed loop at the reference's precision: ``env_step`` on fp64 tensors (``nlc_env_step_f64``) against the golden steps
of the reference's own ``oracle.py``, and ``run_closed_loop`` over one ``MPPIDelay(math_mode="fp64")`` per instance against
the fp64 oracle loop (``oracle.dynamics.closed_loop`` around ``oracle.mppi.command``) and against hand-written loops.

Bounds (``_util.relerr``) are budgets: one fp64 env step is the reference's expression in its own order (a few ulps from
libm's last bits); one fp64 control step agrees with the oracle to 1e-10 and the loop feeds that back through the plant."""
import numpy as np
import pytest
import torch

from _util import DT, injected_noise, load, relerr, short, weights
from test_gpu_parity import make_model, make_planner

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

ENVS = ["oderl-pendulum", "oderl-cartpole", "oderl-acrobot"]


def _nlc():
    import neurallaplacecontrol_b200 as nlc

    return nlc


@pytest.mark.parametrize("env", ENVS)
@pytest.mark.parametrize("delay", [0, 1, 3])
def test_env_step_f64_matches_reference(env, delay):
    """Six consecutive golden steps of 48 instances (generated in fp64 with the reference's oracle.py)."""
    nlc = _nlc()
    g = load("env_step_" + short(env))
    states = torch.tensor(g[f"d{delay}_state0"], dtype=torch.float64).cuda().contiguous()
    bufs = torch.tensor(g[f"d{delay}_buf0"], dtype=torch.float64).cuda().contiguous()
    rewards = torch.zeros(states.shape[0], dtype=torch.float64, device="cuda")
    worst = [0.0, 0.0]
    for it in range(g[f"d{delay}_actions"].shape[0]):
        a = torch.tensor(g[f"d{delay}_actions"][it], dtype=torch.float64).cuda().contiguous()
        nlc.env_step(env, states, bufs, a, delay, DT, rewards)
        torch.cuda.synchronize()
        assert torch.equal(bufs.cpu(), torch.from_numpy(g[f"d{delay}_bufs"][it]))  # pure data movement
        es, er = relerr(g[f"d{delay}_states"][it], states), relerr(g[f"d{delay}_rewards"][it], rewards)
        worst = [max(worst[0], es), max(worst[1], er)]
        assert es <= 1e-12 and er <= 1e-12, (it, es, er)
    print(f"\n{env} delay {delay} fp64 env_step vs reference: states {worst[0]:.1e}  rewards {worst[1]:.1e}")


def _planners(env, dynamics, I, K, T, delay, seeds=None):
    nlc = _nlc()
    nu = 2 if env == "oderl-acrobot" else 1
    m = make_model(env, calibrated=True) if dynamics == "neural_laplace" else None
    dyn = nlc.AnalyticDelayDynamics(env, delay, DT) if m is None else None
    return [make_planner(env, m, K, T, np.zeros((T, nu)), dynamics=dyn, math_mode="fp64", keep_states=False,
                         seed=0 if seeds is None else seeds[i]) for i in range(I)]


@pytest.mark.parametrize("env", ["oderl-pendulum", "oderl-acrobot"])
@pytest.mark.parametrize("dynamics", ["analytic", "neural_laplace"])
def test_closed_loop_matches_fp64_oracle_loop(env, dynamics):
    """3 instances, K = 256, T = 10, 8 control steps, delay 1, the same injected noise per instance and step on both sides."""
    nlc = _nlc()
    from oracle import costs, dynamics as odyn, mppi

    I, K, T, n_steps, delay = 3, 256, 10, 8, 1
    nx, nu = costs.ENV_DIMS[env]
    ah = float(np.float32(costs.ENV_ACT_HIGH[env]))
    noises = [torch.stack([injected_noise(K, T, nu, seed=1000 + it * I + i) for i in range(I)]) for it in range(n_steps)]
    st0 = torch.tensor(load("env_step_" + short(env))["d1_state0"][:I], dtype=torch.float64)

    res = nlc.run_closed_loop(_planners(env, dynamics, I, K, T, delay), env, st0, delay, n_steps, DT, noise_fn=lambda it: noises[it])

    model_dyn = (odyn.make_analytic_dynamics(env, DT, delay) if dynamics == "analytic"
                 else mppi.make_nl_dynamics(weights(env, calibrated=True), DT))
    Us, calls = [torch.zeros(T, nu, dtype=torch.float64) for _ in range(I)], [0]
    lo, hi = torch.tensor(-ah, dtype=torch.float64), torch.tensor(ah, dtype=torch.float64)

    def plan_fn(i, state, buf):
        out = mppi.command(Us[i], state, buf, noises[calls[0] // I][i], model_dyn, costs.running_cost(env),
                           noise_sigma=mppi.noise_sigma_for(nu), u_scale=ah, u_min=lo, u_max=hi)
        Us[i] = out["U"]
        calls[0] += 1
        return out["action"]

    total, final = odyn.closed_loop(env, plan_fn, st0.clone(), delay, n_steps, DT)
    assert res["total_reward_raw"].dtype == np.float64 and res["final_states"].dtype == np.float64
    assert res["total_reward_raw"].shape == (I,) and res["final_states"].shape == (I, nx) and res["n_instances"] == I
    e_r, e_s = relerr(total, res["total_reward_raw"]), relerr(final, res["final_states"])
    print(f"\n{env} {dynamics} fp64 closed loop vs fp64 oracle loop: total reward {e_r:.1e}  final states {e_s:.1e}")
    assert e_r <= 1e-9 and e_s <= 1e-9, (e_r, e_s)
    assert np.allclose(res["total_reward"], res["total_reward_raw"] * (200.0 / n_steps))


def test_driver_adds_nothing():
    """run_closed_loop over I fp64 planners (on-device sampler, distinct seeds) == I hand-written loops of command + fp64
    env_step with I = 1: bit-identical actions at every step, final states and total rewards."""
    nlc = _nlc()
    env, dynamics, I, K, T, n_steps, delay = "oderl-acrobot", "neural_laplace", 3, 256, 10, 6, 1
    nu, seeds = 2, [21, 22, 23]
    st0 = torch.tensor(load("env_step_acrobot")["d1_state0"][:I], dtype=torch.float64)

    planners = _planners(env, dynamics, I, K, T, delay, seeds)
    got = [[] for _ in range(I)]
    for i, p in enumerate(planners):  # record what the driver's command calls return
        p.command = lambda s, b, cmd=p.command, rec=got[i]: rec.append(cmd(s, b).clone()) or rec[-1]
    res = nlc.run_closed_loop(planners, env, st0, delay, n_steps, DT)

    for i, p in enumerate(_planners(env, dynamics, I, K, T, delay, seeds)):
        s = st0[i:i + 1].cuda().contiguous()
        b = torch.zeros(1, 4, nu, dtype=torch.float64, device="cuda")
        r = torch.zeros(1, dtype=torch.float64, device="cuda")
        tot = torch.zeros(1, dtype=torch.float64, device="cuda")
        for it in range(n_steps):
            a = p.command(s[0], b[0])
            assert torch.equal(a, got[i][it]), (i, it)
            nlc.env_step(env, s, b, a.reshape(1, nu).contiguous(), delay, DT, r)
            tot += r
        assert torch.equal(s.cpu(), torch.from_numpy(res["final_states"][i:i + 1])), i
        assert torch.equal(tot.cpu(), torch.from_numpy(res["total_reward_raw"][i:i + 1])), i
    assert len({float(g[0][0]) for g in got}) == I  # the seeds differ, so do the first actions


def test_rejections():
    nlc = _nlc()
    from neurallaplacecontrol_b200.episode import BatchedMPPIDelay

    f64 = dict(dtype=torch.float64, device="cuda")
    s, b, a = torch.zeros(2, 3, **f64), torch.zeros(2, 4, 1, **f64), torch.zeros(2, 1, **f64)
    for args in ((s, b.float(), a), (s, b, a.float()), (s.float(), b, a), (s.cpu(), b, a), (s, b.cpu(), a)):
        with pytest.raises(TypeError):
            nlc.env_step("oderl-pendulum", *args, 1)
    with pytest.raises(TypeError):
        nlc.env_step("oderl-pendulum", s, b, a, 1, DT, torch.zeros(2, device="cuda"))  # fp32 rewards
    with pytest.raises(TypeError):
        nlc.env_step("oderl-pendulum", torch.zeros(3, 2, **f64).t(), b, a, 1)  # non-contiguous
    with pytest.raises(RuntimeError):
        nlc.env_step("oderl-pendulum", s, b, a, 4)  # delay outside the 4-entry buffer
    with pytest.raises(RuntimeError):
        nlc.env_step("oderl-acrobot", torch.zeros(2, 6, **f64), b, a, 1)  # nu mismatch

    env, K, T = "oderl-pendulum", 64, 5
    p64 = make_planner(env, None, K, T, np.zeros((T, 1)), dynamics=nlc.AnalyticDelayDynamics(env, 1, DT), math_mode="fp64")
    p32 = make_planner(env, None, K, T, np.zeros((T, 1)), dynamics=nlc.AnalyticDelayDynamics(env, 1, DT), math_mode="fp32")
    st0 = torch.zeros(2, 3, dtype=torch.float64)
    with pytest.raises(TypeError):
        nlc.run_closed_loop([p64, p32], env, st0, 1, 2, DT)
    cart = make_planner("oderl-cartpole", None, K, T, np.zeros((T, 1)), dynamics=nlc.AnalyticDelayDynamics("oderl-cartpole", 1, DT),
                        math_mode="fp64")
    b2 = make_planner(env, None, K, T, np.zeros((T, 1)), dynamics=nlc.AnalyticDelayDynamics(env, 1, DT), math_mode="fp64",
                      action_buffer_size=2)
    upc = make_planner(env, None, K, T, np.zeros((T, 1)), dynamics=nlc.AnalyticDelayDynamics(env, 1, DT), math_mode="fp64",
                       u_per_command=2)
    for other in (cart, b2, upc):
        with pytest.raises(ValueError):
            nlc.run_closed_loop([p64, other], env, st0, 1, 2, DT)
    with pytest.raises(NotImplementedError, match="run_closed_loop"):
        BatchedMPPIDelay(nlc.AnalyticDelayDynamics(env, 1, DT), nlc.EnvRunningCost(env), 3, nlc.noise_sigma_for(1), n_instances=2,
                         num_samples=K, horizon=T, device="cuda:0", math_mode="fp64")

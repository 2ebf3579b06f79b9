"""One batch over many models and delays (the reference's env x delay x model x seed grid, ``run_exp_multi.py:135-165``):
``BatchedMPPIDelay`` over a sequence of dynamics handles - runs of instances sharing a model, side by side on the handle's
streams - against stand-alone planners, and ``env_step`` / ``run_closed_loop`` with one action delay per instance against
per-delay calls and the golden vectors of the reference's oracle.py dynamics."""
import ctypes as C

import numpy as np
import pytest
import torch

from _util import DT, load, relerr, short

pytestmark = pytest.mark.gpu

ORDER = [0, 1, 0, 2, 1, 2]           # instances over three models, interleaved: A B A C B C (six runs)
DELAYS = [0, 1, 0, 2, 3, 3]          # analytic instances: five runs


def _nlc():
    import neurallaplacecontrol_b200 as nlc

    return nlc


def _models(env):
    """A: hidden 128, S = 17 (the calibrated golden weights); B: hidden_units = 64; C: s_recon_terms = 33 - each with its own
    normalisation constants."""
    from test_gpu_multi_time import _model, _state_dict

    return [_model(env, _state_dict(env, H, S), H, S) for H, S in ((128, 17), (64, 17), (128, 33))]


def _setup(env, mode, I, K, T, B=4, seed=5):
    from oracle import costs

    nlc = _nlc()
    nx, nu = costs.ENV_DIMS[env]
    ah = np.float32(costs.ENV_ACT_HIGH[env])
    common = dict(num_samples=K, horizon=T, device="cuda:0", lambda_=1.0, u_min=torch.tensor(-ah), u_max=torch.tensor(ah),
                  u_scale=ah, math_mode=mode)
    gen = torch.Generator().manual_seed(seed)
    U0 = torch.randn(I, T, nu, generator=gen, dtype=torch.float64) * 0.3
    states = torch.tensor(load("env_step_" + short(env))["d1_state0"][:I], dtype=torch.float64)
    bufs = (torch.rand(I, B, nu, generator=gen, dtype=torch.float64) * 2 - 1) * float(ah)
    return nlc, nx, nu, common, U0, states, bufs


def _batch(nlc, env, dyns, nx, nu, seeds, U0, common):
    return nlc.BatchedMPPIDelay(dyns, nlc.EnvRunningCost(env), nx, nlc.noise_sigma_for(nu), len(seeds), seeds=seeds, U_init=U0, **common)


def _check_against_singles(nlc, env, batch, dyns, nx, nu, seeds, U0, states, bufs, common, calls=2):
    """Instance i of the batch == MPPIDelay(dyns[i], seed=seeds[i]) on the same state / buffer / U: bit-identical samples,
    costs, control sequences and actions over `calls` consecutive control steps."""
    I = len(seeds)
    singles = [nlc.MPPIDelay(dyns[i], nlc.EnvRunningCost(env), nx, nlc.noise_sigma_for(nu), U_init=U0[i], seed=seeds[i],
                             keep_states=False, **common) for i in range(I)]
    bufs = bufs.clone()
    for call in range(calls):
        act_b = batch.command(states, bufs)
        torch.cuda.synchronize()
        for i, p in enumerate(singles):
            a = p.command(states[i].cuda(), bufs[i].cuda())  # device inputs: the on-device sampler path, like the batch
            torch.cuda.synchronize()
            assert torch.equal(p.noise, batch.noise[i]), (call, i)
            assert torch.equal(p.cost_total, batch.cost_total[i]), (call, i)
            assert torch.equal(a.float(), act_b[i].float()), (call, i)
            assert torch.equal(p.U.float(), batch.U[i]), (call, i)
        for i in range(I):
            bufs[i], _ = nlc.get_action(bufs[i], act_b[i].cpu().double(), 1)


@pytest.mark.parametrize("env", ["oderl-pendulum", "oderl-acrobot"])
@pytest.mark.parametrize("mode", ["fp32", "tc_split3"])
def test_multi_model_batch_reproduces_standalone_planners(env, mode, monkeypatch):
    """Six instances over three models (hidden 128 / 64, S = 17 / 33) in interleaved order: six runs on the stream pool."""
    monkeypatch.setenv("NLC_ROLLOUT_TILES", "1")  # both sides on the same rollout form regardless of the run's size
    I, K, T = 6, 200, 6
    nlc, nx, nu, common, U0, states, bufs = _setup(env, mode, I, K, T)
    models = _models(env)
    dyns = [nlc.NLDynamics(models[j], DT) for j in ORDER]
    seeds = [11, 12, 13, 14, 15, 16]
    batch = _batch(nlc, env, dyns, nx, nu, seeds, U0, common)
    _check_against_singles(nlc, env, batch, dyns, nx, nu, seeds, U0, states, bufs, common)
    assert abs(float(batch.omega.sum()) - I) < 1e-4


@pytest.mark.parametrize("env", ["oderl-pendulum", "oderl-acrobot"])
@pytest.mark.parametrize("mode", ["fp32", "tc_split3"])
def test_analytic_delays_batch_reproduces_standalone_planners(env, mode):
    """Six analytic instances with delays 0..3 (five runs)."""
    I, K, T = 6, 200, 6
    nlc, nx, nu, common, U0, states, bufs = _setup(env, mode, I, K, T)
    dyns = [nlc.AnalyticDelayDynamics(env, d, DT) for d in DELAYS]
    seeds = [21, 22, 23, 24, 25, 26]
    batch = _batch(nlc, env, dyns, nx, nu, seeds, U0, common)
    _check_against_singles(nlc, env, batch, dyns, nx, nu, seeds, U0, states, bufs, common)


def _outputs(batch, states, bufs, calls=2):
    out = []
    for _ in range(calls):
        a = batch.command(states, bufs)
        torch.cuda.synchronize()
        out.append([a.clone(), batch.noise.clone(), batch.cost_total.clone(), batch.U.clone()])
    return out


@pytest.mark.parametrize("dynamics", ["neural_laplace", "analytic"])
def test_sequence_of_one_handle_equals_one_handle(dynamics):
    """BatchedMPPIDelay([dyn] * I) is BatchedMPPIDelay(dyn): one run, the same launches, bit-identical results."""
    env, I, K, T = "oderl-acrobot", 4, 1024, 8
    nlc, nx, nu, common, U0, states, bufs = _setup(env, "tc_split3", I, K, T)
    dyn = nlc.NLDynamics(_models(env)[0], DT) if dynamics == "neural_laplace" else nlc.AnalyticDelayDynamics(env, 2, DT)
    seeds = [1, 2, 3, 4]
    one = _outputs(_batch(nlc, env, dyn, nx, nu, seeds, U0, common), states, bufs)
    many = _outputs(_batch(nlc, env, [dyn] * I, nx, nu, seeds, U0, common), states, bufs)
    for a, b in zip(one, many):
        assert all(torch.equal(x, y) for x, y in zip(a, b))


def test_permuted_instances_give_the_same_results(monkeypatch):
    """The per-instance results do not depend on where an instance sits in the batch (which run, which stream)."""
    monkeypatch.setenv("NLC_ROLLOUT_TILES", "1")
    env, I, K, T = "oderl-pendulum", 6, 512, 8
    nlc, nx, nu, common, U0, states, bufs = _setup(env, "tc_split3", I, K, T)
    models = _models(env)
    seeds = [31, 32, 33, 34, 35, 36]
    perm = [5, 2, 0, 4, 1, 3]
    ref = _outputs(_batch(nlc, env, [nlc.NLDynamics(models[j], DT) for j in ORDER], nx, nu, seeds, U0, common), states, bufs)
    got = _outputs(_batch(nlc, env, [nlc.NLDynamics(models[ORDER[p]], DT) for p in perm], nx, nu, [seeds[p] for p in perm], U0[perm], common),
                   states[perm], bufs[perm])
    for a, b in zip(ref, got):
        for x, y in zip(a, b):
            assert torch.equal(x[perm], y)


def test_runs_in_flight_concurrently_are_deterministic():
    """Six runs of 2048 samples on the stream pool: two batches on the same inputs give bit-identical results."""
    env, I, K, T = "oderl-acrobot", 6, 2048, 12
    nlc, nx, nu, common, U0, states, bufs = _setup(env, "tc_split3", I, K, T)
    models = _models(env)
    seeds = [41, 42, 43, 44, 45, 46]
    make = lambda: _batch(nlc, env, [nlc.NLDynamics(models[j], DT) for j in ORDER], nx, nu, seeds, U0, common)  # noqa: E731
    a, b = _outputs(make(), states, bufs, 3), _outputs(make(), states, bufs, 3)
    for x, y in zip(a, b):
        assert all(torch.equal(u, v) for u, v in zip(x, y))


# ---- env_step with one delay per instance ------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("env", ["oderl-pendulum", "oderl-cartpole", "oderl-acrobot"])
def test_env_step_per_instance_delays_equal_per_delay_calls(env, dtype):
    """One call with delays 0..3 cycling over 24 instances == one scalar-delay call per delay on that delay's instances."""
    nlc = _nlc()
    g = load("env_step_" + short(env))
    I, B = 24, 4
    delays = [i % 4 for i in range(I)]
    nu = g["d1_buf0"].shape[2]
    gen = torch.Generator().manual_seed(3)
    st = torch.tensor(g["d1_state0"][:I], dtype=dtype).cuda().contiguous()
    bf = ((torch.rand(I, B, nu, generator=gen, dtype=torch.float64) * 2 - 1)).to(dtype).cuda().contiguous()
    rw = torch.zeros(I, dtype=dtype, device="cuda")
    ref_st, ref_bf, ref_rw = st.clone(), bf.clone(), rw.clone()
    for it in range(3):
        a = (torch.rand(I, nu, generator=gen, dtype=torch.float64) * 2 - 1).to(dtype).cuda().contiguous()
        nlc.env_step(env, st, bf, a, delays, DT, rw)
        for d in range(4):
            idx = torch.tensor([i for i in range(I) if delays[i] == d], device="cuda")
            s, b, r = ref_st[idx].contiguous(), ref_bf[idx].contiguous(), ref_rw[idx].contiguous()
            nlc.env_step(env, s, b, a[idx].contiguous(), d, DT, r)
            ref_st[idx], ref_bf[idx], ref_rw[idx] = s, b, r
        torch.cuda.synchronize()
        assert torch.equal(st, ref_st) and torch.equal(bf, ref_bf) and torch.equal(rw, ref_rw), it


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("env", ["oderl-pendulum", "oderl-cartpole", "oderl-acrobot"])
def test_env_step_per_instance_delays_match_reference_dynamics(env, dtype):
    """The 48 instances of each of the d0 / d1 / d3 goldens, interleaved in ONE call per step (delay tensor on the device),
    held to the bounds of test_gpu_episode.py (fp32) and test_gpu_episode_fp64.py (fp64)."""
    nlc = _nlc()
    g = load("env_step_" + short(env))
    ds = (0, 1, 3)
    n = g["d0_state0"].shape[0]
    # instance 3 k + j is instance k of the d = ds[j] golden
    st = torch.from_numpy(np.stack([g[f"d{d}_state0"] for d in ds], axis=1).reshape(3 * n, -1)).to(dtype).cuda().contiguous()
    bf = torch.from_numpy(np.stack([g[f"d{d}_buf0"] for d in ds], axis=1)).reshape(3 * n, *g["d0_buf0"].shape[1:]).to(dtype).cuda().contiguous()
    delays = torch.tensor(ds * n, dtype=torch.int32, device="cuda")
    rw = torch.zeros(3 * n, dtype=dtype, device="cuda")
    bound = 2e-5 if dtype == torch.float32 else 1e-12
    for it in range(g["d0_actions"].shape[0]):
        a = np.stack([g[f"d{d}_actions"][it] for d in ds], axis=1).reshape(3 * n, -1)
        nlc.env_step(env, st, bf, torch.from_numpy(a).to(dtype).cuda().contiguous(), delays, DT, rw)
        torch.cuda.synchronize()
        for j, d in enumerate(ds):
            assert torch.equal(bf[j::3].cpu(), torch.from_numpy(g[f"d{d}_bufs"][it]).to(dtype))
            es, er = relerr(g[f"d{d}_states"][it], st[j::3]), relerr(g[f"d{d}_rewards"][it], rw[j::3])
            assert es <= bound and er <= bound, (it, d, es, er)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_env_step_device_delay_check(dtype):
    """The C entry points check each delay on the device: an entry outside [0, B) sets the status word and leaves that
    instance untouched; the others step."""
    from neurallaplacecontrol_b200 import _lib

    lib = _lib.load()
    I, B = 3, 4
    st = torch.ones(I, 3, dtype=dtype, device="cuda")
    bf = torch.zeros(I, B, 1, dtype=dtype, device="cuda")
    a = torch.full((I, 1), 0.5, dtype=dtype, device="cuda")
    delays = torch.tensor([0, 4, -1], dtype=torch.int32, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    stream = _lib.current_stream_ptr()
    if dtype == torch.float32:
        ro = _lib.RolloutOpts()
        ro.env, ro.dynamics, ro.dt = 0, _lib.DYN_ANALYTIC_DELAY, DT
        rc = lib.nlc_env_step_delays(C.byref(ro), delays.data_ptr(), st.data_ptr(), bf.data_ptr(), a.data_ptr(), I, B, 1, None,
                                     status.data_ptr(), stream)
    else:
        rc = lib.nlc_env_step_f64_delays(0, delays.data_ptr(), DT, st.data_ptr(), bf.data_ptr(), a.data_ptr(), I, B, 1, None,
                                         status.data_ptr(), stream)
    assert rc == 0
    torch.cuda.synchronize()
    assert int(status) == 1
    assert not torch.equal(st[0], torch.ones(3, dtype=dtype, device="cuda")) and float(bf[0, -1, 0]) == 0.5
    assert torch.equal(st[1:], torch.ones(2, 3, dtype=dtype, device="cuda")) and torch.equal(bf[1:], torch.zeros(2, B, 1, dtype=dtype, device="cuda"))


# ---- the closed loop over the grid -------------------------------------------------------------------------------------
def test_closed_loop_grid_equals_single_instance_loops(monkeypatch):
    """run_closed_loop over 2 models x 2 delays x 2 seeds (one batch, per-instance delays) == 8 single-instance loops
    (MPPIDelay.command + env_step with I = 1), with the checks and bounds of
    test_gpu_episode.py::test_closed_loop_batch_equals_single_instance_loops."""
    monkeypatch.setenv("NLC_ROLLOUT_TILES", "1")
    from test_gpu_parity import make_model

    env, K, T, n_steps = "oderl-pendulum", 256, 10, 8
    nlc, nx, nu, common, _, _, _ = _setup(env, "fp32", 8, K, T)
    models = [make_model(env, True), _models(env)[1]]
    grid = [(m, d, s) for m in range(2) for d in (1, 3) for s in (7, 8)]
    I = len(grid)
    st0 = torch.tensor(load("env_step_pendulum")["d1_state0"][:I], dtype=torch.float64)
    batch = nlc.BatchedMPPIDelay([nlc.NLDynamics(models[m], DT) for m, _, _ in grid], nlc.EnvRunningCost(env), nx, nlc.noise_sigma_for(nu),
                                 I, seeds=[s for _, _, s in grid], **common)
    res = nlc.run_closed_loop(batch, env, st0, [d for _, d, _ in grid], n_steps, DT)
    assert res["total_reward_raw"].shape == (I,) and np.isfinite(res["total_reward_raw"]).all()
    assert list(res["delay"]) == [d for _, d, _ in grid]
    for i, (m, d, s) in enumerate(grid):
        p = nlc.MPPIDelay(nlc.NLDynamics(models[m], DT), nlc.EnvRunningCost(env), nx, nlc.noise_sigma_for(nu),
                          U_init=torch.zeros(T, nu, dtype=torch.float64), seed=s, keep_states=False, **common)
        st = st0[i:i + 1].float().cuda().contiguous()
        b = torch.zeros(1, 4, nu, device="cuda")
        r = torch.zeros(1, device="cuda")
        tot = 0.0
        for it in range(n_steps):
            a = p.command(st[0], b[0])
            nlc.env_step(env, st, b, a.float().reshape(1, nu).contiguous(), d, DT, r)
            tot += float(r[0])
        assert abs(tot - res["total_reward_raw"][i]) <= 1e-5 * max(1.0, abs(tot)), (i, tot, res["total_reward_raw"][i])
        assert relerr(st.double().cpu().numpy()[0], res["final_states"][i]) < 1e-6


def test_fp64_closed_loop_per_instance_delays_equal_single_loops():
    """run_closed_loop over fp64 planners (one model per instance) with per-instance delays == per-instance loops of
    command + fp64 env_step, bit for bit."""
    from test_gpu_parity import make_model, make_planner

    nlc = _nlc()
    env, I, K, T, n_steps, nu = "oderl-pendulum", 4, 256, 10, 6, 1
    delays, seeds = [0, 1, 2, 3], [51, 52, 53, 54]
    models = [make_model(env, True), make_model(env, False)]
    mk = lambda: [make_planner(env, models[i % 2], K, T, np.zeros((T, nu)), math_mode="fp64", keep_states=False, seed=seeds[i])  # noqa: E731
                  for i in range(I)]
    st0 = torch.tensor(load("env_step_pendulum")["d1_state0"][:I], dtype=torch.float64)
    res = nlc.run_closed_loop(mk(), env, st0, torch.tensor(delays), n_steps, DT)
    assert list(res["delay"]) == delays
    for i, p in enumerate(mk()):
        s = st0[i:i + 1].cuda().contiguous()
        b = torch.zeros(1, 4, nu, dtype=torch.float64, device="cuda")
        r = torch.zeros(1, dtype=torch.float64, device="cuda")
        tot = torch.zeros(1, dtype=torch.float64, device="cuda")
        for it in range(n_steps):
            a = p.command(s[0], b[0])
            nlc.env_step(env, s, b, a.reshape(1, nu).contiguous(), delays[i], DT, r)
            tot += r
        assert torch.equal(s.cpu(), torch.from_numpy(res["final_states"][i:i + 1])), i
        assert torch.equal(tot.cpu(), torch.from_numpy(res["total_reward_raw"][i:i + 1])), i


# ---- rejections --------------------------------------------------------------------------------------------------------
def test_rejections_launch_nothing():
    """Wrong lengths, mixed kinds, mismatched dims or dt and out-of-range delays raise before any kernel launch."""
    nlc = _nlc()
    lib = nlc._lib.load()
    env, I, K, T = "oderl-pendulum", 4, 256, 6
    _, nx, nu, common, U0, states, bufs = _setup(env, "tc_split3", I, K, T)
    from test_gpu_multi_time import _model, _state_dict

    m = _models(env)[0]
    acro = _model("oderl-acrobot", _state_dict("oderl-acrobot"))
    nl, an = nlc.NLDynamics(m, DT), nlc.AnalyticDelayDynamics(env, 1, DT)
    cost, sig = nlc.EnvRunningCost(env), nlc.noise_sigma_for(nu)
    n0 = lib.nlc_launch_count()
    bad = [
        (ValueError, [nl] * (I - 1)),                                          # one handle short
        (TypeError, [nl, an, nl, an]),                                         # mixed kinds
        (ValueError, [nl, nlc.NLDynamics(acro, DT), nl, nl]),                  # another environment's model
        (ValueError, [nl, nlc.NLDynamics(m, 0.1), nl, nl]),                    # another dt
        (ValueError, [an, nlc.AnalyticDelayDynamics(env, 4, DT), an, an]),     # delay outside the 4-entry buffer
        (ValueError, [an, nlc.AnalyticDelayDynamics("oderl-cartpole", 1, DT), an, an]),  # another environment
    ]
    for exc, dyns in bad:
        with pytest.raises(exc):
            nlc.BatchedMPPIDelay(dyns, cost, nx, sig, I, **common)
    s = torch.zeros(I, nx, device="cuda")
    b = torch.zeros(I, 4, nu, device="cuda")
    a = torch.zeros(I, nu, device="cuda")
    for exc, delays in ((ValueError, [0, 1, 2]), (ValueError, [0, 1, 2, 4]), (ValueError, [0, -1, 2, 3]), (TypeError, [0.0, 1.0, 2.0, 3.0])):
        with pytest.raises(exc):
            nlc.env_step(env, s, b, a, delays)
        with pytest.raises(exc):
            nlc.env_step(env, s.double(), b.double(), a.double(), delays)
    batch = nlc.BatchedMPPIDelay([an] * I, cost, nx, sig, I, **common)
    with pytest.raises(ValueError):
        nlc.run_closed_loop(batch, env, states, [0, 1, 2, 4], 2, DT)
    torch.cuda.synchronize()
    assert lib.nlc_launch_count() == n0
    assert not s.any() and not b.any()

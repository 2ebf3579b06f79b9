"""Stage 4 with sample costs that overflow fp32, against the fp64 oracle on the same inputs.

A cost of +inf (one cost term past 3.4e38: the cartpole ``state_constraint`` term exp(10 err_x + 7) once err_x > 8.17) or a
cost more than 2.4e38 above the minimum weighs exp(-inf) = 0 in the reference (``mppi_delay.py:210-211``): the plan comes from
the other samples.  These tests hold every fp32-class path to that - the stage kernels at the rows where their loops split
(block boundaries of the sum kernel, the scalar tail of the min kernel), the shard combine with a shard that overflowed
entirely, the planner in every math mode, sharded planners (host gather and device mailboxes), the instance-batched planner
- and pin the cases where the reference itself is NaN (every cost +inf, a NaN cost) so that they stay NaN.  The environment
step keeps a NaN action NaN, as the reference's ``torch.clamp`` does."""
import functools

import numpy as np
import pytest
import torch

from _util import DT, START_STATE, action_relerr, injected_noise, relerr, weights

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

INF = float("inf")
FLT_MAX = float(np.finfo(np.float32).max)
ENV = "oderl-cartpole"
COST_OPTS = dict(state_constraint=True, change_goal=True, change_goal_flipped=True)  # goal x = +2


def _nlc():
    import neurallaplacecontrol_b200 as nlc

    return nlc


def _sum_rows_per_block(K):
    """softmax_sum_kernel's partition of the K rows (stage4_update.cu: sum_grid, rows_per_block)."""
    grid = min(max((K + 255) // 256, 1), 148 * 4)
    return grid, (K + grid - 1) // grid


def _edge_rows(case, K, cost):
    """Rows where the stage-4 kernels change how they walk the costs."""
    grid, rpb = _sum_rows_per_block(K)
    if case == "first_last":
        return [0, K - 1]
    if case == "block_boundary":  # either side of the boundary between two sum-kernel blocks
        b = rpb * max(grid // 2, 1)
        return [r for r in (b - 1, b) if r < K]
    if case == "scalar_tail":  # the min kernel reads float4s, then the last K mod 4 rows one by one
        return list(range(K - K % 4, K))
    if case == "next_to_argmin":
        a = int(torch.argmin(cost))
        return [a + 1 if a + 1 < K else a - 1]
    raise KeyError(case)


def _stage4(cost32, noise32, U, lam, G):
    """nlc_softmax_partial per shard + nlc_softmax_combine: (U, action, stats, weights)."""
    from test_gpu_stages import _lib, _softmax

    L = _lib()
    lib = L.load()
    T, nu = noise32.shape[1:]
    triples, w = _softmax(cost32, noise32, lam, G)
    Ud = U.float().cuda().contiguous()
    action = torch.empty(nu, device="cuda")
    stats = torch.empty(2, device="cuda")
    L.check(lib.nlc_softmax_combine(triples.data_ptr(), G, T, nu, lam, 3.0, Ud.data_ptr(), action.data_ptr(), stats.data_ptr(),
                                    L.current_stream_ptr()))
    torch.cuda.synchronize()
    return Ud, action, stats, w


def _stage4_inputs(K, T=6, nu=2):
    g = torch.Generator().manual_seed(K)
    cost = (torch.rand(K, generator=g, dtype=torch.float64) * 40 - 5).float()
    noise = torch.randn(K, T, nu, generator=g, dtype=torch.float64).float()
    U = torch.randn(T, nu, generator=g, dtype=torch.float64)
    return cost, noise, U


# ---- A: the stage kernels ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["first_last", "block_boundary", "scalar_tail", "next_to_argmin", "all_but_one", "gap_3e38",
                                  "gap_1e36_small_lambda"])
@pytest.mark.parametrize("K", [7, 1027, 65537])
def test_stage4_overflowing_costs_weigh_zero(K, case):
    """+inf costs at the rows where the kernels split their loops, every row but one +inf, and finite gaps to the minimum that
    overflow exp's argument (3e38 at lambda = 1; 1e36 at lambda = 1e-3): U, action and weights as the fp64 oracle computes them
    from the same fp32 costs, weight exactly 0 on those rows, beta exact; the same U from 2, 4 and 8 shards."""
    from oracle import mppi

    cost, noise, U = _stage4_inputs(K)
    lam = 0.7
    if case == "all_but_one":
        rows = [k for k in range(K) if k != K // 3]
    elif case.startswith("gap"):
        rows = [k for k in range(0, K, 3) if k != int(torch.argmin(cost))]
    else:
        rows = _edge_rows(case, K, cost)
    if case == "gap_3e38":
        lam = 1.0
        cost[rows] = 3e38
    elif case == "gap_1e36_small_lambda":
        lam = 1e-3
        cost = cost * 1e-3  # gaps of up to 0.04 between the finite costs: weights down to exp(-40)
        cost[rows] = 1e36
    else:
        cost[rows] = INF
    assert rows
    U_ref, w_ref, _ = mppi.softmax_update(U, cost.double(), noise.double(), lam)
    assert torch.isfinite(U_ref).all() and (w_ref[rows] == 0).all()
    results = []
    for G in (1, 2, 4, 8):
        if K < G:
            continue
        Ud, action, stats, w = _stage4(cost.cuda(), noise.cuda(), U, lam, G)
        assert torch.isfinite(Ud).all(), (G, Ud)
        assert relerr(U_ref, Ud) < 2e-5, (G, relerr(U_ref, Ud))
        assert relerr(U_ref[0] * 3.0, action) < 2e-5
        assert float(stats[0]) == float(cost.min())
        if G == 1:
            assert relerr(w_ref, w) < 1e-5
            assert (w[rows] == 0.0).all()
        results.append(Ud)
    for r in results[1:]:
        assert relerr(results[0], r) < 1e-5


@pytest.mark.parametrize("K", [7, 1027, 65537])
def test_stage4_nan_cases_of_the_reference_stay_nan(K):
    """Where the reference's update is NaN the kernels' is too: every cost +inf (beta = +inf, exp(-(inf - inf))) gives a NaN
    U; one NaN cost makes U and every omega NaN."""
    from oracle import mppi

    cost, noise, U = _stage4_inputs(K)
    every = torch.full_like(cost, INF)
    U_ref, _, _ = mppi.softmax_update(U, every.double(), noise.double(), 0.7)
    assert torch.isnan(U_ref).all()
    Ud, action, _, _ = _stage4(every.cuda(), noise.cuda(), U, 0.7, 1)
    assert torch.isnan(Ud).all() and torch.isnan(action).all()
    one = cost.clone()
    one[K // 2] = float("nan")
    U_ref, _, omega_ref = mppi.softmax_update(U, one.double(), noise.double(), 0.7)
    assert torch.isnan(U_ref).all() and torch.isnan(omega_ref).all()
    Ud, _, stats, w = _stage4(one.cuda(), noise.cuda(), U, 0.7, 1)
    assert torch.isnan(Ud).all() and torch.isnan(w / stats[1]).all()


# ---- B: the shard combine ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["inf_shard", "far_shard"])
@pytest.mark.parametrize("G", [2, 4, 8])
def test_shard_combine_with_an_overflowing_shard(G, case):
    """One shard's costs all +inf (its beta_g is +inf), or all more than 2.4e38 above the global minimum: that shard weighs 0
    in the combine, and every U is finite and the unsharded one."""
    from oracle import mppi

    K = 4099
    cost, noise, U = _stage4_inputs(K)
    idx = torch.tensor_split(torch.arange(K), G)[1]
    lam = 0.7
    if case == "inf_shard":
        cost[idx] = INF
    else:
        lam = 1.0
        cost[idx] = 3e38 + cost[idx] * 1e36
    U_ref, _, _ = mppi.softmax_update(U, cost.double(), noise.double(), lam)
    U1, _, _, _ = _stage4(cost.cuda(), noise.cuda(), U, lam, 1)
    UG, _, _, _ = _stage4(cost.cuda(), noise.cuda(), U, lam, G)
    assert torch.isfinite(U1).all() and torch.isfinite(UG).all()
    assert relerr(U_ref, U1) < 2e-5
    assert relerr(U1, UG) < 1e-5, relerr(U1, UG)


# ---- C: the planner ---------------------------------------------------------------------------------------------------
def _cartpole_states(K, rows11, rows80, seed):
    """Per-sample start states near the start state; rows11 start at x = 11.5 (an fp32 cost of +inf, finite in fp64: ~1e44 -
    x = 11.5 rather than 11 because the calibrated model drifts the cart back by ~0.1 a step), rows80 at x = 80 (+inf in
    both)."""
    g = torch.Generator().manual_seed(seed)
    st = torch.tensor(START_STATE[ENV], dtype=torch.float64).repeat(K, 1) + 0.01 * torch.randn(K, 5, generator=g, dtype=torch.float64)
    st[rows11, 0] = 11.5
    st[rows80, 0] = 80.0
    return st


def _oracle_plan(dynamics, states, noise, T):
    from oracle import costs, mppi

    return mppi.command(torch.zeros(T, 1, dtype=torch.float64), states, torch.zeros(4, 1, dtype=torch.float64), noise, dynamics,
                        costs.running_cost(ENV, **COST_OPTS), noise_sigma=mppi.noise_sigma_for(1), u_scale=3.0, u_min=-3.0, u_max=3.0)


@functools.lru_cache(maxsize=None)
def _planner_scenario(dyn):
    """(states, noise, oracle plan, rows11, rows80) of a K = 1027 cartpole plan, the rows chosen as in the stage tests."""
    from oracle import dynamics, mppi

    K, T = 1027, 5
    noise = injected_noise(K, T, 1, seed=17)
    fn = mppi.make_nl_dynamics(weights(ENV, calibrated=True), DT) if dyn == "nl" else dynamics.make_analytic_dynamics(ENV, DT, 1)
    base = _oracle_plan(fn, _cartpole_states(K, [], [], 3), noise, T)
    a = int(torch.argmin(base["cost_total"]))
    tail = [r for r in _edge_rows("scalar_tail", K, None) if r != a]
    rows11 = sorted({0, K - 1, *_edge_rows("next_to_argmin", K, base["cost_total"]), *tail[::2]})
    rows80 = [r for r in _edge_rows("block_boundary", K, None) + tail[1::2] if r not in rows11]
    states = _cartpole_states(K, rows11, rows80, 3)
    return states, noise, _oracle_plan(fn, states, noise, T), rows11, rows80


@pytest.mark.parametrize("mode", ["analytic", "fp32", "tc_split3_one_tile", "tc_split3_ping_pong", "tc_fp16", "fp64"])
def test_planner_overflowing_sample_costs(mode, monkeypatch):
    """Cartpole with the state_constraint reward: samples that start at x = 11.5 or x = 80 cost +inf in fp32 and weigh 0; the
    plan is the oracle's from the other samples, in every math mode (fp64: the x = 11.5 costs are finite, ~1e44)."""
    from test_gpu_parity import make_model

    nlc = _nlc()
    if mode.startswith("tc_split3"):
        monkeypatch.setenv("NLC_ROLLOUT_TILES", "1" if mode.endswith("one_tile") else "3")
    math_mode = {"analytic": "fp32", "tc_split3_one_tile": "tc_split3", "tc_split3_ping_pong": "tc_split3"}.get(mode, mode)
    states, noise, ref, rows11, rows80 = _planner_scenario("analytic" if mode == "analytic" else "nl")
    K, T = noise.shape[:2]
    c_ref = ref["cost_total"]
    over = torch.zeros(K, dtype=torch.bool)
    over[rows11 + rows80] = True
    # the scenario's premise, from the oracle
    assert (c_ref[rows11] > 1e3 * FLT_MAX).all() and torch.isfinite(c_ref[rows11]).all()
    assert (c_ref[rows80] == INF).all()
    assert (c_ref[~over] < 1e-3 * FLT_MAX).all()
    dyn = nlc.AnalyticDelayDynamics(ENV, 1, DT) if mode == "analytic" else nlc.NLDynamics(make_model(ENV, True, math_mode=math_mode), DT)
    p = nlc.MPPIDelay(dyn, nlc.EnvRunningCost(ENV, **COST_OPTS), 5, nlc.noise_sigma_for(1), num_samples=K, horizon=T,
                      device="cuda:0", lambda_=1.0, u_min=torch.tensor(-3.0), u_max=torch.tensor(3.0), u_scale=3.0,
                      U_init=torch.zeros(T, 1, dtype=torch.float64), math_mode=math_mode)
    p.noise_dist.sample = lambda shape: noise.clone()
    action = p.command(states, torch.zeros(4, 1, dtype=torch.float64))
    torch.cuda.synchronize()
    cost = p.cost_total.double().cpu()
    tol_c, tol_u = {"tc_fp16": (2e-2, 5e-2), "fp64": (1e-10, 1e-10)}.get(mode, (1e-4, 1e-4))
    assert relerr(c_ref[~over], cost[~over]) < tol_c, relerr(c_ref[~over], cost[~over])
    if mode == "fp64":
        assert ((cost[rows11] - c_ref[rows11]).abs() / c_ref[rows11]).max() < 1e-10
        assert (cost[rows80] == INF).all()
    else:
        assert (cost[over] == INF).all(), cost[over]  # +inf, not NaN
    omega, nz = p.omega.double().cpu(), p.cost_total_non_zero.double().cpu()
    assert (omega[over] == 0.0).all() and (nz[over] == 0.0).all()
    assert abs(float(omega.sum()) - 1.0) < 1e-5
    assert relerr(ref["U"], p.U) < tol_u, relerr(ref["U"], p.U)
    assert action_relerr(ref["action"], action, ref["U"], 3.0) < tol_u


# ---- D: the sharded planner -------------------------------------------------------------------------------------------
def test_sharded_planner_with_an_overflowing_shard():
    """Four shards of one plan on one GPU: every sample of shard 2 starts at x = 80 (that shard's beta_g is +inf), scattered
    x = 11.5 samples in the others.  Through the host gather and through the device mailboxes every shard ends with the same
    finite U, the unsharded planner's."""
    from test_gpu_parity import make_model

    nlc = _nlc()
    G, K, T = 4, 1024, 5
    rows11 = [3, 300, 1000, 1023]
    rows80 = list(range(512, 768))
    states = _cartpole_states(K, rows11, rows80, 5)
    noise = injected_noise(K, T, 1, seed=23)
    buf = torch.zeros(4, 1, dtype=torch.float64)
    m = make_model(ENV, True, math_mode="tc_split3")

    def planner(**kw):
        p = nlc.MPPIDelay(nlc.NLDynamics(m, DT), nlc.EnvRunningCost(ENV, **COST_OPTS), 5, nlc.noise_sigma_for(1), num_samples=K,
                          horizon=T, device="cuda:0", lambda_=1.0, u_min=torch.tensor(-3.0), u_max=torch.tensor(3.0), u_scale=3.0,
                          U_init=torch.zeros(T, 1, dtype=torch.float64), **kw)
        p.noise_dist.sample = lambda shape: noise.clone()
        return p

    whole = planner()
    whole.command(states, buf)
    torch.cuda.synchronize()
    U1 = whole.U.clone()
    assert torch.isfinite(U1).all()
    res = {}
    for mode in ("mailbox", "gather"):
        shards = [planner(shard=(r, G)) for r in range(G)]
        if mode == "mailbox":
            shards[0].connect_local_shards(shards)
        for p in shards:
            assert p._begin(states, buf) is None
        assert float(shards[2].shard_triple[0]) == INF
        if mode == "gather":
            triples = torch.stack([p.shard_triple.clone() for p in shards])
            for p in shards:
                p.all_triples.copy_(triples)
        acts = [p._finish().clone() for p in shards]
        torch.cuda.synchronize()
        if mode == "mailbox":
            assert shards[0].exchange_status() == (True, 0)
        for p, a in zip(shards, acts):
            assert torch.isfinite(p.U).all() and torch.isfinite(a).all(), mode
            assert torch.equal(p.U, shards[0].U) and torch.equal(a, acts[0]), mode
        assert relerr(U1, shards[0].U) < 1e-5, (mode, relerr(U1, shards[0].U))
        res[mode] = shards[0].U.clone()
    assert torch.equal(res["mailbox"], res["gather"])


# ---- E: the instance-batched planner ----------------------------------------------------------------------------------
def test_batched_planner_instances_near_and_beyond_overflow():
    """Three analytic cartpole instances: near the start state (finite), near the overflow edge (part of the samples cost +inf
    within the horizon: the oracle's argmin and U), and at x = 80 (every cost +inf: NaN, like the reference).  Each is
    bit-identical to a stand-alone MPPIDelay on the same inputs."""
    from oracle import dynamics

    nlc = _nlc()
    I, K, T = 3, 512, 10
    states = torch.tensor([START_STATE[ENV], [9.6, 1.0, -1.0, 0.0, 0.0], [80.0, 0.0, -1.0, 0.0, 0.0]], dtype=torch.float64)
    bufs = torch.zeros(I, 4, 1, dtype=torch.float64)
    noise = torch.stack([injected_noise(K, T, 1, seed=9 + i) for i in range(I)])
    common = dict(num_samples=K, horizon=T, device="cuda:0", lambda_=1.0, u_min=torch.tensor(-3.0), u_max=torch.tensor(3.0),
                  u_scale=3.0, math_mode="fp32", keep_states=False)
    dyn = nlc.AnalyticDelayDynamics(ENV, 1, DT)
    U0 = torch.zeros(T, 1, dtype=torch.float64)
    batch = nlc.BatchedMPPIDelay(dyn, nlc.EnvRunningCost(ENV, **COST_OPTS), 5, nlc.noise_sigma_for(1), I, seeds=[1, 2, 3], U_init=U0,
                                 **common)
    act_b = batch.command(states, bufs, noise=noise)
    torch.cuda.synchronize()
    refs = [_oracle_plan(dynamics.make_analytic_dynamics(ENV, DT, 1), states[i], noise[i], T) for i in range(I)]
    frac = float((refs[1]["cost_total"] > FLT_MAX).double().mean())
    assert 0.05 < frac < 0.95, frac  # premise: instance 1 sits on the overflow edge
    bits = lambda t: t.float().contiguous().view(torch.int32)  # NaN-safe bit identity
    for i in range(I):
        p = nlc.MPPIDelay(dyn, nlc.EnvRunningCost(ENV, **COST_OPTS), 5, nlc.noise_sigma_for(1), U_init=U0, seed=i + 1, **common)
        p.noise_dist.sample = lambda shape, nz=noise[i]: nz.clone()
        a = p.command(states[i].cuda(), bufs[i].cuda())
        torch.cuda.synchronize()
        assert torch.equal(bits(p.cost_total), bits(batch.cost_total[i])), i
        assert torch.equal(bits(p.U), bits(batch.U[i])) and torch.equal(bits(a), bits(act_b[i])), i
    for i in (0, 1):
        assert torch.isfinite(batch.U[i]).all() and torch.isfinite(act_b[i]).all(), i
    c1 = batch.cost_total[1].double().cpu()
    assert int(torch.argmin(c1)) == int(torch.argmin(refs[1]["cost_total"]))
    assert relerr(refs[1]["U"], batch.U[1]) < 1e-4, relerr(refs[1]["U"], batch.U[1])
    assert torch.isnan(refs[2]["U"]).all() and torch.isnan(batch.U[2]).all() and torch.isnan(act_b[2]).all()


# ---- F: the environment step ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("env", ["oderl-pendulum", "oderl-cartpole", "oderl-acrobot"])
def test_env_step_nan_action_stays_nan(env, dtype):
    """A NaN action reaches the dynamics as NaN (torch.clamp keeps it; a min/max clamp would apply the lower bound): that
    instance's state and reward are NaN where the oracle's are, every other instance is untouched by it."""
    from oracle import costs, dynamics

    nlc = _nlc()
    nx, nu = costs.ENV_DIMS[env]
    I, B, bad = 8, 4, 3
    g = torch.Generator().manual_seed(nx)
    st0 = torch.tensor(START_STATE[env], dtype=torch.float64).repeat(I, 1) + 0.1 * torch.randn(I, nx, generator=g, dtype=torch.float64)
    bf0 = torch.rand(I, B, nu, generator=g, dtype=torch.float64) * 2 - 1
    a_fin = torch.rand(I, nu, generator=g, dtype=torch.float64) * 2 - 1
    a_nan = a_fin.clone()
    a_nan[bad] = float("nan")
    out = {}
    for name, a in (("nan", a_nan), ("finite", a_fin)):
        st, bf = st0.to(dtype).cuda().contiguous(), bf0.to(dtype).cuda().contiguous()
        rw = torch.zeros(I, dtype=dtype, device="cuda")
        nlc.env_step(env, st, bf, a.to(dtype).cuda().contiguous(), 0, DT, rw)
        torch.cuda.synchronize()
        out[name] = (st.cpu(), bf.cpu(), rw.cpu())
    ref_s, _, ref_r = dynamics.env_step(env, st0.to(dtype).double(), bf0.to(dtype).double(), a_nan.to(dtype).double(), 0, DT)
    st, bf, rw = out["nan"]
    assert torch.isnan(ref_s[bad]).any() and torch.isnan(ref_r[bad])
    assert torch.equal(torch.isnan(st[bad]), torch.isnan(ref_s[bad])), (st[bad], ref_s[bad])
    assert torch.isnan(rw[bad])
    keep = [i for i in range(I) if i != bad]
    fs, fb, fr = out["finite"]
    assert torch.equal(st[keep], fs[keep]) and torch.equal(bf[keep], fb[keep]) and torch.equal(rw[keep], fr[keep])

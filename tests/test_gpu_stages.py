"""Stage-level parity through the C ABI: on-device Philox sampling, the two-pass softmax update and its K-sharded
combine, the generic Fourier ILT kernel, and size-independent properties at BASELINE.json's full sizes."""
import ctypes as C

import numpy as np
import pytest
import torch

from _util import DT, relerr, weights

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)


def _lib():
    from neurallaplacecontrol_b200 import _lib as L

    return L


def _params(K, T, nu, B=4, k_offset=0, k_total=None, u_scale=2.0, bound=2.0, lam=1.0):
    from oracle import mppi

    L = _lib()
    p = L.MppiParams()
    p.K, p.T, p.nu, p.B = K, T, nu, B
    p.k_offset, p.k_total = k_offset, K if k_total is None else k_total
    p.lambda_, p.u_scale, p.has_bounds = lam, u_scale, 1
    for i in range(nu):
        p.u_min[i], p.u_max[i] = -bound, bound
    sig = mppi.noise_sigma_for(nu)
    sinv, chol = torch.inverse(sig), torch.linalg.cholesky(sig)
    for i in range(nu):
        for j in range(nu):
            p.sigma_inv[i * nu + j] = float(sinv[i, j])
            p.sigma_chol[i * nu + j] = float(chol[i, j])
    return p, chol


def _perturb(p, U, noise_in, buf, seed=0, call=0):
    L = _lib()
    lib = L.load()
    K, T, nu, B = p.K, p.T, p.nu, p.B
    dev = "cuda"
    out = {k: torch.empty(K, T, nu, device=dev) for k in ("perturbed", "noise", "actions")}
    out["hist"] = torch.empty(K, B - 1 + T, nu, device=dev)
    out["pert_cost"] = torch.empty(K, device=dev)
    Ud = U.to(dev, torch.float32).contiguous()
    Uc = torch.empty_like(Ud)
    bufd = buf.to(dev, torch.float32).contiguous()
    L.check(lib.nlc_perturb(C.byref(p), Ud.data_ptr(), Uc.data_ptr(), 0, L.ptr(noise_in), seed, call, bufd.data_ptr(),
                            out["perturbed"].data_ptr(), out["noise"].data_ptr(), out["hist"].data_ptr(),
                            out["actions"].data_ptr(), out["pert_cost"].data_ptr(), L.current_stream_ptr()))
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("nu", [1, 2])
def test_philox_sampler_matches_oracle_and_is_shard_invariant(nu):
    from oracle import philox

    K, T = 512, 20
    U = torch.zeros(T, nu)
    buf = torch.zeros(4, nu)
    p, chol = _params(K, T, nu, bound=1e9, u_scale=1.0)
    full = _perturb(p, U, None, buf, seed=1234567890123, call=7)
    ref = philox.sampled_noise(K, T, nu, 0, 1234567890123, 7, chol.numpy(), np.zeros(nu))
    assert np.abs(full["noise"].cpu().numpy() - ref).max() < 2e-5
    # a shard starting at global sample 128 draws exactly the same numbers (bit-exact sample indexing)
    ps, _ = _params(64, T, nu, k_offset=128, k_total=K, bound=1e9, u_scale=1.0)
    part = _perturb(ps, U, None, buf, seed=1234567890123, call=7)
    assert torch.equal(part["noise"], full["noise"][128:192])
    other = _perturb(ps, U, None, buf, seed=1234567890123, call=8)
    assert not torch.equal(other["noise"], part["noise"])


def _softmax(cost, noise, lam, G):
    L = _lib()
    lib = L.load()
    K, T, nu = noise.shape
    TN = T * nu
    idx = torch.tensor_split(torch.arange(K), G)
    triples = torch.empty(G, 2 + TN, device="cuda")
    weights_out = torch.empty(K, device="cuda")
    for g, ix in enumerate(idx):
        c = cost[ix].contiguous()
        n = noise[ix].contiguous()
        ws = torch.empty(int(lib.nlc_softmax_workspace_bytes(len(ix), TN)), dtype=torch.uint8, device="cuda")
        w = torch.empty(len(ix), device="cuda")
        L.check(lib.nlc_softmax_partial(c.data_ptr(), n.data_ptr(), len(ix), T, nu, lam, triples[g].data_ptr(),
                                        w.data_ptr(), ws.data_ptr(), L.current_stream_ptr()))
        weights_out[ix.cuda()] = w
    return triples, weights_out


@pytest.mark.parametrize("K,T,nu", [(1, 1, 1), (7, 3, 2), (1000, 20, 1), (8192, 30, 1), (65536, 50, 2), (513, 256, 1), (300, 128, 2)])
def test_softmax_update_and_shard_combine(K, T, nu):
    from oracle import mppi

    L = _lib()
    lib = L.load()
    g = torch.Generator().manual_seed(K)
    cost = (torch.rand(K, generator=g, dtype=torch.float64) * 40 - 5)
    noise = torch.randn(K, T, nu, generator=g, dtype=torch.float64)
    U = torch.randn(T, nu, generator=g, dtype=torch.float64)
    lam = 0.7
    U_ref, w_ref, omega_ref = mppi.softmax_update(U, cost, noise, lam)
    c32, n32 = cost.float().cuda(), noise.float().cuda()
    results = []
    for G in (1, 2, 4, 8):
        if K < G:
            continue
        triples, w = _softmax(c32, n32, lam, G)
        Ud = U.float().cuda().contiguous()
        action = torch.empty(nu, device="cuda")
        stats = torch.empty(2, device="cuda")
        L.check(lib.nlc_softmax_combine(triples.data_ptr(), G, T, nu, lam, 3.0, Ud.data_ptr(), action.data_ptr(),
                                        stats.data_ptr(), L.current_stream_ptr()))
        torch.cuda.synchronize()
        assert relerr(U_ref, Ud) < 2e-5, (G, relerr(U_ref, Ud))
        assert relerr(U_ref[0] * 3.0, action) < 2e-5
        assert abs(float(stats[0]) - float(cost.float().min())) == 0.0  # min is exact
        if G == 1:
            assert relerr(w_ref, w) < 1e-5
        results.append(Ud.clone())
    for r in results[1:]:
        assert relerr(results[0], r) < 1e-5  # sharding changes only the summation order


@pytest.mark.parametrize("S", [1, 2, 17, 18, 33, 34, 48, 64, 65, 129, 200, 300])
@pytest.mark.parametrize("per_row", [False, True])
def test_fourier_ilt_kernel_matches_oracle(S, per_row):
    from neurallaplacecontrol_b200 import fourier_ilt
    from oracle import ilt

    N, n_t = 77, 13  # 1001 rows: 31 full 32-row chunks + a 9-row tail
    g = torch.Generator().manual_seed(S)
    F = torch.complex(torch.rand(N, n_t, S, generator=g) * 2 - 1, torch.rand(N, n_t, S, generator=g) * 2 - 1)
    t = (torch.arange(n_t, dtype=torch.float32) + 1) * 0.05
    if per_row:
        t = 0.01 + torch.rand(N, n_t, generator=g) * 2.0
    out = fourier_ilt(F.cuda(), t.cuda())
    t64 = t.double().expand(N, n_t)
    T64 = ilt.SCALE * (t64 + ilt.EPS)
    ref = ilt.fourier_line_integrate(F.real.double(), F.imag.double(), t64, T64)
    assert relerr(ref, out) < 2e-5, relerr(ref, out)


@pytest.mark.parametrize("N,n_t", [(1, 5), (2, 16), (3, 32), (40, 700)])
def test_fourier_ilt_ragged_shapes(N, n_t):
    """fewer than 32 rows, exactly whole 32-row blocks, and a time grid longer than the kernel's constant table"""
    from neurallaplacecontrol_b200 import fourier_ilt
    from oracle import ilt

    S = 33
    g = torch.Generator().manual_seed(N * 1000 + n_t)
    F = torch.complex(torch.rand(N, n_t, S, generator=g) * 2 - 1, torch.rand(N, n_t, S, generator=g) * 2 - 1)
    t = (torch.arange(n_t, dtype=torch.float32) + 1) * 0.01
    out = fourier_ilt(F.cuda(), t.cuda())
    t64 = t.double().expand(N, n_t)
    ref = ilt.fourier_line_integrate(F.real.double(), F.imag.double(), t64, ilt.SCALE * (t64 + ilt.EPS))
    assert relerr(ref, out) < 2e-5, relerr(ref, out)


def test_fourier_ilt_closed_form_pair():
    """1/(s+1) <-> exp(-t) through the kernel with the oracle's s-points (truncation error of the series itself)."""
    from neurallaplacecontrol_b200 import fourier_ilt
    from oracle import ilt

    t = torch.tensor([0.05, 0.1, 0.2, 0.5, 1.0], dtype=torch.float64)
    S = 129
    s_re, s_im, T = ilt.fourier_s_points(t, S)
    Fs = 1.0 / (torch.complex(s_re, s_im) + 1.0)
    out = fourier_ilt(Fs.to(torch.complex64).unsqueeze(0).cuda(), t.float().cuda())
    want = ilt.fourier_ilt_of(lambda s: 1.0 / (s + 1.0), t, S)
    assert relerr(want, out[0]) < 1e-4
    assert (out[0].double().cpu() - torch.exp(-t)).abs().max() < 0.1


def test_cfg3_full_size_properties():
    """BASELINE config 3 shape (cartpole K=8192 H=30): size-independent properties + sharding invariance of the costs."""
    import neurallaplacecontrol_b200 as nlc
    from oracle import costs
    from test_gpu_parity import make_model

    env = "oderl-cartpole"
    nx, nu = costs.ENV_DIMS[env]
    ah = np.float32(costs.ENV_ACT_HIGH[env])
    K, T = 8192, 30
    m = make_model(env, True)
    g = torch.Generator().manual_seed(1)
    noise = torch.randn(K, T, nu, generator=g, dtype=torch.float64)
    state = np.array([0.0, 0.0, -1.0, 1.2246467991473532e-16, 0.0])
    buf = torch.zeros(4, nu, dtype=torch.float64)

    def run(Kloc, off):
        p = nlc.MPPIDelay(nlc.NLDynamics(m, DT), nlc.EnvRunningCost(env), nx, nlc.noise_sigma_for(nu), num_samples=Kloc,
                          horizon=T, device="cuda:0", u_min=torch.tensor(-ah), u_max=torch.tensor(ah), u_scale=ah,
                          U_init=torch.zeros(T, nu, dtype=torch.float64))
        p.noise_dist.sample = lambda shape: noise[off:off + Kloc].clone()
        a = p.command(state, buf)
        return p, a

    p, a = run(K, 0)
    assert torch.isfinite(p.cost_total).all() and torch.isfinite(a).all()
    assert abs(float(p.omega.sum()) - 1.0) < 1e-4
    assert float(p.perturbed_action.abs().max()) * float(ah) <= float(ah) * (1 + 1e-6)
    assert float(a.abs().max()) <= float(ah) * (1 + 1e-6)
    # per-sample costs do not depend on which shard (which CTA tiling) computed them
    p2, _ = run(K // 4, K // 2)
    assert torch.equal(p2.cost_total, p.cost_total[K // 2:K // 2 + K // 4])
    # a zero-noise plan leaves U at zero cost-weighted mean of zero noise
    p.noise_dist.sample = lambda shape: torch.zeros(K, T, nu, dtype=torch.float64)
    p.U = torch.zeros(T, nu)
    p.command(state, buf)
    assert float(p.U.abs().max()) == 0.0
    assert float((p.cost_total - p.cost_total[0]).abs().max()) == 0.0


# ---------------------------------------------------------------------------------------------------------------------
# tcgen05 path
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,n_off,rows_b", [(64, 0, 64), (128, 0, 192), (192, 0, 192), (64, 128, 192), (256, 0, 256)])
@pytest.mark.parametrize("split3", [0, 1])
def test_umma_selftest_gemm(N, n_off, rows_b, split3):
    """Operand layout / descriptors / TMEM addressing of the tensor-core encoder: D = A B[n_off:n_off+N]^T.
    split3 (fp16 hi+lo, 3 MMAs, fp32 accumulate) must be fp32-class; the single pass carries fp16 input rounding."""
    L = _lib()
    lib = L.load()
    g = torch.Generator().manual_seed(N + n_off + split3)
    A = (torch.rand(128, 64, generator=g, dtype=torch.float64) * 2 - 1)
    Bm = (torch.randn(rows_b, 64, generator=g, dtype=torch.float64) * 0.3)
    D = torch.full((128, N), float("nan"), device="cuda")
    Ad, Bd = A.float().cuda().contiguous(), Bm.float().cuda().contiguous()
    L.check(lib.nlc_selftest_umma_gemm(Ad.data_ptr(), Bd.data_ptr(), rows_b, n_off, N, split3, D.data_ptr(), L.current_stream_ptr()))
    torch.cuda.synchronize()
    ref = A.float().double() @ Bm.float().double()[n_off:n_off + N].T
    err = relerr(ref, D)
    assert err < (2e-6 if split3 else 2e-3), err


@pytest.mark.parametrize("mode,tol", [("tc_split3", 2e-5), ("tc_fp16", 5e-3)])
@pytest.mark.parametrize("env", ["oderl-pendulum", "oderl-acrobot"])
def test_tc_encoder_matches_reference(env, mode, tol):
    """ReverseGRUEncoder on tcgen05 vs the reference's own encoder output (golden p_action) and vs the FFMA kernel on
    a multi-tile, ragged history (K*T = 3*128 + 37 windows)."""
    import ctypes as C

    from oracle import costs
    from test_gpu_parity import make_model
    from _util import load, short

    L = _lib()
    lib = L.load()
    g = load("model_fwd_" + short(env))
    m = make_model(env, calibrated=False, math_mode=mode)
    obs, act = torch.from_numpy(g["obs"]).cuda(), torch.from_numpy(g["act"]).cuda()
    m(obs, act, torch.from_numpy(g["ts_fixed"]).cuda())
    assert relerr(g["p_action"], m.last_p_action) < tol, relerr(g["p_action"], m.last_p_action)
    nx, nu = costs.ENV_DIMS[env]
    K, T, B = 11, 38, 4  # 418 windows (ragged last tile)... plus a second shape below
    gen = torch.Generator().manual_seed(3)
    hist = ((torch.rand(K, B - 1 + T, nu, generator=gen) * 2 - 1) * costs.ENV_ACT_HIGH[env]).cuda().contiguous()
    h = m.set_prediction_time(DT)
    outs = {}
    for name in ("fp32", mode):
        p = torch.full((K, T, 2), float("nan"), device="cuda")
        L.check(lib.nlc_encode_history(h, hist.data_ptr(), K, T, B, p.data_ptr(), L.MATH_MODES[name], L.current_stream_ptr()))
        torch.cuda.synchronize()
        outs[name] = p
    assert torch.isfinite(outs[mode]).all()
    assert relerr(outs["fp32"], outs[mode]) < tol, relerr(outs["fp32"], outs[mode])


@pytest.mark.parametrize("env,B", [("oderl-pendulum", 2), ("oderl-pendulum", 3), ("oderl-pendulum", 8), ("oderl-cartpole", 5),
                                   ("oderl-acrobot", 2), ("oderl-acrobot", 3), ("oderl-acrobot", 4)])
@pytest.mark.parametrize("K,T", [(1, 1), (3, 7), (130, 1), (77, 40), (700, 13)])
def test_tc_encoder_window_lengths_and_ragged_tiles(env, B, K, T):
    """The tensor-core encoder's cell pipeline depends on the window length B (2 <= B, B * nu <= 8) and on how the K*T windows
    fall into 128-window tiles (single partial tile, exactly one tile + 2, many tiles per CTA, one window): same output as
    the fp32 CUDA-core encoder for every combination."""
    from oracle import costs
    from test_gpu_parity import make_model

    L = _lib()
    lib = L.load()
    nx, nu = costs.ENV_DIMS[env]
    m = make_model(env, calibrated=False, math_mode="tc_split3")
    h = m.set_prediction_time(DT)
    gen = torch.Generator().manual_seed(1000 * B + K + T)
    hist = ((torch.rand(K, B - 1 + T, nu, generator=gen) * 2 - 1) * costs.ENV_ACT_HIGH[env]).cuda().contiguous()
    outs = {}
    for name in ("fp32", "tc_split3", "tc_fp16"):
        p = torch.full((K, T, 2), float("nan"), device="cuda")
        L.check(lib.nlc_encode_history(h, hist.data_ptr(), K, T, B, p.data_ptr(), L.MATH_MODES[name], L.current_stream_ptr()))
        torch.cuda.synchronize()
        assert torch.isfinite(p).all(), name
        outs[name] = p
    assert relerr(outs["fp32"], outs["tc_split3"]) < 2e-5, relerr(outs["fp32"], outs["tc_split3"])
    assert relerr(outs["fp32"], outs["tc_fp16"]) < 5e-3, relerr(outs["fp32"], outs["tc_fp16"])


@pytest.mark.parametrize("tiles", ["1", "3"])
@pytest.mark.parametrize("mode,tol", [("tc_split3", 1e-4), ("tc_fp16", 2e-2)])
def test_tc_plan_cfg1(mode, tol, tiles, monkeypatch):
    """BASELINE config 1 end to end with the tensor-core encoder and either form of the tensor-core rollout.  tc_split3
    holds the fp32 bound (1e-4); the single-pass fp16 mode is the stated looser bound."""
    monkeypatch.setenv("NLC_ROLLOUT_TILES", tiles)
    from oracle.gen_golden import START_STATE, injected_noise
    from test_gpu_parity import _run_plan
    from _util import action_relerr, load

    env = "oderl-pendulum"
    g = load("plan_cfg1_pendulum_K1000_H20")
    K, T, nu = 1000, 20, 1
    gg = {"in_U": np.zeros((T, nu)), "in_buffer": np.zeros((4, nu)), "in_state": np.array(START_STATE[env]),
          "in_noise": injected_noise(K, T, nu, seed=int(g["noise_seed"])).numpy()}
    planner, out = _run_plan(env, gg, calibrated=True, math_mode=mode)
    assert relerr(g["cost_total"], out["cost_total"]) < tol
    assert relerr(g["states_last"], out["states"][:, -1]) < tol
    assert relerr(g["U"], out["U"]) < tol * (1 if mode == "tc_split3" else 5)
    assert action_relerr(g["action"], out["action"], g["U"], 2.0) < tol * (1 if mode == "tc_split3" else 5)


@pytest.mark.parametrize("env,K,T", [("oderl-acrobot", 20011, 6), ("oderl-cartpole", 19000, 5), ("oderl-pendulum", 40000, 4)])
def test_rollout_forms_agree_beyond_one_wave(env, K, T, monkeypatch):
    """Plans larger than one wave of 128-sample tiles take the ping-pong rollout (two tiles per CTA; partially filled and
    ragged last tiles, K not a multiple of 32): same costs and states as the one-tile form (which then walks several tiles
    per CTA) and the fp32 anchor kernel."""
    import ctypes as C

    from oracle import costs
    from test_gpu_parity import make_model

    L = _lib()
    lib = L.load()
    nx, nu = costs.ENV_DIMS[env]
    m = make_model(env, calibrated=True, math_mode="tc_split3")
    h = m.set_prediction_time(DT)
    B = 4
    gen = torch.Generator().manual_seed(K)
    hist = ((torch.rand(K, B - 1 + T, nu, generator=gen) * 2 - 1) * costs.ENV_ACT_HIGH[env]).cuda().contiguous()
    state = (torch.tensor(costs_start(env), dtype=torch.float32) + 0.05 * torch.randn(K, nx, generator=gen)).cuda().contiguous()
    p = torch.empty(K, T, 2, device="cuda")
    L.check(lib.nlc_encode_history(h, hist.data_ptr(), K, T, B, p.data_ptr(), L.MATH_MODES["tc_split3"], L.current_stream_ptr()))
    ro = L.RolloutOpts()
    ro.env, ro.state_constraint, ro.goal_x, ro.dynamics, ro.delay, ro.dt = L.ENV_IDS[env], 0, 0.0, 0, 0, DT
    outs = {}
    for name, mode, tiles in (("fp32", "fp32", "1"), ("one_tile", "tc_split3", "1"), ("ping_pong", "tc_split3", "3"), ("auto", "tc_split3", "")):
        if tiles:
            monkeypatch.setenv("NLC_ROLLOUT_TILES", tiles)
        else:
            monkeypatch.delenv("NLC_ROLLOUT_TILES", raising=False)
        cost = torch.full((K,), float("nan"), device="cuda")
        states = torch.full((K, T, nx), float("nan"), device="cuda")
        L.check(lib.nlc_rollout_cost(h, C.byref(ro), state.data_ptr(), 1, p.data_ptr(), hist.data_ptr(), None, K, T, B, nu,
                                     cost.data_ptr(), states.data_ptr(), L.MATH_MODES[mode], L.current_stream_ptr()))
        torch.cuda.synchronize()
        assert torch.isfinite(cost).all() and torch.isfinite(states).all(), name
        outs[name] = (cost, states)
    assert torch.equal(outs["auto"][0], outs["ping_pong"][0])  # the library picks the ping-pong form for this size
    for name in ("one_tile", "ping_pong"):
        assert relerr(outs["fp32"][0], outs[name][0]) < 1e-4, (name, relerr(outs["fp32"][0], outs[name][0]))
        assert relerr(outs["fp32"][1], outs[name][1]) < 1e-4, (name, relerr(outs["fp32"][1], outs[name][1]))


@pytest.mark.parametrize("env,S", [("oderl-pendulum", 17), ("oderl-pendulum", 33), ("oderl-cartpole", 33), ("oderl-acrobot", 33)])
@pytest.mark.parametrize("K,T", [(1, 1), (33, 3), (300, 9), (20000, 4)])
def test_rollout_s_terms_and_tiny_plans(env, S, K, T, monkeypatch):
    """Randomly initialised models with 17 and 33 Fourier terms (33 is the reference class default, w_nl.py:73), plans down to
    a single sample and a single step and up to more than one wave of tiles: every tensor-core rollout form against the fp32
    CUDA-core kernel.  Pendulum S = 33 (198 (theta, phi) columns, 224 in the group-uniform order) takes the one-tile or the
    ping-pong form with W3 resident; cartpole / acrobot S = 33 have 330 / 396 columns - more than the ping-pong form's
    accumulators hold and a W3 image beyond shared memory - and always take the one-tile form with L3 in two halves and W3
    streamed by TMA (whatever form is asked for)."""
    import ctypes as C

    import neurallaplacecontrol_b200 as nlc
    from oracle import costs

    L = _lib()
    lib = L.load()
    (nx, nu), B = costs.ENV_DIMS[env], 4
    if K == 20000 and not (S == 33 and nx > 3):
        pytest.skip("large plans of the resident-W3 shapes are covered by test_rollout_forms_agree_beyond_one_wave")
    torch.manual_seed(S)
    m = nlc.NeuralLaplaceModel(nx, nu, nx, hidden_units=128, s_recon_terms=S, state_mean=np.zeros(nx), state_std=np.ones(nx),
                               action_mean=np.array([0.0] * nu), action_std=np.array([1.0]), normalize=True, normalize_time=True, dt=DT,
                               device="cuda:0").double()
    with torch.no_grad():  # keep the Fourier sum in the operating range of a trained model (cf. oracle/gen_golden.py calibrate_)
        last = m.laplace_rep_func.linear_tanh_stack[4]
        last.weight.mul_(0.05)
        last.bias.mul_(0.05)
        last.bias[nx * S:].sub_(3.0)
    h = m.set_prediction_time(DT)
    gen = torch.Generator().manual_seed(K * 100 + T)
    hist = ((torch.rand(K, B - 1 + T, nu, generator=gen) * 2 - 1) * 2.0).cuda().contiguous()
    state = (torch.tensor(costs_start(env)) + 0.05 * torch.randn(K, nx, generator=gen)).cuda().contiguous()
    p = torch.empty(K, T, 2, device="cuda")
    L.check(lib.nlc_encode_history(h, hist.data_ptr(), K, T, B, p.data_ptr(), L.MATH_MODES["fp32"], L.current_stream_ptr()))
    ro = L.RolloutOpts()
    ro.env, ro.state_constraint, ro.goal_x, ro.dynamics, ro.delay, ro.dt = L.ENV_IDS[env], 0, 0.0, 0, 0, DT
    outs = {}
    for name, mode, tiles in (("fp32", "fp32", "1"), ("one_tile", "tc_split3", "1"), ("ping_pong", "tc_split3", "3")):
        monkeypatch.setenv("NLC_ROLLOUT_TILES", tiles)
        cost = torch.full((K,), float("nan"), device="cuda")
        states = torch.full((K, T, nx), float("nan"), device="cuda")
        L.check(lib.nlc_rollout_cost(h, C.byref(ro), state.data_ptr(), 1, p.data_ptr(), hist.data_ptr(), None, K, T, B, nu,
                                     cost.data_ptr(), states.data_ptr(), L.MATH_MODES[mode], L.current_stream_ptr()))
        torch.cuda.synchronize()
        assert torch.isfinite(cost).all() and torch.isfinite(states).all(), name
        outs[name] = (cost, states)
    for name in ("one_tile", "ping_pong"):
        assert relerr(outs["fp32"][0], outs[name][0]) < 1e-4, (name, relerr(outs["fp32"][0], outs[name][0]))
        assert relerr(outs["fp32"][1], outs[name][1]) < 1e-4, (name, relerr(outs["fp32"][1], outs[name][1]))


def costs_start(env):
    return {"oderl-pendulum": [-1.0, 0.0, 1.0], "oderl-cartpole": [0.0, 0.0, -1.0, 0.0, 0.0], "oderl-acrobot": [1.0, 0.0, 1.0, 0.0, 0.0, 0.0]}[env]


@pytest.mark.parametrize("N,Kdim,rows_b", [(64, 64, 64), (128, 128, 128), (208, 128, 208), (176, 128, 176), (112, 128, 112)])
@pytest.mark.parametrize("split3", [0, 1])
def test_umma_selftest_gemm_a_in_tmem(N, Kdim, rows_b, split3):
    """A operand staged in tensor memory by tcgen05.st (operand path of the fused rollout kernel)."""
    L = _lib()
    lib = L.load()
    g = torch.Generator().manual_seed(N + Kdim + split3)
    A = (torch.rand(128, Kdim, generator=g, dtype=torch.float64) * 2 - 1)
    Bm = (torch.randn(rows_b, Kdim, generator=g, dtype=torch.float64) * 0.3)
    D = torch.full((128, N), float("nan"), device="cuda")
    Ad, Bd = A.float().cuda().contiguous(), Bm.float().cuda().contiguous()
    L.check(lib.nlc_selftest_umma_gemm_ts(Ad.data_ptr(), Bd.data_ptr(), rows_b, N, Kdim, split3, D.data_ptr(), L.current_stream_ptr()))
    torch.cuda.synchronize()
    ref = A.float().double() @ Bm.float().double()[:N].T
    err = relerr(ref, D)
    assert err < (2e-6 if split3 else 2e-3), err

"""``NeuralLaplaceModel.forward`` with several prediction times per sample, ``ts_pred`` (K, n_t)
(``nlc_model_forward_multi`` / ``nlc_model_backward_multi``), against fp64 ``nl_forward`` and its autograd, and against the
per-sample-time path ``nlc_model_forward_ts`` column by column.

Other test modules switch grad mode off process-wide at import; the gradient tests here run under ``torch.enable_grad()``.

Bounds, as in tests/test_gpu_grad.py: 1e-4 of each tensor's magnitude (``_util.relerr``) for the calibrated weight family;
for the raw family max(1e-4, 10x the fp32 floor), the floor measured in each case as the worst relative error of the oracle
itself run in fp32 against fp64."""
import numpy as np
import pytest
import torch

from _util import DT, relerr, weights
from oracle.nl_model import nl_forward

pytestmark = pytest.mark.gpu

ENV_SHAPE = {"oderl-pendulum": (3, 1), "oderl-cartpole": (5, 1), "oderl-acrobot": (6, 2)}
MODES = ("fp32", "tc_split3", "tc_fp16")
TOL = 1e-4


def _nlc():
    import neurallaplacecontrol_b200 as nlc

    return nlc


def _state_dict(env, H=128, S=17, calibrated=True, eot=False):
    nx, nu = ENV_SHAPE[env]
    if H == 128 and S == 17 and not eot:
        sd = dict(weights(env, calibrated=calibrated))
    else:
        torch.manual_seed(2000 + H + S + nx)
        m = _nlc().NeuralLaplaceModel(nx, nu, nx, hidden_units=H, s_recon_terms=S, encode_obs_time=eot).double()
        sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
        if calibrated:
            sd["laplace_rep_func.linear_tanh_stack.4.bias"][nx * S:] += -4.0
    sd["state_mean"] = torch.linspace(-0.2, 0.3, nx, dtype=torch.float64)
    sd["state_std"] = torch.linspace(0.7, 1.6, nx, dtype=torch.float64)
    sd["action_mean"] = torch.full((nu,), 0.1, dtype=torch.float64)
    sd["action_std"] = torch.tensor([1.3], dtype=torch.float64)
    sd["dt"] = torch.tensor(DT, dtype=torch.float32).double()
    return sd


def _model(env, sd, H=128, S=17, eot=False, normalize=True, math_mode="fp32"):
    nx, nu = ENV_SHAPE[env]
    m = _nlc().NeuralLaplaceModel(nx, nu, nx, hidden_units=H, s_recon_terms=S, encode_obs_time=eot, state_mean=np.zeros(nx),
                                  state_std=np.ones(nx), action_mean=np.zeros(nu), action_std=np.ones(1), normalize=normalize,
                                  normalize_time=True, dt=DT, device="cuda:0", math_mode=math_mode).double()
    m.load_state_dict(sd)
    return m


def _inputs(env, K, n_t, B=4, seed=0, eot=False, grid="irregular"):
    """obs, act and (K, n_t) times: per-sample cumulative exponential increments, shuffled within each row ("irregular"),
    or one such grid repeated on every row ("repeated")."""
    nx, nu = ENV_SHAPE[env]
    g = torch.Generator().manual_seed(seed)
    obs = torch.randn(K, nx, generator=g, dtype=torch.float64)
    act = 2.0 * torch.randn(K, B, nu, generator=g, dtype=torch.float64)
    if eot:
        act = torch.cat((act, torch.arange(B - 1, -1, -1, dtype=torch.float64).view(1, B, 1).expand(K, B, 1)), dim=2)
    rows = K if grid == "irregular" else 1
    ts = DT * torch.cumsum(0.2 + torch.empty(rows, n_t, dtype=torch.float64).exponential_(1.0, generator=g), dim=1)
    if grid == "irregular":
        ts = torch.gather(ts, 1, torch.argsort(torch.rand(K, n_t, generator=g), dim=1))
    return obs, act, ts.expand(K, n_t).contiguous()


def _oracle(sd, obs, act, ts, dtype, normalize=True):
    d = {k: v.to(device="cuda", dtype=dtype) for k, v in sd.items()}
    with torch.no_grad():
        return nl_forward(d, obs.to("cuda", dtype), act.to("cuda", dtype), ts.to("cuda", dtype), normalize=normalize).double().cpu()


# ---- forward ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [1, 33, 1000, 20011])
@pytest.mark.parametrize("n_t", [2, 7, 64])
@pytest.mark.parametrize("env", list(ENV_SHAPE))
def test_forward_matches_fp64_oracle(env, n_t, K):
    """K = 20011 with n_t = 7 and 64 walks 3 and 20 chunks of 65536 rows; with n_t = 7 samples straddle chunk boundaries."""
    grids = ("irregular", "repeated") if K in (33, 1000) else ("irregular",)
    for calibrated in (True, False):
        sd = _state_dict(env, calibrated=calibrated)
        for grid in grids:
            obs, act, ts = _inputs(env, K, n_t, seed=K + n_t, grid=grid)
            ref = _oracle(sd, obs, act, ts, torch.float64)
            bound = TOL if calibrated else max(TOL, 10.0 * relerr(ref, _oracle(sd, obs, act, ts, torch.float32)))
            for mode in MODES:
                m = _model(env, sd, math_mode=mode)
                with torch.no_grad():
                    out = m(obs.cuda(), act.cuda(), ts.cuda())
                assert out.shape == ref.shape and out.dtype == torch.float64
                assert m.last_p_action.shape == (K, 2)
                e = relerr(ref, out)
                assert e < bound, (env, K, n_t, calibrated, grid, mode, e, bound)


def _forward_ts(m, obs, act, ts_col):
    lib = _nlc()._lib.load()
    K, B = act.shape[0], act.shape[1]
    out = torch.empty(K, obs.shape[1], dtype=torch.float32, device="cuda")
    scratch = torch.empty(K, 4 + m.hidden_units, dtype=torch.float32, device="cuda")
    _nlc()._lib.check(lib.nlc_model_forward_ts(m.handle(), obs.data_ptr(), act.data_ptr(), ts_col.data_ptr(), K, B, out.data_ptr(),
                                               scratch.data_ptr(), _nlc()._lib.MATH_MODES[m.math_mode], _nlc()._lib.current_stream_ptr()))
    return out


def _forward_multi(m, obs, act, ts):
    lib = _nlc()._lib.load()
    K, B, n_t = act.shape[0], act.shape[1], ts.shape[1]
    out = torch.empty(K, n_t, obs.shape[1], dtype=torch.float32, device="cuda")
    ws = torch.empty(int(lib.nlc_model_forward_multi_workspace_bytes(m.handle(), K, n_t, B)), dtype=torch.uint8, device="cuda")
    _nlc()._lib.check(lib.nlc_model_forward_multi(m.handle(), obs.data_ptr(), act.data_ptr(), ts.data_ptr(), K, n_t, B, out.data_ptr(),
                                                  None, ws.data_ptr(), _nlc()._lib.MATH_MODES[m.math_mode], _nlc()._lib.current_stream_ptr()))
    return out


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("env", list(ENV_SHAPE))
def test_columns_bit_identical_to_per_sample_time_path(env, mode):
    """Column j of the (K, n_t) forward is nlc_model_forward_ts on ts[:, j] bit for bit, and n_t = 1 through the new entry
    point likewise: every row is evaluated by the same kernels on the same per-row data."""
    m = _model(env, _state_dict(env), math_mode=mode)
    for K, n_t in ((33, 7), (1000, 7), (20011, 7), (300, 64)):
        obs, act, ts = _inputs(env, K, n_t, seed=3 * K + n_t)
        obs, act, ts = (x.to("cuda", torch.float32).contiguous() for x in (obs, act, ts))
        multi = _forward_multi(m, obs, act, ts)
        for j in range(n_t):
            col = _forward_ts(m, obs, act, ts[:, j].contiguous())
            assert torch.equal(multi[:, j], col), (env, mode, K, n_t, j)
        one = _forward_multi(m, obs, act, ts[:, :1].contiguous())
        assert torch.equal(one[:, 0], _forward_ts(m, obs, act, ts[:, 0].contiguous())), (env, mode, K)


# ---- backward --------------------------------------------------------------------------------------------------------
def _oracle_grads(sd, obs, act, ts, gout, normalize, dtype, need_inputs=True):
    names = [k for k in sd if k.startswith(("action_encoder", "laplace_rep_func"))]
    d = {k: v.detach().to(device="cuda", dtype=dtype).clone() for k, v in sd.items()}
    ps = [d[n].requires_grad_(True) for n in names]
    o = obs.detach().to("cuda", dtype).clone().requires_grad_(need_inputs)
    a = act.detach().to("cuda", dtype).clone().requires_grad_(need_inputs)
    with torch.enable_grad():
        out = nl_forward(d, o, a, ts.to("cuda", dtype), normalize=normalize, normalize_time=True)
        leaves = ([o, a] if need_inputs else []) + ps
        gr = torch.autograd.grad(out, leaves, gout.to("cuda", dtype).view(out.shape))
    keys = (["obs", "act"] if need_inputs else []) + names
    return {k: v.detach().double().cpu() for k, v in zip(keys, gr)}


def _our_grads(m, obs, act, ts, gout, need_inputs=True):
    o = obs.detach().cuda().requires_grad_(need_inputs)
    a = act.detach().cuda().requires_grad_(need_inputs)
    m.zero_grad(set_to_none=True)
    with torch.enable_grad():
        out = m(o, a, ts.cuda())
        assert out.grad_fn is not None
        (out * gout.cuda().view(out.shape)).sum().backward()
    res = {"obs": o.grad, "act": a.grad} if need_inputs else {}
    if not need_inputs:
        assert o.grad is None and a.grad is None
    res.update({n: p.grad for n, p in m.named_parameters()})
    for n, p in m.named_parameters():
        assert res[n].dtype == p.dtype and res[n].device == p.device, n
    return res


def _check_grads(env, K, n_t, calibrated=True, H=128, S=17, B=4, eot=False, normalize=True, need_inputs=True, two_d_act=False):
    sd = _state_dict(env, H, S, calibrated, eot)
    m = _model(env, sd, H, S, eot, normalize)
    obs, act, ts = _inputs(env, K, n_t, B, seed=K + 5 * n_t, eot=eot)
    if two_d_act:
        act = act[:, 0]
    gout = torch.randn(K, n_t, ENV_SHAPE[env][0], generator=torch.Generator().manual_seed(K + n_t), dtype=torch.float64)
    ours = _our_grads(m, obs, act, ts, gout, need_inputs)
    ref = _oracle_grads(sd, obs, act, ts, gout, normalize, torch.float64, need_inputs)
    bound = TOL
    if not calibrated:
        r32 = _oracle_grads(sd, obs, act, ts, gout, normalize, torch.float32, need_inputs)
        bound = max(TOL, 10.0 * max(relerr(ref[k], r32[k]) for k in ref))
    errs = {k: relerr(ref[k], ours[k]) for k in ref}
    worst = max(errs, key=errs.get)
    print(f"multi grad {env} K={K} n_t={n_t} cal={calibrated} H={H} B={B} eot={eot} norm={normalize}: {errs[worst]:.2e} ({worst})")
    assert errs[worst] < bound, (env, K, n_t, calibrated, worst, errs[worst], bound)


@pytest.mark.parametrize("K,n_t", [(1, 2), (33, 7), (1000, 7), (300, 64)])
@pytest.mark.parametrize("calibrated", [True, False], ids=["cal", "raw"])
@pytest.mark.parametrize("env", list(ENV_SHAPE))
def test_gradients_match_oracle(env, calibrated, K, n_t):
    _check_grads(env, K, n_t, calibrated)


@pytest.mark.parametrize("variant", ["encode_obs_time", "hidden_64", "no_normalize", "window_8", "actions_2d", "null_input_grads"])
def test_gradients_variants(variant):
    kw = {"encode_obs_time": dict(eot=True), "hidden_64": dict(H=64), "no_normalize": dict(normalize=False), "window_8": dict(B=8),
          "actions_2d": dict(B=1, two_d_act=True), "null_input_grads": dict(need_inputs=False)}[variant]
    for calibrated in (True, False):
        _check_grads("oderl-cartpole", 257, 5, calibrated, **kw)


def test_gradients_across_chunks():
    """K n_t = 140077 rows: three chunks of the MLP/ILT stage, samples straddling both chunk boundaries."""
    _check_grads("oderl-acrobot", 20011, 7)


def test_backward_is_deterministic():
    env = "oderl-acrobot"
    m = _model(env, _state_dict(env, calibrated=False))
    obs, act, ts = _inputs(env, 5000, 7, seed=11)
    gout = torch.randn(5000, 7, 6, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    a = _our_grads(m, obs, act, ts, gout)
    b = _our_grads(m, obs, act, ts, gout)
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_forward_unchanged_with_grad():
    env = "oderl-acrobot"
    m = _model(env, _state_dict(env), math_mode="tc_split3")
    obs, act, ts = (x.cuda() for x in _inputs(env, 700, 9, seed=4))
    with torch.no_grad():
        ref = m(obs, act, ts)
        assert ref.grad_fn is None
    with torch.enable_grad():
        out = m(obs, act, ts)
        assert out.grad_fn is not None
    assert torch.equal(ref, out.detach())


def test_multi_horizon_training():
    """loss.backward() through the module fills every .grad; 150 Adam steps on a loss over three horizons per sample
    (analytic pendulum targets) lower the loss."""
    from oracle.dynamics import analytic_step

    env = "oderl-pendulum"
    m = _model(env, _state_dict(env))
    g = torch.Generator().manual_seed(3)
    s0 = torch.randn(32, 3, generator=g, dtype=torch.float64) * 0.5
    th = torch.rand(32, generator=g, dtype=torch.float64) * 6.28
    s0[:, 0], s0[:, 1] = torch.cos(th), torch.sin(th)
    a0 = torch.randn(32, 4, 1, generator=g, dtype=torch.float64)
    hs = (1, 2, 3)
    ts = torch.tensor([h * DT for h in hs], dtype=torch.float64).expand(32, 3).contiguous()
    target = torch.stack([torch.cat([analytic_step(env, s0[i:i + 1], a0[i:i + 1], h * DT, 1) for i in range(32)]) - s0 for h in hs], 1)
    s0, a0, ts, target = s0.cuda(), a0.cuda(), ts.cuda(), target.cuda()
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    with torch.enable_grad():
        loss = torch.nn.functional.mse_loss(m(s0, a0, ts), target)
        loss.backward()
        assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in m.parameters())
        l0 = float(loss.detach())
        for _ in range(150):
            opt.zero_grad()
            loss = torch.nn.functional.mse_loss(m(s0, a0, ts), target)
            loss.backward()
            opt.step()
    with torch.no_grad():
        l1 = float(torch.nn.functional.mse_loss(m(s0, a0, ts), target))
    print(f"multi-horizon Adam: loss {l0:.4e} -> {l1:.4e}")
    assert l1 < 0.5 * l0, (l0, l1)


# ---- rejections and launch counts ------------------------------------------------------------------------------------
def test_rejections():
    env = "oderl-pendulum"
    m = _model(env, _state_dict(env))
    obs, act, ts = (x.cuda() for x in _inputs(env, 8, 5))
    with pytest.raises(ValueError):
        m(obs, act, ts[:1])  # (1, n_t) with K = 8
    with torch.enable_grad(), pytest.raises(NotImplementedError):
        m(obs, act, ts.clone().requires_grad_(True))
    lib = _nlc()._lib.load()
    h = m.handle()
    buf = torch.zeros(1 << 16, dtype=torch.float32, device="cuda")
    p = buf.data_ptr()
    K, n_t = 1 << 16, 1 << 15  # K n_t = 2^31
    assert lib.nlc_model_forward_multi(h, p, p, p, K, n_t, 4, p, p, p, 0, None) == -2  # NLC_ERR_SHAPE
    assert lib.nlc_model_backward_multi(h, p, p, p, K, n_t, 4, p, p, p, p, p, None) == -2
    assert lib.nlc_model_forward_multi_workspace_bytes(h, K, n_t, 4) == -2
    assert lib.nlc_model_backward_multi_workspace_bytes(h, K, n_t, 4) == -2


def test_launch_count_does_not_depend_on_n_t():
    """Below 65536 rows (one chunk) one forward and one backward launch the same number of kernels for every n_t; each
    further chunk of 65536 rows adds its prep and MLP/ILT launches (2 in the forward, 3 in the backward)."""
    env = "oderl-acrobot"
    lib = _nlc()._lib.load()
    counts = {}
    for mode in ("fp32", "tc_split3"):
        m = _model(env, _state_dict(env), math_mode=mode)
        m.handle()  # packing the parameters is not part of a call
        for K, n_t in ((512, 2), (512, 7), (512, 64), (2048, 64)):
            obs, act, ts = (x.cuda() for x in _inputs(env, K, n_t))
            o = obs.clone().requires_grad_(True)
            with torch.enable_grad():
                torch.cuda.synchronize()
                n0 = lib.nlc_launch_count()
                out = m(o, act, ts)
                n1 = lib.nlc_launch_count()
                out.sum().backward()
                torch.cuda.synchronize()
                n2 = lib.nlc_launch_count()
            counts[mode, K, n_t] = (n1 - n0, n2 - n1)
        fwd, bwd = counts[mode, 512, 2]
        assert counts[mode, 512, 7] == counts[mode, 512, 64] == (fwd, bwd), counts
        assert counts[mode, 2048, 64] == (fwd + 2, bwd + 3), counts  # 131072 rows: two chunks

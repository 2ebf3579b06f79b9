"""``NeuralLaplaceModel(..., math_mode="fp64")``: forward and backward in fp64 throughout (``nlc_model_forward_f64`` /
``nlc_model_backward_f64``), against the reference's own fp64 outputs (``tests/golden/model_fwd_*.npz``), fp64 ``nl_forward``
and its autograd, and fp64 training.

Bounds (``_util.relerr``: max |ref - got| / max |ref|, per tensor): 1e-10 for forward outputs, 1e-9 for gradients and for the
parameter change of a training run.  Other test modules switch grad mode off process-wide at import; the gradient tests
here run under ``torch.enable_grad()``."""
import functools

import numpy as np
import pytest
import torch

from _util import DT, load, relerr, short, weights
from oracle.nl_model import nl_forward
from test_gpu_grad import _dataset
from test_gpu_multi_time import ENV_SHAPE, _inputs, _state_dict
from test_gpu_multi_time import _model as _model_mt

pytestmark = pytest.mark.gpu

TOL_FWD = 1e-10
TOL_GRAD = 1e-9
_model = functools.partial(_model_mt, math_mode="fp64")


def _nlc():
    import neurallaplacecontrol_b200 as nlc

    return nlc


def _ts_form(ts, form):
    """ts_pred in one of the reference's forms, and the (K, n_t) times the oracle evaluates it at."""
    K = ts.shape[0]
    if form == "scalar":
        t = ts[0, 0].clone()
        return t, t.expand(K, 1)
    if form == "K":
        return ts[:, 0].clone(), ts[:, :1]
    if form == "K1":
        return ts[:, :1].clone(), ts[:, :1]
    return ts, ts


def _oracle(sd, obs, act, ts, normalize=True):
    d = {k: v.to(device="cuda", dtype=torch.float64) for k, v in sd.items()}
    with torch.no_grad():
        out, p = nl_forward(d, obs.cuda(), act.cuda(), ts.cuda(), normalize=normalize, return_parts=True)
    return out.cpu(), p.cpu()


def _check_forward(env, sd, K, n_t, form, H=128, S=17, B=4, eot=False, normalize=True, two_d_act=False, seed=0):
    m = _model(env, sd, H, S, eot, normalize)
    obs, act, ts = _inputs(env, K, n_t, B, seed=seed, eot=eot)
    if two_d_act:
        act = act[:, 0]
    ts_pred, ts_ref = _ts_form(ts, form)
    ref, p_ref = _oracle(sd, obs, act, ts_ref, normalize)
    with torch.no_grad():
        out = m(obs.cuda(), act.cuda(), ts_pred.cuda())
    assert out.dtype == torch.float64 and out.shape == ref.shape, (out.shape, ref.shape)
    e, ep = relerr(ref, out), relerr(p_ref, m.last_p_action)
    print(f"fp64 fwd {env} K={K} n_t={n_t} {form} H={H} S={S} B={B} eot={eot} norm={normalize}: out {e:.2e} p_action {ep:.2e}")
    assert e < TOL_FWD and ep < TOL_FWD, (env, K, n_t, form, e, ep)


# ---- forward ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("env", list(ENV_SHAPE))
def test_matches_reference_golden_outputs(env):
    """The reference's own ReverseGRUEncoder / LaplaceRepresentationFunc outputs (fp64), at fixed and irregular times."""
    g = load("model_fwd_" + short(env))
    m = _model(env, weights(env))
    obs, act = torch.from_numpy(g["obs"]).cuda(), torch.from_numpy(g["act"]).cuda()
    for key in ("fixed", "irreg"):
        with torch.no_grad():
            out = m(obs, act, torch.from_numpy(g["ts_" + key]).cuda())
        e, ep = relerr(g["out_" + key], out), relerr(g["p_action"], m.last_p_action)
        print(f"golden {env} {key}: out {e:.2e} p_action {ep:.2e}")
        assert e < TOL_FWD and ep < TOL_FWD, (env, key, e, ep)


@pytest.mark.parametrize("K", [1, 33, 1000, 20011])
@pytest.mark.parametrize("form", ["scalar", "K", "K1", "Knt"])
@pytest.mark.parametrize("env", list(ENV_SHAPE))
def test_forward_matches_fp64_oracle(env, form, K):
    """Every ts_pred form; (K, n_t) with n_t = 7 at K = 20011 walks 140077 rows, three chunks of 65536."""
    for calibrated in (True, False):
        _check_forward(env, _state_dict(env, calibrated=calibrated), K, 7 if form == "Knt" else 1, form, seed=K)


@pytest.mark.parametrize("variant", ["encode_obs_time", "hidden_64", "S_33", "no_normalize", "window_1", "window_8", "actions_2d"])
def test_forward_variants(variant):
    kw = {"encode_obs_time": dict(eot=True), "hidden_64": dict(H=64), "S_33": dict(S=33), "no_normalize": dict(normalize=False),
          "window_1": dict(B=1), "window_8": dict(B=8), "actions_2d": dict(B=1, two_d_act=True)}[variant]
    # the oracle broadcasts action_mean over the extra time channel only for one action (nu = 1), as the reference does
    for env in ("oderl-cartpole",) if variant == "encode_obs_time" else ("oderl-cartpole", "oderl-acrobot"):
        for calibrated in (True, False):
            sd = _state_dict(env, kw.get("H", 128), kw.get("S", 17), calibrated, kw.get("eot", False))
            for n_t, form in ((1, "K1"), (7, "Knt")):
                _check_forward(env, sd, 257, n_t, form, seed=11, **kw)


# ---- backward --------------------------------------------------------------------------------------------------------
def _oracle_grads(sd, obs, act, ts, gout, normalize, need_obs=True, need_act=True):
    names = [k for k in sd if k.startswith(("action_encoder", "laplace_rep_func"))]
    d = {k: v.detach().to(device="cuda", dtype=torch.float64).clone() for k, v in sd.items()}
    ps = [d[n].requires_grad_(True) for n in names]
    o = obs.detach().cuda().clone().requires_grad_(need_obs)
    a = act.detach().cuda().clone().requires_grad_(need_act)
    with torch.enable_grad():
        out = nl_forward(d, o, a, ts.cuda(), normalize=normalize)
        leaves = ([o] if need_obs else []) + ([a] if need_act else []) + ps
        gr = torch.autograd.grad(out, leaves, gout.cuda().view(out.shape))
    keys = (["obs"] if need_obs else []) + (["act"] if need_act else []) + names
    return {k: v.detach().cpu() for k, v in zip(keys, gr)}


def _our_grads(m, obs, act, ts, gout, need_obs=True, need_act=True):
    o = obs.detach().cuda().requires_grad_(need_obs)
    a = act.detach().cuda().requires_grad_(need_act)
    m.zero_grad(set_to_none=True)
    with torch.enable_grad():
        out = m(o, a, ts.cuda())
        (out * gout.cuda().view(out.shape)).sum().backward()
    res = {}
    if need_obs:
        res["obs"] = o.grad
    if need_act:
        res["act"] = a.grad
    assert (o.grad is None) != need_obs and (a.grad is None) != need_act
    res.update({n: p.grad for n, p in m.named_parameters()})
    for n, p in m.named_parameters():
        assert res[n].dtype == p.dtype and res[n].device == p.device, n
    return res


def _check_grads(env, K, n_t, calibrated=True, H=128, S=17, B=4, eot=False, normalize=True, need_obs=True, need_act=True):
    sd = _state_dict(env, H, S, calibrated, eot)
    m = _model(env, sd, H, S, eot, normalize)
    obs, act, ts = _inputs(env, K, n_t, B, seed=K + 5 * n_t, eot=eot)
    gout = torch.randn(K, n_t, ENV_SHAPE[env][0], generator=torch.Generator().manual_seed(K + n_t), dtype=torch.float64)
    ours = _our_grads(m, obs, act, ts, gout, need_obs, need_act)
    ref = _oracle_grads(sd, obs, act, ts, gout, normalize, need_obs, need_act)
    assert len(ref) == 16 + need_obs + need_act
    errs = {k: relerr(ref[k], ours[k]) for k in ref}
    worst = max(errs, key=errs.get)
    print(f"fp64 grad {env} K={K} n_t={n_t} cal={calibrated} H={H} B={B} eot={eot}: {errs[worst]:.2e} ({worst})")
    assert errs[worst] < TOL_GRAD, (env, K, n_t, calibrated, worst, errs[worst])


@pytest.mark.parametrize("K,n_t", [(1, 1), (1000, 1), (33, 7), (1000, 7)])
@pytest.mark.parametrize("calibrated", [True, False], ids=["cal", "raw"])
@pytest.mark.parametrize("env", list(ENV_SHAPE))
def test_gradients_match_oracle(env, calibrated, K, n_t):
    _check_grads(env, K, n_t, calibrated)


@pytest.mark.parametrize("variant", ["no_obs_grad", "no_act_grad", "encode_obs_time", "hidden_64", "window_8", "no_normalize"])
def test_gradients_variants(variant):
    kw = {"no_obs_grad": dict(need_obs=False), "no_act_grad": dict(need_act=False), "encode_obs_time": dict(eot=True),
          "hidden_64": dict(H=64), "window_8": dict(B=8), "no_normalize": dict(normalize=False)}[variant]
    for calibrated in (True, False):
        for n_t in (1, 7):
            _check_grads("oderl-cartpole", 257, n_t, calibrated, **kw)


def test_gradients_across_chunks():
    _check_grads("oderl-acrobot", 20011, 7)


def test_forward_and_backward_are_deterministic():
    env = "oderl-acrobot"
    m = _model(env, _state_dict(env, calibrated=False))
    obs, act, ts = _inputs(env, 5000, 7, seed=11)
    gout = torch.randn(5000, 7, 6, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    with torch.no_grad():
        f1, f2 = m(obs.cuda(), act.cuda(), ts.cuda()), m(obs.cuda(), act.cuda(), ts.cuda())
    assert torch.equal(f1, f2)
    a = _our_grads(m, obs, act, ts, gout)
    b = _our_grads(m, obs, act, ts, gout)
    for k in a:
        assert torch.equal(a[k], b[k]), k


# ---- training --------------------------------------------------------------------------------------------------------
def test_training_parity_sgd():
    """20 plain-SGD steps of the reference's loss (train_utils.py:388-407) in fp64 mode beside the oracle's fp64 parameters:
    the parameters' total change agrees within 1e-9 of its magnitude, per tensor."""
    env = "oderl-pendulum"
    sd = _state_dict(env)
    m = _model(env, sd)
    names = [n for n, _ in m.named_parameters()]
    ref = {k: v.clone() for k, v in sd.items()}
    for n in names:
        ref[n].requires_grad_(True)
    opt = torch.optim.SGD(m.parameters(), lr=0.05)
    opt_ref = torch.optim.SGD([ref[n] for n in names], lr=0.05)
    with torch.enable_grad():
        for s0, a0, ts, sn in _dataset(env, 20, 1):
            opt.zero_grad()
            torch.nn.functional.mse_loss(m(s0.cuda(), a0.cuda(), ts.cuda()), (sn - s0).cuda()).backward()
            opt.step()
            opt_ref.zero_grad()
            torch.nn.functional.mse_loss(nl_forward(ref, s0, a0, ts), sn - s0).backward()
            opt_ref.step()
    worst = 0.0
    for n, p in m.named_parameters():
        e = relerr(ref[n].detach() - sd[n], p.detach().cpu() - sd[n])
        worst = max(worst, e)
        assert e < TOL_GRAD, (n, e)
    print(f"fp64 SGD parity: worst relerr of the parameter change {worst:.2e}")


def _plan_costs(model, env="oderl-pendulum", K=256, T=10):
    from _util import START_STATE, injected_noise
    from oracle import costs

    nlc = _nlc()
    nx, nu = ENV_SHAPE[env]
    ah = costs.ENV_ACT_HIGH[env]
    noise = injected_noise(K, T, nu, seed=7)
    planner = nlc.MPPIDelay(nlc.NLDynamics(model, DT), nlc.EnvRunningCost(env), nx, nlc.noise_sigma_for(nu), num_samples=K,
                            horizon=T, device="cuda:0", lambda_=1.0, u_min=torch.tensor(-ah), u_max=torch.tensor(ah), u_scale=ah,
                            U_init=torch.zeros(T, nu, dtype=torch.float64))
    planner.noise_dist.sample = lambda shape: noise
    planner.command(np.array(START_STATE[env]), torch.zeros(4, nu, dtype=torch.float64))
    torch.cuda.synchronize()
    return planner.cost_total.clone()


def test_optimizer_step_needs_no_new_handle_and_planner_sees_new_weights():
    env = "oderl-pendulum"
    sd = _state_dict(env)
    m = _model(env, sd)
    obs, act, ts = _inputs(env, 300, 1, seed=5)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    with torch.enable_grad():
        m(obs.cuda(), act.cuda(), ts.cuda()).square().sum().backward()
    h = m._handle
    assert h is not None
    opt.step()
    with torch.no_grad():
        out = m(obs.cuda(), act.cuda(), ts.cuda())
    assert m._handle is h  # the forward after the step reused the handle
    new_sd = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    ref, _ = _oracle(new_sd, obs, act, ts)
    assert relerr(ref, out) < TOL_FWD
    # a planner on the same model plans with the current weights: the same costs as on a freshly built model
    costs_same = _plan_costs(m)
    costs_fresh = _plan_costs(_model(env, new_sd))
    assert torch.equal(costs_same, costs_fresh)
    # switching the mode on a live model gives what a fresh model in that mode gives
    x = (obs.cuda(), act.cuda(), ts.cuda())
    with torch.no_grad():
        fresh = {mode: _model(env, new_sd, math_mode=mode)(*x) for mode in ("fp64", "tc_split3")}
        for mode in ("fp64", "tc_split3", "fp64"):
            m.math_mode = mode
            assert torch.equal(m(*x), fresh[mode]), mode


# ---- rejections ------------------------------------------------------------------------------------------------------
def test_rejections():
    env = "oderl-pendulum"
    m = _model(env, _state_dict(env))
    obs, act, ts = (x.cuda() for x in _inputs(env, 8, 5))
    with torch.enable_grad(), pytest.raises(NotImplementedError):
        m(obs, act, ts.clone().requires_grad_(True))
    lib = _nlc()._lib.load()
    h = m.handle()
    buf = torch.zeros(1 << 20, dtype=torch.float64, device="cuda")
    p = buf.data_ptr()
    ARG, SHAPE = -1, -2
    assert lib.nlc_model_forward_f64(h, None, p, p, p, 8, 1, 4, p, None, p, None) == ARG  # params
    assert lib.nlc_model_forward_f64(h, p, None, p, p, 8, 1, 4, p, None, p, None) == ARG  # obs
    assert lib.nlc_model_forward_f64(h, p, p, p, p, 8, 1, 4, None, None, p, None) == ARG  # out
    assert lib.nlc_model_backward_f64(h, None, p, p, p, 8, 1, 4, p, p, None, None, p, None) == ARG
    assert lib.nlc_model_backward_f64(h, p, None, p, p, 8, 1, 4, p, p, None, None, p, None) == ARG
    assert lib.nlc_model_backward_f64(h, p, p, p, p, 8, 1, 4, p, None, None, None, p, None) == ARG  # grad_params
    K, n_t = 1 << 16, 1 << 15  # K n_t = 2^31
    assert lib.nlc_model_forward_f64(h, p, p, p, p, K, n_t, 4, p, None, p, None) == SHAPE
    assert lib.nlc_model_backward_f64(h, p, p, p, p, K, n_t, 4, p, p, None, None, p, None) == SHAPE
    assert lib.nlc_model_forward_f64_workspace_bytes(h, K, n_t, 4) == SHAPE
    assert lib.nlc_model_backward_f64_workspace_bytes(h, K, n_t, 4) == SHAPE
    assert lib.nlc_model_forward_f64(h, p, p, p, p, 8, 1, 4, p, None, p + 8, None) == ARG  # unaligned workspace
    assert lib.nlc_model_backward_f64(h, p, p, p, p, 8, 1, 4, p, p, None, None, p + 8, None) == ARG

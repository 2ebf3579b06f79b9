"""Backward of ``NeuralLaplaceModel.forward`` (``nlc_model_backward_ts``, csrc/model_grad.cu) against fp64 autograd of the
oracle forward (``oracle.nl_model.nl_forward``) on the same state_dict.

Other test modules switch grad mode off process-wide at import; every test here runs under ``torch.enable_grad()``.

Bounds: 1e-4 of each tensor's magnitude (``_util.relerr``) for the calibrated weight family, the forward's bound; for the
raw family (random init, whose phi outputs sit in the steep tail of the sphere map) 10x the fp32 floor, measured in each
case as the worst relative error of the oracle's own autograd run in fp32 against fp64, with 1e-4 as the least bound."""
import numpy as np
import pytest
import torch

from _util import DT, relerr, weights
from oracle.nl_model import nl_forward

pytestmark = pytest.mark.gpu

ENV_SHAPE = {"oderl-pendulum": (3, 1), "oderl-cartpole": (5, 1), "oderl-acrobot": (6, 2)}
TOL = 1e-4


def _nlc():
    import neurallaplacecontrol_b200 as nlc

    return nlc


def _state_dict(env, H, S, calibrated, eot=False):
    """Golden weights at (128, 17); the reference's seeded random init elsewhere, with the same phi-bias shift for the
    calibrated family (oracle/gen_golden.py)."""
    nx, nu = ENV_SHAPE[env]
    if H == 128 and S == 17 and not eot:
        sd = weights(env, calibrated=calibrated)
    else:
        torch.manual_seed(1000 + H + S + nx)
        m = _nlc().NeuralLaplaceModel(nx, nu, nx, hidden_units=H, s_recon_terms=S, encode_obs_time=eot).double()
        sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
        if calibrated:
            sd["laplace_rep_func.linear_tanh_stack.4.bias"][nx * S:] += -4.0
    sd = dict(sd)
    sd["state_mean"] = torch.linspace(-0.2, 0.3, nx, dtype=torch.float64)  # non-trivial normalisation
    sd["state_std"] = torch.linspace(0.7, 1.6, nx, dtype=torch.float64)
    sd["action_mean"] = torch.full((nu,), 0.1, dtype=torch.float64)
    sd["action_std"] = torch.tensor([1.3], dtype=torch.float64)
    sd["dt"] = torch.tensor(DT, dtype=torch.float32).double()
    return sd


def _model(env, H, S, sd, eot=False, normalize=True, math_mode="fp32"):
    nx, nu = ENV_SHAPE[env]
    m = _nlc().NeuralLaplaceModel(nx, nu, nx, hidden_units=H, s_recon_terms=S, encode_obs_time=eot, state_mean=np.zeros(nx),
                                  state_std=np.ones(nx), action_mean=np.zeros(nu), action_std=np.ones(1), normalize=normalize,
                                  normalize_time=True, dt=DT, device="cuda:0", math_mode=math_mode).double()
    m.load_state_dict(sd)
    return m


def _inputs(env, K, B, seed, eot=False, uniform_ts=False):
    nx, nu = ENV_SHAPE[env]
    g = torch.Generator().manual_seed(seed)
    obs = torch.randn(K, nx, generator=g, dtype=torch.float64)
    act = 2.0 * torch.randn(K, B, nu, generator=g, dtype=torch.float64)
    if eot:  # the caller-supplied time channel B-1 .. 0 (mppi_with_model.py:110-119)
        act = torch.cat((act, torch.arange(B - 1, -1, -1, dtype=torch.float64).view(1, B, 1).expand(K, B, 1)), dim=2)
    if uniform_ts:
        ts = torch.full((K, 1), 1.7 * DT, dtype=torch.float64)
    else:  # exponentially distributed per-sample prediction times, bounded away from 0
        ts = DT * (0.2 + torch.empty(K, 1, dtype=torch.float64).exponential_(1.0, generator=g))
    return obs, act, ts


def _oracle_grads(sd, obs, act, ts, gout, normalize, dtype, device="cpu"):
    names = [k for k in sd if k.startswith(("action_encoder", "laplace_rep_func"))]
    d = {k: v.detach().to(device=device, dtype=dtype).clone() for k, v in sd.items()}  # leaves of its own: sd stays as it is
    ps = [d[n].requires_grad_(True) for n in names]
    o = obs.detach().to(device=device, dtype=dtype).clone().requires_grad_(True)
    a = act.detach().to(device=device, dtype=dtype).clone().requires_grad_(True)
    with torch.enable_grad():
        out = torch.atleast_2d(nl_forward(d, o, a, ts.to(device=device, dtype=dtype), normalize=normalize, normalize_time=True))
        gr = torch.autograd.grad(out, [o, a] + ps, gout.to(device=device, dtype=dtype).view(out.shape))
    res = {"obs": gr[0], "act": gr[1]}
    res.update(zip(names, gr[2:]))
    return {k: v.detach().cpu().double() for k, v in res.items()}, out.detach()


def _our_grads(m, obs, act, ts, loss_fn):
    o = obs.detach().cuda().requires_grad_(True)
    a = act.detach().cuda().requires_grad_(True)
    m.zero_grad(set_to_none=True)
    with torch.enable_grad():
        out = m(o, a, ts.cuda())
        loss_fn(out).backward()
    res = {"obs": o.grad, "act": a.grad}
    res.update({n: p.grad for n, p in m.named_parameters()})
    return res, out.detach()


def _check_case(env, H, S, calibrated, K, B=4, eot=False, normalize=True, uniform_ts=False, seed=0):
    sd = _state_dict(env, H, S, calibrated, eot)
    m = _model(env, H, S, sd, eot, normalize)
    obs, act, ts = _inputs(env, K, B, seed, eot, uniform_ts)
    nx = ENV_SHAPE[env][0]
    if B == 1:
        act = act[:, 0]
    g = torch.Generator().manual_seed(seed + 7)
    target = torch.randn(K, nx, generator=g, dtype=torch.float64)
    gout_rand = torch.randn(K, nx, generator=g, dtype=torch.float64)
    worst = {}
    for kind in ("mse", "vjp"):
        if kind == "mse":
            ours, out = _our_grads(m, obs, act, ts, lambda y: torch.nn.functional.mse_loss(torch.atleast_2d(y), target.cuda().view(-1, nx)))
            gout = 2.0 * (out.double().cpu().view(-1, nx) - target) / (K * nx)
        else:
            ours, _ = _our_grads(m, obs, act, ts, lambda y: (torch.atleast_2d(y) * gout_rand.cuda().view(-1, nx)).sum())
            gout = gout_rand
        # the oracle's gradient at the same output gradient (for MSE: at our fp32 output, which the loss saw)
        ref, _ = _oracle_grads(sd, obs, act, ts, gout, normalize, torch.float64)
        bound = TOL
        if not calibrated:
            r32, _ = _oracle_grads(sd, obs, act, ts, gout, normalize, torch.float32)
            floor = max(relerr(ref[k], r32[k]) for k in ref)
            bound = max(TOL, 10.0 * floor)
        for k in ref:
            e = relerr(ref[k], ours[k])
            worst[k] = max(worst.get(k, 0.0), e)
            assert e < bound, (env, H, S, calibrated, K, kind, k, e, bound)
        for n, p in m.named_parameters():
            assert ours[n].dtype == p.dtype and ours[n].device == p.device
    print(f"grad {env} H={H} S={S} {'cal' if calibrated else 'raw'} K={K} B={B} eot={eot} norm={normalize} uniform={uniform_ts}: "
          f"worst relerr {max(worst.values()):.2e} ({max(worst, key=worst.get)}) bound {bound:.1e}")
    return worst


@pytest.mark.parametrize("K", [16, 512, 1])
@pytest.mark.parametrize("calibrated", [True, False], ids=["cal", "raw"])
@pytest.mark.parametrize("H,S", [(128, 17), (128, 33), (64, 17)])
@pytest.mark.parametrize("env", list(ENV_SHAPE))
def test_gradients_match_oracle(env, H, S, calibrated, K):
    _check_case(env, H, S, calibrated, K)


@pytest.mark.parametrize("variant", ["encode_obs_time", "no_normalize", "window_1", "uniform_ts"])
def test_gradients_variants(variant):
    kw = {"encode_obs_time": dict(eot=True), "no_normalize": dict(normalize=False), "window_1": dict(B=1),
          "uniform_ts": dict(uniform_ts=True)}[variant]
    for calibrated in (True, False):
        _check_case("oderl-cartpole", 128, 17, calibrated, 512, **kw)


def test_large_ragged_case_fp64_oracle_on_gpu():
    """K = 20011: 626 tiles of 32 samples over 148 CTAs (every CTA reduces 4-5 tiles), the last tile holds 11 samples."""
    env, K = "oderl-acrobot", 20011
    sd = _state_dict(env, 128, 17, True)
    m = _model(env, 128, 17, sd)
    obs, act, ts = _inputs(env, K, 4, 3)
    gout = torch.randn(K, 6, generator=torch.Generator().manual_seed(5), dtype=torch.float64)
    ours, _ = _our_grads(m, obs, act, ts, lambda y: (y * gout.cuda()).sum())
    ref, _ = _oracle_grads(sd, obs, act, ts, gout, True, torch.float64, device="cuda")
    errs = {k: relerr(ref[k], ours[k]) for k in ref}
    print("large case worst relerr", max(errs.values()), max(errs, key=errs.get))
    assert max(errs.values()) < TOL, errs


def test_backward_is_deterministic():
    env, K = "oderl-acrobot", 5000
    m = _model(env, 128, 17, _state_dict(env, 128, 17, False))
    obs, act, ts = _inputs(env, K, 4, 11)
    gout = torch.randn(K, 6, generator=torch.Generator().manual_seed(2), dtype=torch.float64).cuda()
    a, _ = _our_grads(m, obs, act, ts, lambda y: (y * gout).sum())
    b, _ = _our_grads(m, obs, act, ts, lambda y: (y * gout).sum())
    for k in a:
        assert torch.equal(a[k], b[k]), k


@pytest.mark.parametrize("math_mode", ["fp32", "tc_split3"])
@pytest.mark.parametrize("uniform", [False, True])
def test_forward_unchanged_with_grad(math_mode, uniform):
    env = "oderl-acrobot"
    m = _model(env, 128, 17, _state_dict(env, 128, 17, True), math_mode=math_mode)
    obs, act, ts = _inputs(env, 700, 4, 4, uniform_ts=uniform)
    obs, act, ts = obs.cuda(), act.cuda(), ts.cuda()
    with torch.no_grad():
        ref = m(obs, act, ts)
        assert ref.grad_fn is None
    with torch.enable_grad():
        out = m(obs, act, ts)
        assert out.grad_fn is not None
    assert torch.equal(ref, out.detach())


def test_ts_requires_grad_raises():
    env = "oderl-pendulum"
    m = _model(env, 128, 17, _state_dict(env, 128, 17, True))
    obs, act, ts = _inputs(env, 8, 4, 0)
    with torch.enable_grad(), pytest.raises(NotImplementedError):
        m(obs.cuda(), act.cuda(), ts.cuda().requires_grad_(True))


def test_backward_after_planner_folded_another_time():
    """The backward reads only the unfolded weights: a prediction time folded into the same handle in between (as a
    planner does) changes nothing."""
    env = "oderl-cartpole"
    sd = _state_dict(env, 128, 17, True)
    m = _model(env, 128, 17, sd)
    obs, act, ts = _inputs(env, 300, 4, 9)
    gout = torch.randn(300, 5, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    o, a = obs.cuda().requires_grad_(True), act.cuda().requires_grad_(True)
    with torch.enable_grad():
        out = m(o, a, ts.cuda())
        m.set_prediction_time(0.37)
        (out * gout.cuda()).sum().backward()
    ref, _ = _oracle_grads(sd, obs, act, ts, gout, True, torch.float64)
    ours = {"obs": o.grad, "act": a.grad}
    ours.update({n: p.grad for n, p in m.named_parameters()})
    for k in ref:
        assert relerr(ref[k], ours[k]) < TOL, k


def _dataset(env, n_batches, seed):
    from oracle.dynamics import analytic_step

    nx, nu = ENV_SHAPE[env]
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n_batches):
        s0 = torch.randn(16, nx, generator=g, dtype=torch.float64) * 0.5
        if env == "oderl-pendulum":
            th = torch.rand(16, generator=g, dtype=torch.float64) * 6.28
            s0[:, 0], s0[:, 1] = torch.cos(th), torch.sin(th)
        a0 = torch.randn(16, 4, nu, generator=g, dtype=torch.float64)
        ts = torch.tensor([DT, 2 * DT, 3 * DT], dtype=torch.float64)[torch.randint(0, 3, (16,), generator=g)].view(16, 1)
        sn = torch.cat([analytic_step(env, s0[i:i + 1], a0[i:i + 1], float(ts[i]), 1) for i in range(16)])
        out.append((s0, a0, ts, sn))
    return out


def test_training_parity_sgd():
    """20 plain-SGD steps (the reference's loss, train_utils.py:388-407) on our model and on the oracle's fp64 parameters.
    Bound: the parameters' total change agrees within 1e-3 of its magnitude, per tensor."""
    env = "oderl-pendulum"
    sd = _state_dict(env, 128, 17, True)
    m = _model(env, 128, 17, sd)
    names = [n for n, _ in m.named_parameters()]
    ref = {k: v.clone() for k, v in sd.items()}
    for n in names:
        ref[n].requires_grad_(True)
    opt = torch.optim.SGD(m.parameters(), lr=0.05)
    opt_ref = torch.optim.SGD([ref[n] for n in names], lr=0.05)

    with torch.enable_grad():
        for s0, a0, ts, sn in _dataset(env, 20, 1):
            opt.zero_grad()
            loss = torch.nn.functional.mse_loss(m(s0.cuda(), a0.cuda(), ts.cuda()), (sn - s0).cuda())
            loss.backward()
            opt.step()
            opt_ref.zero_grad()
            torch.nn.functional.mse_loss(nl_forward(ref, s0, a0, ts), sn - s0).backward()
            opt_ref.step()
    worst = 0.0
    for n, p in m.named_parameters():
        d_ref = ref[n].detach() - sd[n]
        e = relerr(d_ref, p.detach() - sd[n])
        worst = max(worst, e)
        assert e < 1e-3, (n, e)
    print(f"SGD parity: worst relerr of the parameter change {worst:.2e}")


def test_training_smoke_adam():
    """200 Adam steps with the reference's gradient clip (0.1) on a seeded dataset: the loss falls below half its start."""
    env = "oderl-pendulum"
    m = _model(env, 128, 17, _state_dict(env, 128, 17, True))
    data = _dataset(env, 8, 2)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)

    def full_loss():
        with torch.no_grad():
            return float(sum(torch.nn.functional.mse_loss(m(s0.cuda(), a0.cuda(), ts.cuda()), (sn - s0).cuda()) for s0, a0, ts, sn in data))

    l0 = full_loss()
    with torch.enable_grad():
        for step in range(200):
            s0, a0, ts, sn = data[step % len(data)]
            opt.zero_grad()
            torch.nn.functional.mse_loss(m(s0.cuda(), a0.cuda(), ts.cuda()), (sn - s0).cuda()).backward()
            torch.nn.utils.clip_grad_norm_(m.parameters(), 0.1)
            opt.step()
    l1 = full_loss()
    print(f"Adam smoke: loss {l0:.4e} -> {l1:.4e}")
    assert l1 < 0.5 * l0, (l0, l1)

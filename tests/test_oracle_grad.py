"""CPU checks of the backward's anchor and of the host-side gradient layout: fp64 ``gradcheck`` of the oracle forward (the
reference gradient of ``tests/test_gpu_grad.py``), and ``nlc_model_grad_floats`` against the module's parameter count."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import nl_model


def _random_sd(nx, nu, H, S, encode_obs_time=False, seed=0):
    import neurallaplacecontrol_b200 as nlc

    torch.manual_seed(seed)
    m = nlc.NeuralLaplaceModel(nx, nu, nx, hidden_units=H, s_recon_terms=S, encode_obs_time=encode_obs_time,
                               state_mean=np.linspace(-0.3, 0.3, nx), state_std=np.linspace(0.5, 2.0, nx),
                               action_mean=np.full(nu, 0.2), action_std=np.array([1.5]), normalize=True, normalize_time=True,
                               dt=0.05).double()
    return m, {k: v.detach().clone() for k, v in m.state_dict().items()}


def _small_sd(nx, gin, H, S, g):
    """A reference-layout state_dict at a width the oracle accepts but the kernels do not (H = 8): gradcheck perturbs every
    parameter entry, so the anchor is checked where that stays cheap."""
    Hg, r = H // 2, lambda *shape: 0.5 * torch.randn(*shape, generator=g, dtype=torch.float64)
    pre, mlp = "action_encoder.gru.", "laplace_rep_func.linear_tanh_stack."
    sd = {"state_mean": r(nx), "state_std": 1.0 + torch.rand(nx, generator=g, dtype=torch.float64), "action_mean": r(1),
          "action_std": torch.tensor([1.5], dtype=torch.float64), "dt": torch.tensor(0.05, dtype=torch.float64)}
    for l, n_in in ((0, gin), (1, Hg)):
        sd.update({f"{pre}weight_ih_l{l}": r(3 * Hg, n_in), f"{pre}weight_hh_l{l}": r(3 * Hg, Hg), f"{pre}bias_ih_l{l}": r(3 * Hg),
                   f"{pre}bias_hh_l{l}": r(3 * Hg)})
    sd.update({"action_encoder.linear_out.weight": r(2, Hg), "action_encoder.linear_out.bias": r(2),
               mlp + "0.weight": r(H, 2 * S + nx + 2), mlp + "0.bias": r(H), mlp + "2.weight": r(H, H), mlp + "2.bias": r(H),
               mlp + "4.weight": r(2 * nx * S, H), mlp + "4.bias": r(2 * nx * S)})
    return sd


@pytest.mark.parametrize("encode_obs_time", [False, True])
def test_oracle_forward_gradcheck(encode_obs_time):
    """Every parameter (including the 2S sphere-coordinate columns of the first layer) and the obs / action inputs."""
    nx, nu, H, S, K, B = 3, 1, 8, 5, 3, 3
    g = torch.Generator().manual_seed(1)
    sd = _small_sd(nx, nu + int(encode_obs_time), H, S, g)
    names = [k for k in nl_model.STATE_DICT_KEYS if k.startswith(("action_encoder", "laplace_rep_func"))]
    obs = torch.randn(K, nx, generator=g, dtype=torch.float64, requires_grad=True)
    act = torch.randn(K, B, nu + int(encode_obs_time), generator=g, dtype=torch.float64, requires_grad=True)
    ts = 0.05 * (0.3 + torch.rand(K, 1, generator=g, dtype=torch.float64))
    params = [sd[n].clone().requires_grad_(True) for n in names]

    def f(o, a, *ps):
        d = dict(sd)
        d.update(zip(names, ps))
        return nl_model.nl_forward(d, o, a, ts, normalize=True, normalize_time=True)

    with torch.enable_grad():  # other test modules switch grad mode off process-wide at import
        assert torch.autograd.gradcheck(f, (obs, act, *params), eps=1e-6, atol=1e-5, rtol=1e-4)


@pytest.mark.parametrize("nx,nu,H,S,eot", [(3, 1, 128, 17, False), (5, 1, 64, 33, True), (6, 2, 128, 136, False), (6, 2, 64, 2, False)])
def test_grad_floats_matches_parameter_count(nx, nu, H, S, eot):
    from neurallaplacecontrol_b200 import _lib

    m, _ = _random_sd(nx, nu, H, S, eot)
    d = _lib.ModelDesc()
    d.state_dim, d.action_dim, d.hidden_units, d.s_terms, d.encode_obs_time = nx, nu, H, S, int(eot)
    assert _lib.load().nlc_model_grad_floats(C.byref(d)) == sum(p.numel() for p in m.parameters())

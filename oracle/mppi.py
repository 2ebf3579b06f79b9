"""MPPI-with-delay control step, restated with an injected noise tensor (CPU oracle).

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).

Follows ``planners/mppi_delay.py`` of the reference:
* ``perturb``        - stage 1, ``_compute_total_cost_batch`` ``:315-335`` + ``_bound_action`` ``:347-356``
  (net effect of the per-t slice loop with scalar bounds = elementwise clamp).
* ``rollout_costs``  - stages 2+3, ``_compute_rollout_costs`` ``:232-313`` for M=1, no terminal
  cost, ``encode_obs_time=False`` (the configuration every caller uses).
* ``softmax_update`` - stage 4, ``command`` ``:210-224``.
* ``command``        - ``command`` ``:193-224`` end to end; returns every tensor the reference
  leaves on the planner object (``noise perturbed_action cost_total cost_total_non_zero omega
  states actions U``) plus the action.
* ``combine_shards`` - the K-sharded form of stage 4 (not in the reference; SURVEY 8e): per-shard
  (beta_g, eta_g, W_g) triples merged with the log-sum-exp rescale.
* ``get_action``     - ``mppi_with_model.py:25-28``.
"""
from __future__ import annotations

import torch


def noise_sigma_for(nu, sigma=1.0, dtype=torch.float64):
    """Covariance the callers build (``mppi_with_model.py:66-70``)."""
    gamma = sigma ** 2
    off = 0.5 * gamma
    return torch.ones((nu, nu), dtype=dtype) * off + torch.eye(nu, dtype=dtype) * (gamma - off)


def perturb(U, noise, noise_sigma_inv, lambda_, u_scale, u_min, u_max, sample_null_action=False,
            noise_abs_cost=False):
    """U (T,nu), noise (K,T,nu) -> perturbed (K,T,nu), bounded noise (K,T,nu), perturbation cost (K)."""
    perturbed = U + noise
    if sample_null_action:
        perturbed[-1] = 0
    if u_max is not None:
        perturbed = torch.max(torch.min(perturbed * u_scale, torch.as_tensor(u_max)), torch.as_tensor(u_min))
    else:
        perturbed = perturbed * u_scale
    perturbed = perturbed / u_scale
    noise = perturbed - U
    if noise_abs_cost:
        action_cost = lambda_ * torch.abs(noise) @ noise_sigma_inv
    else:
        action_cost = lambda_ * noise @ noise_sigma_inv
    perturbation_cost = torch.sum(U * action_cost, dim=(1, 2))
    return perturbed, noise, perturbation_cost


def rollout_costs(dynamics, running_cost, state, perturbed, action_buffer, u_scale):
    """state (nx,) or (K,nx); perturbed (K,T,nu) normalised; action_buffer (B,nu) env units.
    Returns cost (K), states (K,T,nx), actions (K,T,nu) (env units, as ``:288,296``)."""
    K, T, nu = perturbed.shape
    nx = state.shape[-1]
    if state.shape != (K, nx):
        state = state.view(1, -1).repeat(K, 1)
    B = action_buffer.shape[0]
    hist = torch.cat((action_buffer[1:].view(1, -1, nu).repeat(K, 1, 1), u_scale * perturbed), dim=1)
    cost = torch.zeros(K, dtype=perturbed.dtype)
    states, actions = [], []
    for t in range(T):
        state = dynamics(state, hist[:, t:t + B, :])
        u = hist[:, t + B - 1, :]
        cost = cost + running_cost(state, u)
        states.append(state)
        actions.append(u)
    return cost, torch.stack(states, dim=-2), torch.stack(actions, dim=-2)


def softmax_update(U, cost_total, noise, lambda_):
    beta = torch.min(cost_total)
    w = torch.exp(-(1.0 / lambda_) * (cost_total - beta))
    eta = torch.sum(w)
    omega = (1.0 / eta) * w
    U = U.clone()
    for t in range(U.shape[0]):
        U[t] += torch.sum(omega.view(-1, 1) * noise[:, t], dim=0)
    return U, w, omega


def command(U, state, action_buffer, noise, dynamics, running_cost, *, noise_sigma, lambda_=1.0,
            u_scale=1.0, u_min=None, u_max=None, u_init=None):
    """One ``MPPIDelay.command`` call with the sampled noise injected."""
    dtype = noise_sigma.dtype
    nu = noise_sigma.shape[0]
    U = torch.roll(U, -1, dims=0)
    U[-1] = torch.zeros(nu, dtype=dtype) if u_init is None else u_init
    state = torch.as_tensor(state).to(dtype)
    sigma_inv = torch.inverse(noise_sigma)
    perturbed, bnoise, pert_cost = perturb(U, noise, sigma_inv, lambda_, u_scale, u_min, u_max)
    cost, states, actions = rollout_costs(dynamics, running_cost, state, perturbed, action_buffer, u_scale)
    actions = actions / u_scale
    cost_total = cost + pert_cost
    U_new, w, omega = softmax_update(U, cost_total, bnoise, lambda_)
    return {
        "noise": bnoise, "perturbed_action": perturbed, "cost_total": cost_total,
        "cost_total_non_zero": w, "omega": omega, "states": states, "actions": actions,
        "U": U_new, "action": U_new[0] * u_scale, "rollout_cost": cost, "perturbation_cost": pert_cost,
    }


def shard_triple(cost_total, noise, lambda_):
    """Per-shard partial of stage 4: (beta_g, eta_g, W_g[T,nu]).  A +inf cost weighs 0 as in ``softmax_update``, also when
    every cost of the shard is +inf (beta_g = +inf, where exp(-(inf - inf)) would be NaN): such a shard adds nothing."""
    beta = torch.min(cost_total)
    w = torch.exp(-(1.0 / lambda_) * (cost_total - beta))
    w = torch.where(cost_total == float("inf"), torch.zeros_like(w), w)
    return beta, torch.sum(w), torch.einsum("k,ktu->tu", w, noise)


def combine_shards(U, triples, lambda_):
    """Merge per-shard triples with the log-sum-exp rescale and apply the update."""
    beta = torch.min(torch.stack([b for b, _, _ in triples]))
    eta = sum(e * torch.exp(-(b - beta) / lambda_) for b, e, _ in triples)
    W = sum(w * torch.exp(-(b - beta) / lambda_) for b, _, w in triples)
    return U + W / eta, beta, eta


def get_action(action_buffer, action, action_delay):
    action_buffer = torch.roll(action_buffer, -1, dims=0)
    action_buffer[-1] = action
    return action_buffer, action_buffer[-(action_delay + 1)]


def make_nl_dynamics(sd, dt, encode_obs_time=False):
    """The ``dynamics`` closure of ``mppi_with_model.py:103-122`` over the oracle model.  With ``encode_obs_time`` the
    window gets the extra channel ``B-1 .. 0`` (``:110-119``)."""
    from . import nl_model

    def dynamics(state, window):
        ts = torch.full((state.shape[0], 1), dt, dtype=state.dtype)
        if encode_obs_time:
            B = window.shape[1]
            tchan = torch.flip(torch.arange(B), (0,)).view(1, B, 1).to(window.dtype).repeat(window.shape[0], 1, 1)
            window = torch.cat((window, tchan), dim=2)
        return state + nl_model.nl_forward(sd, state, window, ts)

    return dynamics

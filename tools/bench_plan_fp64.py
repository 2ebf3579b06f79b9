"""The fp64 planner (``MPPIDelay(math_mode="fp64")``) at BASELINE configs 1, 3 and 4 (SURVEY 8d inputs, calibrated weights,
the injected noise of ``_util.injected_noise``), timed with CUDA events against, alternating in the same process:

  (a) the composition a user can write without it: the reference's control step (``oracle.mppi.command``'s structure) on the
      GPU with ``NeuralLaplaceModel(math_mode="fp64")`` as ``dynamics`` - T model calls and torch glue per step;
  (b) the default ``tc_split3`` planner, for context.

Prints ms per control step (host inputs and device inputs), model rollout-steps/s, achieved fp64 FLOP/s from the hoisted
per-step operation counts of SURVEY 8d (no share of peak: the card's DFMA rate is not measured here), the max relative
difference of the fp64 planner against (a) on every post-call tensor, and the card's name and power limit.

    python tools/bench_plan_fp64.py [--configs cfg1,cfg3,cfg4] [--steps 10] [--warmup 2]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CONFIGS = {"cfg1": ("oderl-pendulum", 1000, 20), "cfg3": ("oderl-cartpole", 8192, 30), "cfg4": ("oderl-acrobot", 65536, 50)}
KEYS = ("noise", "perturbed_action", "cost_total", "cost_total_non_zero", "omega", "states", "actions", "U")


def model_flops_per_step(nx, nu, H=128, S=17, B=4):
    """fp64 operations of one model evaluation per sample (multiply-add = 2): the B-step two-layer GRU, linear_out, the MLP
    after the hoisted s-point columns, and the S-term ILT (counted as one multiply-add per term and channel)."""
    Hg = H // 2
    gin = nu
    gru = B * 2 * (3 * Hg * gin + 3 * Hg * Hg) + B * 2 * (3 * Hg * Hg + 3 * Hg * Hg)
    mlp = 2 * (H * (nx + 2) + H * H + 2 * nx * S * H)
    return gru + 2 * 2 * Hg + mlp + 2 * nx * S


def composition(model, env, U, state, buf, noise, u_scale, dt, lam=1.0, bounds=None):
    """The reference's control step (oracle.mppi.command: perturb, T calls of ``state + model(state, window, dt)``, running
    cost, softmax update) on CUDA tensors with the given model as dynamics.  Returns the post-call tensors and the action."""
    from oracle import costs, mppi

    dev = noise.device
    nu = noise.shape[-1]
    K, T = noise.shape[0], noise.shape[1]
    B = buf.shape[0]
    U = torch.roll(U, -1, dims=0)
    U[-1] = 0
    sigma_inv = torch.inverse(mppi.noise_sigma_for(nu)).to(dev)
    lo, hi = (None, None) if bounds is None else bounds
    perturbed, bnoise, pert_cost = mppi.perturb(U, noise, sigma_inv, lam, u_scale, lo, hi)
    hist = torch.cat((buf[1:].view(1, -1, nu).repeat(K, 1, 1), u_scale * perturbed), dim=1)
    s = state.view(1, -1).repeat(K, 1)
    ts = torch.full((K, 1), dt, dtype=torch.float64, device=dev)
    run = costs.running_cost(env)
    cost = torch.zeros(K, dtype=torch.float64, device=dev)
    states = []
    for t in range(T):
        s = s + model(s, hist[:, t:t + B], ts).reshape(K, -1)
        cost = cost + run(s, hist[:, t + B - 1])
        states.append(s)
    cost_total = cost + pert_cost
    U_new, w, omega = mppi.softmax_update(U, cost_total, bnoise, lam)
    return {"noise": bnoise, "perturbed_action": perturbed, "cost_total": cost_total, "cost_total_non_zero": w, "omega": omega,
            "states": torch.stack(states, dim=1), "actions": hist[:, B - 1:] / u_scale, "U": U_new, "action": U_new[0] * u_scale}


def build(env, K, T, math_mode, seed=1):
    import neurallaplacecontrol_b200 as nlc
    from _util import DT, S_TERMS, START_STATE, injected_noise, weights
    from oracle import costs

    nx, nu = costs.ENV_DIMS[env]
    ah = np.float32(costs.ENV_ACT_HIGH[env])
    m = nlc.NeuralLaplaceModel(nx, nu, nx, hidden_units=128, s_recon_terms=S_TERMS, state_mean=np.zeros(nx), state_std=np.ones(nx),
                               action_mean=np.zeros(nu), action_std=np.ones(1), normalize=True, normalize_time=True, dt=DT,
                               math_mode="fp64" if math_mode == "composition" else math_mode, device="cuda:0").double().cuda()
    m.load_state_dict(weights(env, calibrated=True))
    noise = injected_noise(K, T, nu, seed=seed)
    state = np.array(START_STATE[env])
    if math_mode == "composition":
        return m, noise.cuda(), state, ah
    p = nlc.MPPIDelay(nlc.NLDynamics(m, DT), nlc.EnvRunningCost(env), nx, nlc.noise_sigma_for(nu), num_samples=K, horizon=T,
                      device="cuda:0", lambda_=1.0, u_min=torch.tensor(-ah), u_max=torch.tensor(ah), u_scale=ah,
                      U_init=torch.zeros(T, nu, dtype=torch.float64), math_mode=math_mode)
    return p, noise, state, ah


def relerr(ref, got):
    ref, got = ref.double(), got.double().reshape(ref.shape)
    return float((ref - got).abs().max() / ref.abs().max().clamp_min(1e-30))


def time_it(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception:
        return "unknown"


def run_config(name, steps, warmup):
    from _util import DT
    from oracle import costs

    env, K, T = CONFIGS[name]
    nx, nu = costs.ENV_DIMS[env]
    p64, noise, state, ah = build(env, K, T, "fp64")
    noise_dev = noise.cuda()
    p64.noise_dist.sample = lambda shape: noise_dev
    ptc, _, _, _ = build(env, K, T, "tc_split3")
    ptc.noise_dist.sample = lambda shape: noise_dev
    m, _, _, _ = build(env, K, T, "composition")
    buf_h = torch.zeros(4, nu, dtype=torch.float64)
    buf_d, state_d = buf_h.cuda(), torch.from_numpy(state).cuda()
    lo, hi = torch.tensor(-float(ah), dtype=torch.float64), torch.tensor(float(ah), dtype=torch.float64)

    # accuracy: one step from U = 0 against the composition on the same inputs
    p64.U = torch.zeros(T, nu, dtype=torch.float64)
    a64 = p64.command(state_d, buf_d)
    with torch.no_grad():
        ref = composition(m, env, torch.zeros(T, nu, dtype=torch.float64, device="cuda"), state_d, buf_d, noise_dev, float(ah), DT,
                          bounds=(lo, hi))
    errs = {k: relerr(ref[k], getattr(p64, k)) for k in KEYS}
    errs["action"] = relerr(ref["action"], a64)

    def f64_host():  # the fp64 planner with host inputs: one C call (the on-device sampler: no injection on this path)
        del p64.noise_dist.sample
        p64.command(state, buf_h)
        p64.noise_dist.sample = lambda shape: noise_dev

    def f64_dev():
        p64.command(state_d, buf_d)

    def comp():
        with torch.no_grad():
            composition(m, env, torch.zeros(T, nu, dtype=torch.float64, device="cuda"), state_d, buf_d, noise_dev, float(ah), DT,
                        bounds=(lo, hi))

    def tc():
        ptc.command(state_d, buf_d)

    res = {k: [] for k in ("fp64_host", "fp64_device", "composition", "tc_split3")}
    for rnd in range(2):  # alternate the forms
        for k, fn in (("fp64_host", f64_host), ("fp64_device", f64_dev), ("composition", comp), ("tc_split3", tc)):
            res[k].append(time_it(fn, steps, warmup if rnd == 0 else 1))
    ms = {k: min(v) for k, v in res.items()}
    flop = model_flops_per_step(nx, nu) * K * T
    out = {"config": name, "env": env, "K": K, "T": T, "ms": {k: round(v, 4) for k, v in ms.items()},
           "ms_all": {k: [round(x, 4) for x in v] for k, v in res.items()},
           "fp64_rollout_steps_per_s": K * T / (ms["fp64_device"] * 1e-3),
           "fp64_model_gflops": flop / (ms["fp64_device"] * 1e-3) / 1e9, "model_flop_per_step": flop,
           "speedup_vs_composition": ms["composition"] / ms["fp64_device"],
           "max_relerr_vs_composition": max(errs.values()), "relerr_vs_composition": errs}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="cfg1,cfg3,cfg4")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_plan_fp64 needs a CUDA device")
    torch.set_grad_enabled(False)
    print(json.dumps({"card": card(), "torch": torch.__version__}))
    for name in args.configs.split(","):
        print(json.dumps(run_config(name, args.steps, args.warmup)), flush=True)


if __name__ == "__main__":
    main()

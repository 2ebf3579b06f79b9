"""The fp64 closed loop (``run_closed_loop`` over one ``MPPIDelay(math_mode="fp64")`` per instance, fp64 ``env_step``) timed
with CUDA events around ``--steps`` loop steps after a warm-up loop, in ms per control step of all instances, for two shapes
(calibrated weights, Neural Laplace dynamics, delay 1, on-device sampler):

  (a) pendulum, 8 instances, K = 1000, H = 20;
  (b) acrobot, 4 instances, K = 4096, H = 30 (the per-instance size of BASELINE config 5).

Beside each: the instance-batched ``BatchedMPPIDelay`` loop (default ``tc_split3`` arithmetic, fp32 state) at the same shape,
the fp64 ``env_step`` alone on the shape's I instances (CUDA events around 1000 calls, and ``env_step_f64_kernel``'s own
device time from ``torch.profiler`` in a separate pass), and at (a) the CPU fp64 oracle
loop (``oracle.dynamics.closed_loop`` around ``oracle.mppi.command``, host clock, ``--cpu-steps`` steps) with the core count.
The first line is the card's name and power limit, read in the same run.

    python tools/bench_episode_fp64.py [--steps 10] [--warmup 2] [--cpu-steps 2]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SHAPES = {"a": ("oderl-pendulum", 8, 1000, 20), "b": ("oderl-acrobot", 4, 4096, 30)}
DELAY = 1


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=30).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def start_states(env, I):
    from _util import START_STATE

    rng = np.random.default_rng(0)
    s0 = np.array(START_STATE[env])
    return torch.tensor(np.stack([s0 + rng.uniform(-0.05, 0.05, s0.shape) for _ in range(I)]), dtype=torch.float64)


def build(env, I, K, T, kind):
    """``kind`` "fp64": a list of fp64 planners (seeds 0 .. I-1); "batched": one BatchedMPPIDelay with the same seeds."""
    import neurallaplacecontrol_b200 as nlc
    from _util import DT, S_TERMS, weights
    from oracle import costs

    nx, nu = costs.ENV_DIMS[env]
    ah = np.float32(costs.ENV_ACT_HIGH[env])
    m = nlc.NeuralLaplaceModel(nx, nu, nx, hidden_units=128, s_recon_terms=S_TERMS, state_mean=np.zeros(nx), state_std=np.ones(nx),
                               action_mean=np.zeros(nu), action_std=np.ones(1), normalize=True, normalize_time=True, dt=DT,
                               device="cuda:0").double()
    m.load_state_dict(weights(env, calibrated=True))
    args = (nlc.NLDynamics(m, DT), nlc.EnvRunningCost(env), nx, nlc.noise_sigma_for(nu))
    kw = dict(num_samples=K, horizon=T, device="cuda:0", lambda_=1.0, u_min=torch.tensor(-ah), u_max=torch.tensor(ah), u_scale=ah,
              keep_states=False)
    if kind == "batched":
        return nlc.BatchedMPPIDelay(*args, I, seeds=list(range(I)), U_init=torch.zeros(T, nu, dtype=torch.float64), **kw)
    return [nlc.MPPIDelay(*args, U_init=torch.zeros(T, nu, dtype=torch.float64), seed=i, math_mode="fp64", **kw) for i in range(I)]


def time_loop(planner, env, st0, steps, warmup):
    """ms per control step of ``run_closed_loop`` (its own per-step synchronise included), CUDA events around the call."""
    import neurallaplacecontrol_b200 as nlc
    from _util import DT

    nlc.run_closed_loop(planner, env, st0, DELAY, warmup, DT)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res = nlc.run_closed_loop(planner, env, st0, DELAY, steps, DT)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, res


def time_env_step(env, I, n=1000):
    """(us per env_step call, us of env_step_f64_kernel on the device) on I instances (device tensors, rewards written): CUDA
    events around n back-to-back calls (launch-bound at these sizes), then the kernel's own duration from torch.profiler in
    a separate pass."""
    import neurallaplacecontrol_b200 as nlc
    from _util import DT
    from oracle import costs
    from torch.profiler import ProfilerActivity, profile

    nx, nu = costs.ENV_DIMS[env]
    s = start_states(env, I).cuda()
    b = torch.zeros(I, 4, nu, dtype=torch.float64, device="cuda")
    a = torch.full((I, nu), 0.1, dtype=torch.float64, device="cuda")
    r = torch.zeros(I, dtype=torch.float64, device="cuda")
    for _ in range(10):
        nlc.env_step(env, s, b, a, DELAY, DT, r)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        nlc.env_step(env, s, b, a, DELAY, DT, r)
    e1.record()
    torch.cuda.synchronize()
    call_us = 1e3 * e0.elapsed_time(e1) / n
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(200):
            nlc.env_step(env, s, b, a, DELAY, DT, r)
        torch.cuda.synchronize()
    rows = [k for k in prof.key_averages() if "env_step_f64_kernel" in k.key]
    total = sum(getattr(k, "self_device_time_total", 0.0) or k.self_cuda_time_total for k in rows)
    return call_us, total / max(sum(k.count for k in rows), 1)


def time_cpu_oracle(env, I, K, T, steps):
    """ms per control step of the fp64 oracle loop on the CPU (on-host sampler: torch.randn @ chol^T per instance and step)."""
    from _util import DT, weights
    from oracle import costs, dynamics as odyn, mppi

    nx, nu = costs.ENV_DIMS[env]
    ah = float(np.float32(costs.ENV_ACT_HIGH[env]))
    dyn = mppi.make_nl_dynamics(weights(env, calibrated=True), DT)
    chol = torch.linalg.cholesky(mppi.noise_sigma_for(nu))
    lo, hi = torch.tensor(-ah, dtype=torch.float64), torch.tensor(ah, dtype=torch.float64)
    Us = [torch.zeros(T, nu, dtype=torch.float64) for _ in range(I)]

    def plan_fn(i, state, buf):
        noise = torch.randn(K, T, nu, dtype=torch.float64) @ chol.T
        out = mppi.command(Us[i], state, buf, noise, dyn, costs.running_cost(env), noise_sigma=mppi.noise_sigma_for(nu), u_scale=ah,
                           u_min=lo, u_max=hi)
        Us[i] = out["U"]
        return out["action"]

    t0 = time.perf_counter()
    odyn.closed_loop(env, plan_fn, start_states(env, I), DELAY, steps, DT)
    return 1e3 * (time.perf_counter() - t0) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="a,b")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--cpu-steps", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_episode_fp64 needs a CUDA device")
    torch.set_grad_enabled(False)
    print(json.dumps({"card": card(), "torch": torch.__version__, "cpu_cores": os.cpu_count(), "torch_threads": torch.get_num_threads()}))
    for name in args.shapes.split(","):
        env, I, K, T = SHAPES[name]
        st0 = start_states(env, I)
        f64, bat = build(env, I, K, T, "fp64"), build(env, I, K, T, "batched")
        ms = {"fp64_loop": [], "batched_tc_split3_loop": []}
        for rnd in range(2):  # alternate the two loops
            for key, p in (("fp64_loop", f64), ("batched_tc_split3_loop", bat)):
                t, res = time_loop(p, env, st0, args.steps, args.warmup if rnd == 0 else 1)
                ms[key].append(round(t, 4))
                assert np.isfinite(res["total_reward_raw"]).all(), (name, key)
        call_us, kernel_us = time_env_step(env, I)
        out = {"shape": name, "env": env, "I": I, "K": K, "H": T, "steps": args.steps,
               "ms_per_control_step": {k: min(v) for k, v in ms.items()}, "ms_all": ms,
               "env_step_f64_call_us": round(call_us, 3), "env_step_f64_kernel_us": round(kernel_us, 3)}
        out["fp64_rollout_steps_per_s"] = I * K * T / (out["ms_per_control_step"]["fp64_loop"] * 1e-3)
        if name == "a":
            out["cpu_fp64_oracle_loop_ms"] = round(time_cpu_oracle(env, I, K, T, args.cpu_steps), 1)
            out["cpu_steps"] = args.cpu_steps
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()

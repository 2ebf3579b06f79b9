"""hidden_units = 64 (the reference class default, w_nl.py:71) against hidden_units = 128, timed with CUDA events in one process:

  * the device control step (``MPPIDelay.set_inputs`` once, then ``MPPIDelay.step``: one graph launch per step) at BASELINE
    configs 1, 3 and 4, hidden 64 with S in {17, 33} in ``fp32``, ``tc_split3`` and ``tc_fp16``, and hidden 128 ``tc_split3``
    (S = 17, the calibrated golden weights) beside them;
  * ``NeuralLaplaceModel.forward`` at one prediction time, K = 65536 acrobot samples, window 4, the same models.

Hidden-64 weights are the seeded models of tests/test_gpu_hidden64_tc.py (phi bias in the trained operating range).  Every
variant is timed twice, the variants alternating, and the smaller time is reported.  The first line names the card and its
power limit, read in the same run.

    python tools/bench_hidden64.py [--configs cfg1,cfg3,cfg4] [--steps 20] [--warmup 3]
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
VARIANTS = [(64, 17, "fp32"), (64, 17, "tc_split3"), (64, 17, "tc_fp16"), (64, 33, "fp32"), (64, 33, "tc_split3"), (64, 33, "tc_fp16"),
            (128, 17, "tc_split3")]
FWD_K = 65536


def model(env, H, S, mode):
    import neurallaplacecontrol_b200 as nlc
    from _util import DT, weights
    from oracle import costs
    from test_gpu_multi_time import _model, _state_dict

    if H == 64:
        return _model(env, _state_dict(env, H, S, calibrated=True), H, S, math_mode=mode)
    nx, nu = costs.ENV_DIMS[env]
    m = nlc.NeuralLaplaceModel(nx, nu, nx, hidden_units=128, s_recon_terms=S, state_mean=np.zeros(nx), state_std=np.ones(nx),
                               action_mean=np.zeros(nu), action_std=np.ones(1), normalize=True, normalize_time=True, dt=DT,
                               math_mode=mode, device="cuda:0").double()
    m.load_state_dict(weights(env, calibrated=True))
    return m


def planner(env, K, T, H, S, mode):
    import neurallaplacecontrol_b200 as nlc
    from _util import DT, START_STATE, injected_noise
    from oracle import costs

    nx, nu = costs.ENV_DIMS[env]
    ah = np.float32(costs.ENV_ACT_HIGH[env])
    p = nlc.MPPIDelay(nlc.NLDynamics(model(env, H, S, mode), DT), nlc.EnvRunningCost(env), nx, nlc.noise_sigma_for(nu), num_samples=K,
                      horizon=T, device="cuda:0", lambda_=1.0, u_min=torch.tensor(-ah), u_max=torch.tensor(ah), u_scale=ah,
                      U_init=torch.zeros(T, nu, dtype=torch.float64), math_mode=mode)
    noise = injected_noise(K, T, nu, seed=1).cuda()
    p.noise_dist.sample = lambda shape: noise
    p.set_inputs(np.array(START_STATE[env]), torch.zeros(4, nu, dtype=torch.float64))
    return p


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


def key(H, S, mode):
    return f"H{H}_S{S}_{mode}"


def run_config(name, steps, warmup):
    env, K, T = CONFIGS[name]
    ps = {key(*v): planner(env, K, T, *v) for v in VARIANTS}
    res = {k: [] for k in ps}
    for rnd in range(2):  # alternate the variants
        for k, p in ps.items():
            res[k].append(time_it(p.step, steps, warmup if rnd == 0 else 1))
    ms = {k: min(v) for k, v in res.items()}
    return {"what": "device step", "config": name, "env": env, "K": K, "T": T, "ms": {k: round(v, 4) for k, v in ms.items()},
            "ms_all": {k: [round(x, 4) for x in v] for k, v in res.items()},
            "rollout_steps_per_s_M": {k: round(K * T / (v * 1e-3) / 1e6, 1) for k, v in ms.items()},
            "tc_split3_vs_fp32_H64": {f"S{S}": round(ms[key(64, S, "fp32")] / ms[key(64, S, "tc_split3")], 2) for S in (17, 33)}}


def run_forward(steps, warmup):
    from _util import DT
    from test_gpu_multi_time import _inputs

    env = "oderl-acrobot"
    obs, act, _ = _inputs(env, FWD_K, 1, seed=2)
    obs, act, t = obs.cuda(), act.cuda(), torch.tensor(DT, dtype=torch.float64).cuda()
    ms = {k: [] for k in (key(*v) for v in VARIANTS)}
    models = {key(*v): model(env, *v) for v in VARIANTS}
    for rnd in range(2):
        for k, m in models.items():
            ms[k].append(time_it(lambda m=m: m(obs, act, t), steps, warmup if rnd == 0 else 1))
    best = {k: min(v) for k, v in ms.items()}
    return {"what": "model forward", "env": env, "K": FWD_K, "B": 4, "ms": {k: round(v, 4) for k, v in best.items()},
            "ms_all": {k: [round(x, 4) for x in v] for k, v in ms.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="cfg1,cfg3,cfg4")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_hidden64 needs a CUDA device")
    torch.set_grad_enabled(False)
    print(json.dumps({"card": card(), "torch": torch.__version__}), flush=True)
    for name in args.configs.split(","):
        print(json.dumps(run_config(name, args.steps, args.warmup)), flush=True)
    print(json.dumps(run_forward(args.steps, args.warmup)), flush=True)


if __name__ == "__main__":
    main()

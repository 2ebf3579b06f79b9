#!/usr/bin/env python
"""One GPU's config-5 share as the reference's delay x seed grid of ONE environment with a model per task: acrobot,
32 instances, K = 4096, H = 30, tc_split3, on-device sampler; action delays cycle 0..3 over the instances and M of them
share a model (M distinct models: seeded perturbations of the calibrated weights; instance i has model i // (32 / M)).

A control step of all instances is the planner's command plus one env_step with the per-instance delays.  Three ways to
plan it:
  (a) single   - today's single-model batch: BatchedMPPIDelay(dyn), M = 1 (one run);
  (b) multi    - BatchedMPPIDelay([dyn_0, ..., dyn_31]): one run per model, the runs on the handle's stream pool;
  (c) sequence - M single-model batches of 32 / M instances, stepped one after another on one stream.
--streams also times (b) with fan-out pools of other sizes (NLC_FANOUT_STREAMS).

Timing: CUDA events on the current stream around `--steps` control steps after `--warmup`, every configuration measured
`--reps` times in alternation; the median (and the spread) is printed with the card's name and power limit.

    python tools/bench_fanout.py [--models 1,4,8,32] [--streams 1,2,4,8] [--steps 20] [--reps 3]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import neurallaplacecontrol_b200 as nlc  # noqa: E402
from _util import DT, S_TERMS, START_STATE, weights  # noqa: E402
from oracle import costs  # noqa: E402

ENV = "oderl-acrobot"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else torch.cuda.get_device_name(0) + ", power limit unknown"


def models(M, dev, math):
    nx, nu = costs.ENV_DIMS[ENV]
    base = weights(ENV, calibrated=True)
    out = []
    for j in range(M):
        g = torch.Generator().manual_seed(1000 + j)
        sd = {k: (v + 0.02 * v.std() * torch.randn(v.shape, generator=g, dtype=v.dtype) if j and v.numel() > 1 and
                  (k.endswith("weight") or ".weight_" in k or k.endswith("bias") or ".bias_" in k) else v) for k, v in base.items()}
        m = nlc.NeuralLaplaceModel(nx, nu, nx, hidden_units=128, s_recon_terms=S_TERMS, state_mean=np.zeros(nx), state_std=np.ones(nx),
                                   action_mean=np.zeros(nu), action_std=np.ones(1), normalize=True, normalize_time=True, dt=DT,
                                   device=dev, math_mode=math).double()
        m.load_state_dict(sd)
        out.append(m)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--instances", type=int, default=32)
    ap.add_argument("--K", type=int, default=4096)
    ap.add_argument("--H", type=int, default=30)
    ap.add_argument("--math", default="tc_split3")
    ap.add_argument("--models", default="1,4,8,32")
    ap.add_argument("--streams", default="", help="fan-out pool sizes to time (b) with, e.g. 1,2,4,8 (default: the built-in size)")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    I, K, H = args.instances, args.K, args.H
    nx, nu = costs.ENV_DIMS[ENV]
    ah = costs.ENV_ACT_HIGH[ENV]
    kw = dict(num_samples=K, horizon=H, device=dev, u_min=torch.tensor(-ah), u_max=torch.tensor(ah), u_scale=ah, math_mode=args.math)
    Ms = [int(x) for x in args.models.split(",")]
    pools = [int(x) for x in args.streams.split(",")] if args.streams else [None]
    all_models = models(max(Ms), dev, args.math)
    delays = [i % 4 for i in range(I)]
    st0 = torch.stack([torch.tensor(np.array(START_STATE[ENV]) + np.random.default_rng(i).uniform(-0.05, 0.05, nx), dtype=torch.float32)
                       for i in range(I)])
    cost, sig = nlc.EnvRunningCost(ENV), nlc.noise_sigma_for(nu)

    def batch(dyn, ids, pool=None):
        if pool is None:
            os.environ.pop("NLC_FANOUT_STREAMS", None)
        else:
            os.environ["NLC_FANOUT_STREAMS"] = str(pool)
        b = nlc.BatchedMPPIDelay(dyn, cost, nx, sig, len(ids), seeds=ids, **kw)
        b.command(st0[ids].to(dev), torch.zeros(len(ids), 4, nu, device=dev))  # creates the device handle (reads the pool size)
        os.environ.pop("NLC_FANOUT_STREAMS", None)
        return b

    configs = []  # (name, M, pool, [(planner, instance ids)])
    ids = list(range(I))
    configs.append(("a_single", 1, None, [(batch(nlc.NLDynamics(all_models[0], DT), ids), ids)]))
    for M in Ms:
        per = I // M
        dyns = [nlc.NLDynamics(all_models[i // per], DT) for i in ids]
        for pool in pools:
            configs.append(("b_multi", M, pool, [(batch(dyns, ids, pool), ids)]))
        configs.append(("c_sequence", M, None, [(batch(nlc.NLDynamics(all_models[j], DT), ids[j * per:(j + 1) * per]), ids[j * per:(j + 1) * per])
                                                for j in range(M)]))

    states = st0.to(dev).contiguous()
    bufs = torch.zeros(I, 4, nu, device=dev)
    reward = torch.zeros(I, device=dev)
    actions = torch.zeros(I, nu, device=dev)

    def control_step(parts):
        for p, sel in parts:
            if len(parts) == 1:
                actions.copy_(p.command(states, bufs))
            else:
                i0, i1 = sel[0], sel[-1] + 1
                actions[i0:i1] = p.command(states[i0:i1], bufs[i0:i1])
        nlc.env_step(ENV, states, bufs, actions, delays, DT, reward)

    def timed(parts):
        states.copy_(st0.to(dev))
        bufs.zero_()
        for _ in range(args.warmup):
            control_step(parts)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            control_step(parts)
        e1.record()
        e1.synchronize()
        assert bool(torch.isfinite(states).all())
        return e0.elapsed_time(e1) / args.steps

    times = {i: [] for i in range(len(configs))}
    for _ in range(args.reps):
        for i, (_, _, _, parts) in enumerate(configs):
            times[i].append(timed(parts))
    gpu = card()
    print(f"# {gpu}; acrobot, {I} instances x K={K} H={H}, {args.math}, delays cycling 0..3", flush=True)
    for i, (name, M, pool, parts) in enumerate(configs):
        ms = statistics.median(times[i])
        print(json.dumps({"variant": name, "models": M, "runs_or_batches": len(parts) if name != "b_multi" else M,
                          "fanout_streams": pool if pool is not None else ("built-in" if name == "b_multi" and M > 1 else None),
                          "ms_per_control_step_all_instances": round(ms, 4), "spread_ms": [round(min(times[i]), 4), round(max(times[i]), 4)],
                          "rollout_steps_per_s": round(I * K * H / (ms * 1e-3)), "card": gpu}), flush=True)


if __name__ == "__main__":
    main()

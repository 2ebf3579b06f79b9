#!/usr/bin/env python
"""Rollout microbenchmark (representation MLP + Fourier ILT + cost over the horizon, encoder output given), timed alone
with CUDA events over a sweep of K.     python tools/bench_rollout.py [--env oderl-acrobot] [--H 50] [--math tc_split3] K ...
NLC_ROLLOUT_TILES=1|3 in the environment forces the one-tile or the ping-pong form (default: by plan size)."""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import neurallaplacecontrol_b200 as nlc  # noqa: E402
from neurallaplacecontrol_b200 import _lib  # noqa: E402
from _util import DT, S_TERMS, weights  # noqa: E402
from oracle import costs  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--env", default="oderl-acrobot")
    ap.add_argument("--H", type=int, default=50)
    ap.add_argument("--math", default="tc_split3")
    ap.add_argument("Ks", nargs="*", type=int, default=[65536])
    args = ap.parse_args()
    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    nx, nu = costs.ENV_DIMS[args.env]
    model = nlc.NeuralLaplaceModel(nx, nu, nx, hidden_units=128, s_recon_terms=S_TERMS, state_mean=np.zeros(nx), state_std=np.ones(nx),
                                   action_mean=np.array([0] * nu), action_std=np.array([1.0]), normalize=True, normalize_time=True,
                                   dt=DT, device=dev).double()
    model.load_state_dict(weights(args.env, calibrated=True))
    mh = model.set_prediction_time(DT)
    lib = _lib.load()
    B, H = 4, args.H
    mode = _lib.MATH_MODES[args.math]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    start = {"oderl-pendulum": [-1.0, 0.0, 1.0], "oderl-cartpole": [0.0, 0.0, -1.0, 0.0, 0.0], "oderl-acrobot": [1.0, 0.0, 1.0, 0.0, 0.0, 0.0]}
    st = torch.tensor(start[args.env], dtype=torch.float32, device=dev)
    ro = _lib.RolloutOpts()
    ro.env, ro.state_constraint, ro.goal_x, ro.dynamics, ro.delay, ro.dt = _lib.ENV_IDS[args.env], 0, 0.0, 0, 0, DT
    for K in args.Ks:
        g = torch.Generator(device=dev).manual_seed(3)
        hist = torch.randn(K, B - 1 + H, nu, generator=g, device=dev, dtype=torch.float32)
        p = torch.empty(K, H, 2, device=dev, dtype=torch.float32)
        _lib.check(lib.nlc_encode_history(mh, hist.data_ptr(), K, H, B, p.data_ptr(), mode, _lib.current_stream_ptr()))
        cost = torch.empty(K, device=dev, dtype=torch.float32)
        states = torch.empty(K, H, nx, device=dev, dtype=torch.float32)

        def run():
            _lib.check(lib.nlc_rollout_cost(mh, C.byref(ro), st.data_ptr(), 0, p.data_ptr(), hist.data_ptr(), None, K, H, B, nu,
                                            cost.data_ptr(), states.data_ptr(), mode, _lib.current_stream_ptr()))
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        ms = []
        for _ in range(5):
            if not os.environ.get("NO_FLUSH"):
                flush.fill_(1)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(); run(); e.record(); e.synchronize()
            ms.append(s.elapsed_time(e))
        m = sorted(ms)[len(ms) // 2]
        print(json.dumps({"K": K, "H": H, "env": args.env, "math": args.math, "tiles": os.environ.get("NLC_ROLLOUT_TILES", "auto"), "ms": m,
                          "rollout_steps_per_s": K * H / (m * 1e-3), "cost_checksum": float(cost.double().sum())}), flush=True)


if __name__ == "__main__":
    main()

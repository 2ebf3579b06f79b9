#!/usr/bin/env python
"""History-encoder microbenchmark: the K x H window pass of BASELINE config 4 (acrobot, K=65536, H=50) timed alone with
CUDA events for each kernel form / measurement ablation given on the command line.

    python tools/bench_encoder.py [--env oderl-acrobot] [--K 65536] [--H 50] [--math tc_split3] VARIANT ...

A VARIANT is a comma-separated list of NAME=VALUE environment settings applied before each timing (any name works as a
label for repeated runs).  The NLC_ENC_ABLATE bit mask behind profiles/r1_encoder_ablation.md and the NLC_ENC_RCP
reciprocal flavours of DESIGN.md §3a were removed from the production kernel after those measurements.
"""
import argparse
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
    ap.add_argument("--K", type=int, default=65536)
    ap.add_argument("--H", type=int, default=50)
    ap.add_argument("--math", default="tc_split3")
    ap.add_argument("variants", nargs="*", default=["NLC_ENC_ABLATE=0"])
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
    B = 4
    g = torch.Generator(device=dev).manual_seed(3)
    hist = torch.randn(args.K, B - 1 + args.H, nu, generator=g, device=dev, dtype=torch.float32)
    p = torch.empty(args.K, args.H, 2, device=dev, dtype=torch.float32)
    mode = _lib.MATH_MODES[args.math]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def run():
        _lib.check(lib.nlc_encode_history(mh, hist.data_ptr(), args.K, args.H, B, p.data_ptr(), mode, _lib.current_stream_ptr()))

    ref = None
    for var in args.variants:
        for kv in var.split(","):
            k, v = kv.split("=")
            os.environ[k] = v
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        ms = []
        for _ in range(5):
            flush.fill_(1)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(); run(); e.record(); e.synchronize()
            ms.append(s.elapsed_time(e))
        out = p.double().cpu()
        if ref is None:
            ref = out
        print(json.dumps({"variant": var, "ms": sorted(ms)[len(ms) // 2], "windows_per_s": args.K * args.H / (sorted(ms)[len(ms) // 2] * 1e-3),
                          "max_abs_diff_vs_first": float((out - ref).abs().max())}), flush=True)


if __name__ == "__main__":
    main()

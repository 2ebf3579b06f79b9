"""Times NeuralLaplaceModel.forward with several prediction times per sample, ts_pred (K, n_t) (nlc_model_forward_multi /
nlc_model_backward_multi), against the same outputs by other routes, on acrobot at hidden 128, S 17, window B 4:
  * "multi":    the module with ts_pred (K, n_t): each window encoded once, the MLP + ILT over the K n_t rows;
  * "repeated": every row repeated n_t times and the module called with (K n_t, 1) times (nlc_model_forward_ts /
                nlc_model_backward_ts), which encodes every window n_t times;
  * "eager":    fp32 torch-eager autograd of oracle.nl_forward on the same GPU.
For each, "fwd" is the forward alone (no grad), "fwd_bwd" forward + backward of a fixed output gradient into every
parameter and obs / act, both by CUDA events around `--iters` calls after `--warmup` calls.  With n_t = 1 "multi" is the
(K, 1) path itself.  Prints the card's name and power limit, then one JSON line per (K, n_t, route).
usage: python tools/bench_multi_time.py [--iters N] [--warmup W]"""
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

ENV, NX, NU = "oderl-acrobot", 6, 2
H, S, B, DT = 128, 17, 4, 0.05


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True, check=True)
    name, plim = [x.strip() for x in q.stdout.strip().split(",")]
    return {"card": name, "power_limit_w": float(plim)}


def timed(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_multi_time.py needs a CUDA device")
    import neurallaplacecontrol_b200 as nlc
    from _util import weights
    from oracle.nl_model import nl_forward

    print(json.dumps(card()), flush=True)
    sd = weights(ENV, calibrated=True)
    m = nlc.NeuralLaplaceModel(NX, NU, NX, hidden_units=H, s_recon_terms=S, state_mean=np.zeros(NX), state_std=np.ones(NX),
                               action_mean=np.zeros(NU), action_std=np.ones(1), normalize=True, normalize_time=True, dt=DT,
                               device="cuda:0", math_mode="tc_split3").double()
    m.load_state_dict(sd)
    sd32 = {k: v.to("cuda", torch.float32) for k, v in sd.items()}
    names = [k for k in sd32 if k.startswith(("action_encoder", "laplace_rep_func"))]
    for K in (1024, 16384):
        for n_t in (1, 8, 64):
            g = torch.Generator().manual_seed(K + n_t)
            obs = torch.randn(K, NX, generator=g, dtype=torch.float64).cuda()
            act = torch.randn(K, B, NU, generator=g, dtype=torch.float64).cuda()
            ts = (DT * torch.cumsum(0.2 + torch.empty(K, n_t, dtype=torch.float64).exponential_(1.0, generator=g), 1)).cuda()
            gout = torch.randn(K, n_t, NX, generator=g, dtype=torch.float64).cuda()
            rep = (obs.repeat_interleave(n_t, 0), act.repeat_interleave(n_t, 0), ts.reshape(-1, 1))

            def fwd(o, a, t):
                with torch.no_grad():
                    m(o, a, t)

            def fwd_bwd(o, a, t):
                o, a = o.detach().requires_grad_(True), a.detach().requires_grad_(True)
                with torch.enable_grad():
                    out = m(o, a, t)
                    out.backward(gout.view(out.shape))

            leaves32 = [sd32[n].detach().requires_grad_(True) for n in names]
            d32 = dict(sd32)
            d32.update(zip(names, leaves32))
            o32, a32, t32, g32 = obs.float(), act.float(), ts.float(), gout.float()

            def eager(backward):
                def run():
                    o, a = o32.detach().requires_grad_(backward), a32.detach().requires_grad_(backward)
                    with torch.set_grad_enabled(backward):
                        out = nl_forward(d32, o, a, t32)
                        if backward:
                            out.backward(g32.view(out.shape))
                return run

            routes = {"multi": (obs, act, ts), "repeated": rep}
            for route, inp in routes.items():
                if route == "repeated" and n_t == 1:
                    continue
                f = timed(lambda: fwd(*inp), args.iters, args.warmup)
                fb = timed(lambda: fwd_bwd(*inp), args.iters, args.warmup)
                print(json.dumps({"K": K, "n_t": n_t, "route": route, "fwd_ms": round(f, 4), "fwd_bwd_ms": round(fb, 4)}), flush=True)
            f = timed(eager(False), args.iters, args.warmup)
            fb = timed(eager(True), args.iters, args.warmup)
            print(json.dumps({"K": K, "n_t": n_t, "route": "eager", "fwd_ms": round(f, 4), "fwd_bwd_ms": round(fb, 4)}), flush=True)
            del rep
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()

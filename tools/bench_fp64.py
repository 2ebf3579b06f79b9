"""Times NeuralLaplaceModel in math_mode="fp64" (nlc_model_forward_f64 / nlc_model_backward_f64, csrc/model_grad.cu) beside
the tc_split3 and fp32 modes, fp64 torch-eager autograd and fp64 CPU autograd.  Acrobot, hidden 128, S 17, B 4.

Prints one JSON line per measurement:
  * "device": card name, power limit, maximum SM clock and SM count, read in the same run (tools/bench_grad.py card());
  * "forward": forward without grad through the module, per mode, CUDA events;
  * "fwd_bwd": out = model(obs, act, ts); out.backward(g) through the module, per mode, CUDA events;
  * "torch_eager_fp64": the same forward + backward as fp64 torch-eager autograd of oracle.nl_forward on the same GPU;
  * "cpu_fp64": fp64 autograd of oracle.nl_forward on the CPU (the reference's setting), with the core count;
  * "train_step": forward, backward, clip_grad_norm_(0.1) and Adam at batch 16 on fp64 parameters (train_utils.py), host
    clock around synchronised steps, per mode, with the handle rebuilds the steps triggered and the rebuild share of a step.
Shapes: K in {16, 1024, 65536} at n_t = 1 and K = 16384 at n_t = 8.
usage: python tools/bench_fp64.py [--quick]"""
from __future__ import annotations

import argparse
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_grad import card, cuda_time_ms, emit  # noqa: E402  (card name, power limit and SMs read in the same run)

ENV, NX, NU = "oderl-acrobot", 6, 2
H, S, B, DT = 128, 17, 4, 0.05
SHAPES = ((16, 1), (1024, 1), (65536, 1), (16384, 8))
MODES = ("fp64", "tc_split3", "fp32")


def model(mode):
    import neurallaplacecontrol_b200 as nlc
    from _util import weights

    m = nlc.NeuralLaplaceModel(NX, NU, NX, hidden_units=H, s_recon_terms=S, state_mean=np.zeros(NX), state_std=np.ones(NX),
                               action_mean=np.zeros(NU), action_std=np.ones(1), normalize=True, normalize_time=True, dt=DT,
                               device="cuda:0", math_mode=mode).double()
    sd = weights(ENV, calibrated=True)
    m.load_state_dict(sd)
    return m, sd


def inputs(K, n_t, seed=0):
    g = torch.Generator().manual_seed(seed)
    obs = torch.randn(K, NX, generator=g, dtype=torch.float64)
    act = torch.randn(K, B, NU, generator=g, dtype=torch.float64)
    ts = DT * torch.cumsum(0.2 + torch.empty(K, n_t, dtype=torch.float64).exponential_(1.0, generator=g), dim=1)
    gout = torch.randn(K, n_t, NX, generator=g, dtype=torch.float64)
    return obs, act, ts, gout


def bench_shape(K, n_t, iters):
    from oracle.nl_model import nl_forward

    obs, act, ts, gout = inputs(K, n_t)
    oc, ac, tc = obs.cuda(), act.cuda(), ts.cuda()
    g = gout.cuda().view(K, NX) if n_t == 1 else gout.cuda()
    og, ag = oc.clone().requires_grad_(True), ac.clone().requires_grad_(True)
    for mode in MODES:
        m, _ = model(mode)

        def fwd():
            with torch.no_grad():
                m(oc, ac, tc)

        def fwd_bwd():
            with torch.enable_grad():
                m(og, ag, tc).backward(g.view(-1) if K == 1 else g)

        emit({"what": "forward", "mode": mode, "K": K, "n_t": n_t, "ms": cuda_time_ms(fwd, iters)})
        emit({"what": "fwd_bwd", "mode": mode, "K": K, "n_t": n_t, "ms": cuda_time_ms(fwd_bwd, iters)})
    _, sd = model("fp64")
    names = [k for k in sd if k.startswith(("action_encoder", "laplace_rep_func"))]
    d = {k: v.cuda() for k, v in sd.items()}
    for k in names:
        d[k].requires_grad_(True)

    def eager():
        with torch.enable_grad():
            out = nl_forward(d, og, ag, tc)
            out.backward(g.view(out.shape))

    emit({"what": "torch_eager_fp64", "K": K, "n_t": n_t, "ms": cuda_time_ms(eager, max(3, iters // 2))})


def bench_cpu(K, n_t):
    from oracle.nl_model import nl_forward

    _, sd = model("fp64")
    obs, act, ts, gout = inputs(K, n_t)
    names = [k for k in sd if k.startswith(("action_encoder", "laplace_rep_func"))]
    for k in names:
        sd[k].requires_grad_(True)
    o, a = obs.clone().requires_grad_(True), act.clone().requires_grad_(True)

    def run():
        with torch.enable_grad():
            out = nl_forward(sd, o, a, ts)
            out.backward(gout.view(out.shape))

    run()
    n = 5 if K * n_t <= 1024 else 2
    t0 = time.perf_counter()
    for _ in range(n):
        run()
    emit({"what": "cpu_fp64", "K": K, "n_t": n_t, "ms": (time.perf_counter() - t0) / n * 1e3, "cpu_count": os.cpu_count(),
          "torch_threads": torch.get_num_threads()})


def bench_train_step(mode, steps):
    m, _ = model(mode)
    obs, act, ts, _ = inputs(16 * 8, 1, seed=3)
    target = 0.1 * torch.randn(16 * 8, NX, dtype=torch.float64)
    opt = torch.optim.Adam(m.parameters(), lr=1e-4)
    batches = [(obs[i::8].cuda(), act[i::8].cuda(), ts[i::8].cuda(), target[i::8].cuda()) for i in range(8)]

    def step(i):
        s0, a0, t0, y = batches[i % 8]
        with torch.enable_grad():
            opt.zero_grad()
            loss = torch.nn.functional.mse_loss(m(s0, a0, t0), y)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(m.parameters(), 0.1)
            opt.step()

    for i in range(10):
        step(i)
    torch.cuda.synchronize()
    rebuilds, h = 0, m._handle
    t0 = time.perf_counter()
    for i in range(steps):
        step(i)
        if m._handle is not h:
            rebuilds, h = rebuilds + 1, m._handle
    torch.cuda.synchronize()
    t_step = (time.perf_counter() - t0) / steps * 1e3
    # what one rebuild costs (host repack + upload), as tools/bench_grad.py measures it
    p0 = next(m.parameters())
    t_reb = 0.0
    for _ in range(steps):
        with torch.no_grad():
            p0.add_(0.0)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        m.handle()
        torch.cuda.synchronize()
        t_reb += time.perf_counter() - t1
    t_reb = t_reb / steps * 1e3
    emit({"what": "train_step", "mode": mode, "batch": 16, "B": B, "ms": t_step, "handle_rebuilds_per_step": rebuilds / steps,
          "handle_rebuild_ms": t_reb, "handle_rebuild_share": rebuilds / steps * t_reb / t_step})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="K = 16 and 1024 only, few iterations")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fp64.py measures on a CUDA device; none is visible")
    torch.backends.cuda.matmul.allow_tf32 = False
    emit({"what": "device", **card()})
    shapes = SHAPES[:2] if args.quick else SHAPES
    for K, n_t in shapes:
        bench_shape(K, n_t, 3 if args.quick else 20)
    for K, n_t in shapes:
        bench_cpu(K, n_t)
    for mode in ("fp64", "tc_split3"):
        bench_train_step(mode, 20 if args.quick else 100)


if __name__ == "__main__":
    main()

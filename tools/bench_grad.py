"""Times the backward of NeuralLaplaceModel.forward (nlc_model_backward_ts, csrc/model_grad.cu) and a full training step.

Prints one JSON line per measurement:
  * "backward": the four backward launches alone (CUDA events around N calls of nlc_model_backward_ts);
  * "fwd_bwd": forward + backward through the module (out = model(obs, act, ts); out.backward(g)), CUDA events;
  * "torch_eager": the same forward + backward as fp32 torch-eager autograd of oracle.nl_forward on the same GPU;
  * "cpu_fp64": fp64 autograd of oracle.nl_forward on the CPU (the reference's dtype), with the core count;
  * "train_step": forward, backward, clip_grad_norm_(0.1) and Adam at batch 16 on fp64 parameters (train_utils.py), host
    clock around synchronised steps, and the share of it spent rebuilding the model handle (host repack + upload) that
    every optimizer step triggers.
FLOPs are counted from the shapes (multiply-adds x 2 of the matrix products; the backward kernel recomputes the forward,
so it counts three times the forward's products).  The FP32 peak is COMPUTED as SMs x 128 FFMA lanes x 2 x the maximum SM
clock that nvidia-smi reports for the card - a bound, not a measured rate.
usage: python tools/bench_grad.py [--quick]"""
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

ENV_SHAPE = {"oderl-acrobot": (6, 2), "oderl-cartpole": (5, 1), "oderl-pendulum": (3, 1)}
H, S, B, DT = 128, 17, 4, 0.05


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True)
    name, plim, clk = [x.strip() for x in q.stdout.strip().split(",")]
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return {"card": name, "power_limit_w": float(plim), "max_sm_clock_mhz": float(clk), "sms": sms,
            "fp32_peak_tflops_computed": sms * 128 * 2 * float(clk) * 1e6 / 1e12}


def forward_flops(nx, nu):
    """Multiply-adds x 2 of the forward's products per sample (zero-state products skipped, s-column fold included)."""
    Hg, G3, N3 = H // 2, 3 * H // 2, 2 * nx * S
    gru = 2 * (nu * G3 * B + Hg * G3 * (B - 1) + Hg * G3 * B + Hg * G3 * (B - 1)) + 2 * 2 * Hg
    mlp = 2 * (H * 2 * S + H * (nx + 2) + H * H + H * N3)
    return gru + mlp


def model_and_inputs(env, K, seed=0):
    import neurallaplacecontrol_b200 as nlc
    from _util import weights

    nx, nu = ENV_SHAPE[env]
    m = nlc.NeuralLaplaceModel(nx, nu, nx, hidden_units=H, s_recon_terms=S, state_mean=np.zeros(nx), state_std=np.ones(nx),
                               action_mean=np.zeros(nu), action_std=np.ones(1), normalize=True, normalize_time=True, dt=DT,
                               device="cuda:0", math_mode="tc_split3").double()
    sd = weights(env, calibrated=True)
    m.load_state_dict(sd)
    g = torch.Generator().manual_seed(seed)
    obs = torch.randn(K, nx, generator=g, dtype=torch.float64)
    act = torch.randn(K, B, nu, generator=g, dtype=torch.float64)
    ts = DT * (0.2 + torch.empty(K, 1, dtype=torch.float64).exponential_(1.0, generator=g))
    return m, sd, obs, act, ts


def cuda_time_ms(fn, iters):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def emit(rec):
    print(json.dumps(rec), flush=True)


def bench_kernels(env, K, peak, warm):
    from neurallaplacecontrol_b200 import _lib
    from oracle.nl_model import nl_forward

    nx, nu = ENV_SHAPE[env]
    m, sd, obs, act, ts = model_and_inputs(env, K)
    lib = _lib.load()
    o32, a32, t32 = obs.float().cuda().contiguous(), act.float().cuda().contiguous(), ts.float().cuda().reshape(-1).contiguous()
    gout = torch.randn(K, nx, device="cuda")
    h = m.handle()
    n = sum(p.numel() for p in m.parameters())
    gp, go, ga = torch.empty(n, device="cuda"), torch.empty_like(o32), torch.empty_like(a32)
    ws = torch.empty(int(lib.nlc_model_backward_workspace_bytes(h, K, B)), dtype=torch.uint8, device="cuda")

    def bwd():
        _lib.check(lib.nlc_model_backward_ts(h, o32.data_ptr(), a32.data_ptr(), t32.data_ptr(), K, B, gout.data_ptr(), gp.data_ptr(),
                                             go.data_ptr(), ga.data_ptr(), ws.data_ptr(), _lib.current_stream_ptr()), "backward")

    iters = 20 if warm else 3
    for _ in range(3 if warm else 1):
        bwd()
    t_bwd = cuda_time_ms(bwd, iters)
    flops_bwd = 3 * forward_flops(nx, nu) * K
    emit({"what": "backward", "env": env, "K": K, "B": B, "H": H, "S": S, "ms": t_bwd, "gflop": flops_bwd / 1e9,
          "tflops": flops_bwd / t_bwd / 1e9, "share_of_fp32_peak_computed": flops_bwd / t_bwd / 1e9 / peak})

    oc, ac, tc = obs.cuda().requires_grad_(True), act.cuda().requires_grad_(True), ts.cuda()
    g64 = gout.double()

    def fwd_bwd():
        with torch.enable_grad():
            out = m(oc, ac, tc)
            out.backward(g64)

    t_fb = cuda_time_ms(fwd_bwd, iters)
    flops_fb = 4 * forward_flops(nx, nu) * K
    emit({"what": "fwd_bwd", "env": env, "K": K, "ms": t_fb, "tflops": flops_fb / t_fb / 1e9,
          "share_of_fp32_peak_computed": flops_fb / t_fb / 1e9 / peak})

    names = [k for k in sd if k.startswith(("action_encoder", "laplace_rep_func"))]
    d = {k: v.float().cuda() for k, v in sd.items()}
    for k in names:
        d[k].requires_grad_(True)
    oe, ae, te = obs.float().cuda().requires_grad_(True), act.float().cuda().requires_grad_(True), ts.float().cuda()

    def eager():
        with torch.enable_grad():
            out = nl_forward(d, oe, ae, te)
            out.backward(gout.view(out.shape))

    t_e = cuda_time_ms(eager, max(3, iters // 2))
    emit({"what": "torch_eager", "env": env, "K": K, "ms": t_e, "ours_fwd_bwd_ms": t_fb, "speedup": t_e / t_fb,
          "allow_tf32": torch.backends.cuda.matmul.allow_tf32})


def bench_cpu(env, K):
    from oracle.nl_model import nl_forward

    _, sd, obs, act, ts = model_and_inputs(env, K)
    names = [k for k in sd if k.startswith(("action_encoder", "laplace_rep_func"))]
    for k in names:
        sd[k].requires_grad_(True)
    o, a = obs.clone().requires_grad_(True), act.clone().requires_grad_(True)
    g = torch.randn(K, ENV_SHAPE[env][0], dtype=torch.float64)

    def run():
        with torch.enable_grad():
            nl_forward(sd, o, a, ts).backward(g.view(-1) if K == 1 else g)

    run()
    n, t0 = 5, time.perf_counter()
    for _ in range(n):
        run()
    emit({"what": "cpu_fp64", "env": env, "K": K, "ms": (time.perf_counter() - t0) / n * 1e3, "cpu_count": os.cpu_count(),
          "torch_threads": torch.get_num_threads()})


def bench_train_step(env, steps):
    m, _, obs, act, ts = model_and_inputs(env, 16 * 8, seed=3)
    nx = ENV_SHAPE[env][0]
    target = 0.1 * torch.randn(16 * 8, nx, dtype=torch.float64)
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
    t0 = time.perf_counter()
    for i in range(steps):
        step(i)
    torch.cuda.synchronize()
    t_step = (time.perf_counter() - t0) / steps * 1e3
    p0 = next(m.parameters())
    t_reb = 0.0
    for _ in range(steps):
        with torch.no_grad():
            p0.add_(0.0)  # a new parameter version, as every optimizer step makes
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        m.handle()
        torch.cuda.synchronize()
        t_reb += time.perf_counter() - t1
    t_reb = t_reb / steps * 1e3
    emit({"what": "train_step", "env": env, "batch": 16, "B": B, "ms": t_step, "handle_rebuild_ms": t_reb,
          "handle_rebuild_share": t_reb / t_step})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="K = 16 and 1024 only, few iterations")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_grad.py measures on a CUDA device; none is visible")
    torch.backends.cuda.matmul.allow_tf32 = False  # fp32 baseline, as torch's default
    info = card()
    emit({"what": "device", **info})
    Ks = (16, 1024) if args.quick else (16, 1024, 65536)
    for env in ENV_SHAPE:
        for K in Ks:
            bench_kernels(env, K, info["fp32_peak_tflops_computed"], warm=not args.quick)
    for K in (16, 1024):
        bench_cpu("oderl-acrobot", K)
    bench_train_step("oderl-acrobot", 20 if args.quick else 100)


if __name__ == "__main__":
    main()

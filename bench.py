#!/usr/bin/env python
"""Benchmark of the MPPI / Neural Laplace planning hot path (BASELINE.json metric: model rollout-steps/s and
per-control-step plan latency).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload cfg4|cfg3|cfg1]
                    [--scaling strong|weak] [--no-extra] [--no-cpu-baseline] [--dump-outputs DIR]

One "step" = one MPPI control step (``MPPIDelay.command``): K x H Neural Laplace rollout-steps.

Headline at every N: BASELINE config 4 as north_star names it - acrobot-delay, K = 65536 samples, H = 50 - with the K
samples SHARDED over the N GPUs (``"scaling": "strong"``; 8192 samples per GPU at N = 8) and one exchange of the
(beta, eta, W) triple per control step.  At N > 1 the same run also measures the weak-scaled step (every GPU plans the
named K, K_total = N x 65536) and reports it under ``"weak"``, and checks OUTSIDE the timed region that the sharded
plan returns the unsharded plan's U and action (``"sharded_vs_unsharded"``).  Synthetic inputs: random-init weights of
the reference architecture (golden fixture, calibrated phi-bias), on-device Philox action noise keyed on the global
sample index.

* ``value``    - device-timed (CUDA events), state / action buffer already resident in HBM.
* ``e2e``      - the same control step through the drop-in ``MPPIDelay.command(state, action_buffer)`` with HOST buffers:
                 host->device copies of the inputs and the device->host read of the action inside the timing.
* ``roofline`` - the dominant kernel (history encoder) timed ALONE with CUDA events (L2 flushed): hoisted FLOPs / duration
                 against the measured BURST bf16 tensor peak of MEASURED_PEAKS.json; ``in_step`` holds the same kernels
                 timed inside one control step (events between the stages, ``nlc_planner_step_profile``) against the
                 sustained peak.
* ``cpu_baseline`` / ``--impl reference`` - the CPU oracle port of the reference path (fp64 as the reference runs, and
                 fp32; all host threads) on a bounded sample of the same workload.
* ``extra``    - (N = 1) the other BASELINE configs in the same run: config 1 and 3 plans (latency, fill factor), the
                 config 2 Fourier-ILT microbenchmark (GB/s against the measured HBM peak, S = 33 / 65 / 129) and config 5
                 (32 closed-loop instances per GPU, instance-batched).

``--dump-outputs DIR`` writes, after the headline's timed steps (``value``, then ``e2e``), what the last of them left the
caller (``dump_outputs``) as ``DIR/<name>.npy``.  The inputs depend on the arguments only, so two builds run with the
same arguments can be compared array by array.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    # name: (env, K, H, description)
    "cfg1": ("oderl-pendulum", 1000, 20, "oderl Pendulum-delay MPPI K=1000 H=20"),
    "cfg3": ("oderl-cartpole", 8192, 30, "oderl Cartpole-delay MPPI K=8192 H=30"),
    "cfg4": ("oderl-acrobot", 65536, 50, "oderl Acrobot-delay MPPI K=65536 H=50"),
}
START_STATE = {
    "oderl-pendulum": [-1.0, 1.2246467991473532e-16, 1.0],
    "oderl-cartpole": [0.0, 0.0, -1.0, 1.2246467991473532e-16, 0.0],
    "oderl-acrobot": [1.0, 0.0, 1.0, 0.0, 0.0, 0.0],
}
# algorithmic work per rollout-step, FLOP = 2 MAC, "hoisted minimum" (SURVEY 8d / BASELINE.md 4)
HOISTED_FLOP = {"oderl-pendulum": 307712, "oderl-cartpole": 325632, "oderl-acrobot": 336128}
ENCODER_FLOP = 2 * 10 * 192 * 64  # ten 64x192 products per window: the hoisted GRU work (+ a 2x64 output layer)
METRIC, UNIT = "mppi_rollout_steps_per_sec", "rollout-steps/s"
N_SM = 148
DUMP_SAMPLES = 4096  # per-sample trajectories kept by --dump-outputs: all of config 4's would be 130 MB


def load_peaks():
    """Measured peaks of this pool's B200s (driver-written MEASURED_PEAKS.json), else the fallback the profiling recipe
    states.  A file that cannot be read or lacks a key falls back key by key rather than failing the bench."""
    fb = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    d = {}
    if os.path.isfile(path):
        try:
            with open(path) as f:
                d = json.load(f)
        except (OSError, ValueError):
            d = {}

    def num(key, default):
        try:
            v = float(d.get(key))
            return v if v > 0 else default
        except (TypeError, ValueError):
            return default

    burst = num("bf16_tflops", fb["bf16_tflops"])
    measured = all(k in d for k in ("hbm_gbs", "bf16_tflops"))
    return {"hbm_gbs": num("hbm_gbs", fb["hbm_gbs"]), "bf16_tflops": burst,
            "bf16_tflops_sustained": num("bf16_tflops_sustained", burst if measured else fb["bf16_tflops_sustained"]),
            "source": "measured" if measured else "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_inputs(env):
    import numpy as np
    import torch

    from _util import DT, S_TERMS, weights
    from oracle import costs

    nx, nu = costs.ENV_DIMS[env]
    return {"nx": nx, "nu": nu, "ah": float(costs.ENV_ACT_HIGH[env]), "sd": weights(env, calibrated=True), "dt": DT, "S": S_TERMS,
            "state": np.array(START_STATE[env], dtype=np.float64), "buffer": torch.zeros(4, nu, dtype=torch.float64)}


# ------------------------------------------------------------------------------------------------------------------
# CPU legs (the oracle port: the one place besides tests/ and smoke() that executes oracle/)
# ------------------------------------------------------------------------------------------------------------------
def cpu_plan_rate(env, K, H, Ks, dtype, n_warm, n_steps, budget_s=None):
    """rollout-steps/s of the oracle port of ``MPPIDelay.command`` on ``Ks`` of the K samples, all host threads."""
    import torch

    from oracle import costs, mppi

    torch.set_grad_enabled(False)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    inp = build_inputs(env)
    nu, ah = inp["nu"], inp["ah"]
    sd = {k: v.to(dtype) for k, v in inp["sd"].items()}
    dyn, cost = mppi.make_nl_dynamics(sd, inp["dt"]), costs.running_cost(env)
    sig = mppi.noise_sigma_for(nu, dtype=dtype)
    chol = torch.linalg.cholesky(sig)
    U = torch.zeros(H, nu, dtype=dtype)
    state, buf = torch.from_numpy(inp["state"]).to(dtype), inp["buffer"].to(dtype)
    g = torch.Generator().manual_seed(1)
    times, t_start = [], time.perf_counter()
    for it in range(n_warm + n_steps):
        noise = torch.randn(Ks, H, nu, generator=g, dtype=dtype) @ chol.T
        t0 = time.perf_counter()
        out = mppi.command(U, state, buf, noise, dyn, cost, noise_sigma=sig, u_scale=ah, u_min=-ah, u_max=ah)
        dt_ = time.perf_counter() - t0
        U = out["U"]
        if it >= n_warm:
            times.append(dt_)
        if budget_s is not None and times and time.perf_counter() - t_start > budget_s:
            break
    t = sum(times) / len(times)
    return Ks * H / t, 1e3 * t, len(times), cores


def run_reference(args, env, K, H, desc):
    """CPU arm: the oracle port of the reference's PyTorch CPU path, fp64 as the reference runs it (plus an fp32 leg),
    all host threads; each step = ``--cpu-samples`` of the K samples (the whole K when it fits the time box)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    Ks = K if K * H <= 300_000 else min(K, args.cpu_samples)
    sample = (f"{Ks} of the {K} samples x H={H} per step" if Ks < K else f"all {K} samples x H={H} per step") + \
        ", fp64, oracle port of the reference path (the reference classes need torchlaplace / gym: not installable)"
    val, ms, n, cores = cpu_plan_rate(env, K, H, Ks, __import__("torch").float64, args.warmup, args.steps)
    val32, ms32, _, _ = cpu_plan_rate(env, K, H, Ks, __import__("torch").float32, 1, max(2, min(args.steps, 5)))
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": desc, "K": K, "H": H, "env": env, "sample": sample, "samples_per_step": Ks,
                       "plan_latency_ms_full_K_extrapolated": ms * K / Ks},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "fp32": {"value": val32, "ms_per_step": ms32}},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def cpu_baseline(env, K, H, cpu_samples):
    import torch

    Ks = K if K * H <= 300_000 else min(K, cpu_samples)
    val, ms, n, cores = cpu_plan_rate(env, K, H, Ks, torch.float64, 1, 6, budget_s=18.0)
    val32, ms32, n32, _ = cpu_plan_rate(env, K, H, Ks, torch.float32, 1, 4, budget_s=8.0)
    return {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n} control steps of {Ks} of the {K} samples x H={H}, fp64 oracle port, {cores} threads",
            "plan_latency_ms_sample": ms, "fp32": {"value": val32, "plan_latency_ms_sample": ms32, "steps": n32}}


# ------------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------------
class Ctx:
    """Process-wide state of the GPU arm: device, process group, timing helpers."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        self.torch, self.dist, self.args = torch, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.group = None
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
            self.group = dist.group.WORLD
        from neurallaplacecontrol_b200 import _lib

        self._lib = _lib
        self.lib = _lib.load()
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps, warmup, collective=True):
        """(device ms per step, wall ms per step, launches) - L2 flushed before every timed step (outside its span), barrier +
        synchronize on both sides, max over ranks."""
        torch = self.torch
        idle = float(getattr(self.args, "idle", 0.0) or 0.0)
        if idle > 0:
            # every timed region starts from the same power state: on this pool's power-capped B200s a region measured right
            # after another runs ~10 % slower (tools/diag_e2e.py: the same call 3.55 ms first, 3.93 ms after three other loops,
            # 3.49 ms again after 2 s of idle), which otherwise shows up as a difference BETWEEN the numbers of one line
            torch.cuda.synchronize()
            time.sleep(idle)
        for _ in range(warmup):
            fn()
        self.barrier() if collective else torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        wall = []
        launches0 = self.lib.nlc_launch_count()
        for s, e in ev:
            self.flush.fill_(1)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            s.record()
            fn()
            e.record()
            e.synchronize()
            wall.append(time.perf_counter() - t0)
        launches = self.lib.nlc_launch_count() - launches0
        self.barrier() if collective else torch.cuda.synchronize()
        t = torch.tensor([sum(s.elapsed_time(e) for s, e in ev), 1e3 * sum(wall)], dtype=torch.float64, device=self.dev)
        if collective and self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t[0]) / steps, float(t[1]) / steps, launches


def make_planner(ctx, env, K, H, group=None, seed=1234, math=None, S=None, **kw):
    import numpy as np
    import torch

    import neurallaplacecontrol_b200 as nlc

    inp = build_inputs(env)
    nx, nu, ah = inp["nx"], inp["nu"], inp["ah"]
    math = math or ctx.args.math
    if S is not None and S != inp["S"]:
        torch.manual_seed(0)  # another number of Fourier terms: the module's own random init (no fixture of that shape)
    model = nlc.NeuralLaplaceModel(nx, nu, nx, hidden_units=128, s_recon_terms=S or inp["S"], state_mean=np.zeros(nx),
                                   state_std=np.ones(nx), action_mean=np.array([0] * nu), action_std=np.array([1.0]),
                                   normalize=True, normalize_time=True, dt=inp["dt"], device=ctx.dev, math_mode=math).double()
    if S is not None and S != inp["S"]:
        with torch.no_grad():  # keep the Fourier sum in a trained model's operating range (cf. oracle/gen_golden.py calibrate_)
            last = model.laplace_rep_func.linear_tanh_stack[4]
            last.weight.mul_(0.05)
            last.bias.mul_(0.05)
            last.bias[nx * S:].sub_(3.0)
    else:
        model.load_state_dict(inp["sd"])
    planner = nlc.MPPIDelay(nlc.NLDynamics(model, inp["dt"]), nlc.EnvRunningCost(env), nx, nlc.noise_sigma_for(nu), num_samples=K,
                            horizon=H, device=ctx.dev, lambda_=1.0, u_min=torch.tensor(-ah), u_max=torch.tensor(ah), u_scale=ah,
                            U_init=torch.zeros(H, nu, dtype=torch.float64), process_group=group, seed=seed, math_mode=math, **kw)
    return inp, model, planner


def time_plan(ctx, env, K, H, group, steps, warmup, S=None, math=None):
    """Device-timed and end-to-end control step of one workload; returns a dict and the live objects."""
    torch = ctx.torch
    inp, model, planner = make_planner(ctx, env, K, H, group=group, S=S, math=math)
    state_dev = torch.tensor(inp["state"], dtype=torch.float64, device=ctx.dev)
    buf_dev = inp["buffer"].to(ctx.dev)
    # `value`: the control step on inputs already resident in the planner's device buffers - one graph launch per step
    # (MPPIDelay.step); shards without the device-side exchange go through command() with device tensors
    planner.set_inputs(state_dev, buf_dev)
    resident = planner.G == 1 or planner._exchange
    ms_dev, _, launches = ctx.timed(planner.step if resident else (lambda: planner.command(state_dev, buf_dev)), steps, warmup)

    def e2e_step():
        a = planner.command(inp["state"], inp["buffer"])  # host buffers in
        # one shard / device-connected shards: the C entry point already synchronised and left the action on the host;
        # shards exchanging through NCCL: read it back here
        return planner.last_action_host if planner.last_action_host is not None else a.cpu()

    _, ms_e2e, _ = ctx.timed(e2e_step, steps, warmup)
    return {"ms_dev": ms_dev, "ms_e2e": ms_e2e, "launches": launches, "inp": inp, "model": model, "planner": planner,
            "state_dev": state_dev, "buf_dev": buf_dev}


def dump_outputs(out_dir, planner):
    """What the planner's last control step left its caller, as float32 ``out_dir/<name>.npy``: the action, the updated plan
    ``U``, every sample's ``cost_total`` and ``omega``, and ``states``, ``perturbed_action`` and ``noise`` of DUMP_SAMPLES
    samples drawn with a fixed seed.  Sharded plans: this rank's samples."""
    import numpy as np
    import torch

    from neurallaplacecontrol_b200 import _lib

    torch.cuda.synchronize()
    Kl = planner.K_local
    rows = np.sort(np.random.default_rng(0).choice(Kl, size=min(DUMP_SAMPLES, Kl), replace=False))
    rows = torch.from_numpy(rows).to(planner.d)
    out = {"action": planner._buf(_lib.BUF_ACTION, (planner.nu,)), "U": planner.U, "cost_total": planner.cost_total,
           "omega": planner.omega, "states": planner.states[rows], "perturbed_action": planner.perturbed_action[rows],
           "noise": planner.noise[rows]}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def kernels_alone(ctx, r, env, H, steps):
    """The two hot kernels of the step, each timed ALONE (own launch, L2 flushed) on the planner's buffers."""
    _lib, lib, torch = ctx._lib, ctx.lib, ctx.torch
    planner, model, inp = r["planner"], r["model"], r["inp"]
    nx, nu = inp["nx"], inp["nu"]
    Kl, B = planner.K_local, 4
    hist = planner._buf(_lib.BUF_HIST, (Kl, B - 1 + H, nu))
    pbuf = planner._buf(_lib.BUF_P, (Kl, H, 2))
    mh = model.set_prediction_time(inp["dt"])
    mode = _lib.MATH_MODES[ctx.args.math]

    def enc():
        _lib.check(lib.nlc_encode_history(mh, hist.data_ptr(), Kl, H, B, pbuf.data_ptr(), mode, _lib.current_stream_ptr()))

    ms_enc, _, _ = ctx.timed(enc, max(3, steps), 2)
    ro = _lib.RolloutOpts()
    ro.env, ro.state_constraint, ro.goal_x, ro.dynamics, ro.delay, ro.dt = _lib.ENV_IDS[env], 0, 0.0, 0, 0, inp["dt"]
    st32 = r["state_dev"].float().contiguous()
    cost_buf = planner._buf(_lib.BUF_COST_TOTAL, (Kl,))
    states_buf = planner._buf(_lib.BUF_STATES, (Kl, H, nx))

    def roll():
        _lib.check(lib.nlc_rollout_cost(mh, C.byref(ro), st32.data_ptr(), 0, pbuf.data_ptr(), hist.data_ptr(), None, Kl, H, B, nu,
                                        cost_buf.data_ptr(), states_buf.data_ptr(), mode, _lib.current_stream_ptr()))

    ms_roll, _, _ = ctx.timed(roll, max(3, steps), 2)
    return ms_enc, ms_roll


def in_step_split(ctx, r, steps):
    """The stages timed INSIDE one control step (direct launches, events at the stage boundaries): median over ``steps``."""
    _lib, lib, torch = ctx._lib, ctx.lib, ctx.torch
    planner = r["planner"]
    if planner.G != 1:
        return None
    planner.command(r["state_dev"], r["buf_dev"])  # inputs into the planner's own buffers
    out = (C.c_float * 6)()
    rows = []
    for _ in range(max(3, steps)):
        ctx.flush.fill_(1)
        torch.cuda.synchronize()
        _lib.check(lib.nlc_planner_step_profile(planner._handle, out, _lib.current_stream_ptr()), "nlc_planner_step_profile")
        rows.append([float(out[i]) for i in range(6)])
    med = [statistics.median(col) for col in zip(*rows)]
    d = dict(zip(("perturb_ms", "encoder_ms", "rollout_ms", "softmax_update_ms", "encoder_and_rollout_ms"), med))
    d["encoder_beside_rollout"] = bool(med[5])
    return d


def roofline_block(ctx, env, K_local, H, ms_enc, ms_roll, split, ms_step, clocks, peaks, workload):
    args = ctx.args
    nx, S = {"oderl-pendulum": 3, "oderl-cartpole": 5, "oderl-acrobot": 6}[env], 17
    enc_flop = ENCODER_FLOP * K_local * H
    roll_flop = (HOISTED_FLOP[env] - ENCODER_FLOP) * K_local * H
    pp = (K_local + 127) // 128 > N_SM  # the library's own choice: the ping-pong form (two tiles per CTA) beyond one wave
    roll_name = "rollout_nl_kernel" if args.math == "fp32" else ("rollout_pp_kernel" if pp else "rollout_tc2_kernel")
    kernels = {"encoder": {"name": "encode_gru_kernel" if args.math == "fp32" else "encode_tc2_kernel", "ms": ms_enc, "flop": enc_flop},
               "rollout": {"name": roll_name, "ms": ms_roll, "flop": roll_flop}}
    dom = max(kernels, key=lambda k: kernels[k]["ms"])
    # MMA FLOPs the tensor pipe executes per algorithmic FLOP: 3 fp16 products per fp32-class product in tc_split3
    issue_mult = {"tc_split3": 3.0, "tc_fp16": 1.0, "fp32": 0.0}[args.math]
    burst, sustained = peaks["bf16_tflops"], peaks["bf16_tflops_sustained"]
    sm_hz = 1e6 * ((clocks or {}).get("sm_mhz") or 1965.0)
    mufu_peak = 15.9 * N_SM * sm_hz  # tools/mufu_bench.cu: 15.9 MUFU results /clk/SM
    per_step_mufu = {"encoder": 8 * 64 * (4 if args.math == "tc_split3" else 3), "rollout": 2 * 128 + nx * S * 4}
    for name, kv in kernels.items():
        kv["tflops"] = kv["flop"] / (kv["ms"] * 1e-3) / 1e12
        kv["frac"] = kv["tflops"] / burst  # timed alone: the burst peak applies
        kv["issued_tflops"] = issue_mult * kv["tflops"]
        kv["issued_frac"] = kv["issued_tflops"] / burst
        if args.math != "fp32":
            kv["mufu_per_s"] = per_step_mufu[name] * K_local * H / (kv["ms"] * 1e-3)
            kv["mufu_frac"] = kv["mufu_per_s"] / mufu_peak
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get(f"{kernels[dom]['name']}_{args.math}_{workload}")
    achieved = kernels[dom]["tflops"]
    block = {"bound": "tensor", "kernel": kernels[dom]["name"], "achieved": achieved, "peak": burst, "unit": "TFLOP/s",
             "frac": achieved / burst, "issued_frac": kernels[dom]["issued_frac"], "traffic": traffic,
             "peak_source": peaks["source"], "peak_kind": "burst (kernel timed alone)", "kernel_ms": kernels[dom]["ms"],
             "flop_per_launch": kernels[dom]["flop"], "kernels": kernels,
             "whole_step": {"achieved": HOISTED_FLOP[env] * K_local * H / (ms_step * 1e-3) / 1e12, "peak": sustained,
                            "peak_kind": "sustained (kernels back to back inside the step)"},
             "note": "frac = algorithmic (hoisted) FLOPs per launch / CUDA-event time / measured bf16 tensor TFLOP/s.  tc_split3 issues 3 "
                     "fp16 MMAs per algorithmic product (fp32-class result), so frac <= 1/3 by construction; issued_frac counts the MMA "
                     "FLOPs the tensor pipe executes.  Both hot kernels are co-limited by the MUFU pipe (mufu_frac): DESIGN.md 3."}
    block["whole_step"]["frac"] = block["whole_step"]["achieved"] / sustained
    if split:
        block["in_step"] = dict(split)
        for key, name in (("encoder_ms", "encoder"), ("rollout_ms", "rollout")):
            tf = kernels[name]["flop"] / (split[key] * 1e-3) / 1e12
            block["in_step"][name + "_tflops"] = tf
            block["in_step"][name + "_frac_sustained"] = tf / sustained
    return block


def sharded_vs_unsharded(ctx, env, K, H):
    """Outside every timed region: one control step of the K-sharded plan against the same plan on ONE GPU (rank 0).
    The sampler is keyed on the global sample index, so both draw the same noise; only stage 4's summation order differs."""
    torch, dist = ctx.torch, ctx.dist
    inp, _, sharded = make_planner(ctx, env, K, H, group=ctx.group, seed=99)
    state_dev = torch.tensor(inp["state"], dtype=torch.float64, device=ctx.dev)
    buf_dev = inp["buffer"].to(ctx.dev)
    a_sh = sharded.command(state_dev, buf_dev).double()
    U_sh = sharded.U.double().clone()
    res = torch.zeros(3, dtype=torch.float64, device=ctx.dev)
    if ctx.rank == 0:
        # the whole plan through the same rollout kernel form as the shards (a 65536-sample plan would pick the ping-pong
        # form on its own: same arithmetic, other summation order), so that per-sample costs are bit-identical and the
        # comparison isolates what sharding changes: the order of stage 4's sums
        pp_shard = (sharded.K_local + 127) // 128 >= 89  # (the overlapped step's own choice: rollout.cu rollout_overlap_is_ping_pong)
        os.environ["NLC_ROLLOUT_TILES"] = "3" if pp_shard else "1"
        _, _, whole = make_planner(ctx, env, K, H, group=None, seed=99)
        a1 = whole.command(state_dev, buf_dev).double()
        torch.cuda.synchronize()
        del os.environ["NLC_ROLLOUT_TILES"]
        U1 = whole.U.double()
        scale = max(float(U1.abs().max()), 1e-30)
        res[0] = (U1 - U_sh).abs().max() / scale
        res[1] = (a1 - a_sh).abs().max() / (scale * inp["ah"])
    # every rank holds the same U bit for bit (no broadcast is ever needed)
    Umax, Umin = U_sh.clone(), U_sh.clone()
    dist.all_reduce(Umax, op=dist.ReduceOp.MAX)
    dist.all_reduce(Umin, op=dist.ReduceOp.MIN)
    res[2] = (Umax - Umin).abs().max()
    dist.broadcast(res, src=0)
    out = {"U_relerr": float(res[0]), "action_relerr": float(res[1]), "U_spread_over_ranks": float(res[2]), "tolerance": 1e-5}
    if not (out["U_relerr"] <= 1e-5 and out["action_relerr"] <= 1e-5 and out["U_spread_over_ranks"] == 0.0):
        raise SystemExit(f"sharded plan differs from the unsharded plan: {out}")
    return out


# ---- extras (N = 1): the other BASELINE configs -------------------------------------------------------------------------
def extra_plan(ctx, name, peaks, S=None, math=None):
    env, K, H, desc = WORKLOADS[name]
    r = time_plan(ctx, env, K, H, None, max(5, ctx.args.steps), 3, S=S, math=math)
    tiles = (K + 127) // 128
    split = in_step_split(ctx, r, ctx.args.steps)
    if math is not None:
        # the single-pass fp16 tensor-core mode: ONE MMA per product and tanh.approx gates - north_star's "stated looser bound"
        # path (tests/test_gpu_parity.py::test_full_size_plan_fp16_mode_stated_bound: 5e-2 over the whole horizon, measured 1-3e-2
        # on trajectories and U at this shape, against 1e-4 / ~1e-5 for the default fp32-class mode)
        flop = HOISTED_FLOP[env] * K * H
        return {"workload": f"{desc}, math={math} (looser stated bound: 5e-2 over the horizon, measured 1-3e-2; the default mode holds 1e-4)", "in_step": split,
                "ms_per_step": r["ms_dev"], "plan_latency_ms_e2e": r["ms_e2e"], "value": K * H / (r["ms_dev"] * 1e-3),
                "e2e_value": K * H / (r["ms_e2e"] * 1e-3), "unit": UNIT, "math": math,
                "frac_of_sustained_peak": flop / (r["ms_dev"] * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"]}
    if S is not None:
        # the reference CLASS default number of Fourier terms (w_nl.py:73; config.py runs S = 17): 396 (theta, phi) columns for the
        # acrobot - the one-tile rollout with L3 in two column halves and W3 streamed half by half by TMA, whatever the plan size
        return {"workload": f"{desc}, S={S} Fourier terms (reference class default), random-init weights", "in_step": split,
                "ms_per_step": r["ms_dev"], "plan_latency_ms_e2e": r["ms_e2e"], "value": K * H / (r["ms_dev"] * 1e-3),
                "e2e_value": K * H / (r["ms_e2e"] * 1e-3), "unit": UNIT, "rollout_form": "one tile per CTA, W3 streamed by TMA bulk copies",
                "math": ctx.args.math}
    return {"workload": desc, "in_step": split, "ms_per_step": r["ms_dev"], "plan_latency_ms_e2e": r["ms_e2e"], "value": K * H / (r["ms_dev"] * 1e-3),
            "e2e_value": K * H / (r["ms_e2e"] * 1e-3), "unit": UNIT, "tiles_of_128": tiles, "sm_fill": min(1.0, tiles / N_SM),
            "frac_of_sustained_peak": HOISTED_FLOP[env] * K * H / (r["ms_dev"] * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"],
            "math": ctx.args.math, "note": "latency-bound: the horizon is sequential and the plan fills sm_fill of the SMs"}


def extra_ilt(ctx, peaks, N=1_000_000, n_t=100):
    """BASELINE config 2: complex64 F (N, n_t, S), t_j = (j+1) 0.05, out fp32 (N, n_t); 8 S + 8 algorithmic bytes per point."""
    torch = ctx.torch
    from neurallaplacecontrol_b200 import fourier_ilt
    from oracle import ilt

    out_rows = []
    t = (torch.arange(n_t, dtype=torch.float32, device=ctx.dev) + 1) * 0.05
    for S in (33, 65, 129):
        need = N * n_t * (8 * S + 4) + (4 << 30)
        free, _ = torch.cuda.mem_get_info(ctx.dev)
        if need > free:
            out_rows.append({"S": S, "skipped": f"needs {need / 1e9:.0f} GB, {free / 1e9:.0f} GB free"})
            continue
        g = torch.Generator(device=ctx.dev).manual_seed(2)
        F = torch.empty((N, n_t, S, 2), dtype=torch.float32, device=ctx.dev)
        for i in range(0, N, 100_000):  # U(-1,1), chunked to bound the temporaries
            F[i:i + 100_000].uniform_(-1, 1, generator=g)
        Fc = torch.view_as_complex(F)
        out = torch.empty((N, n_t), dtype=torch.float32, device=ctx.dev)
        for _ in range(3):
            fourier_ilt(Fc, t, out=out)
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(5)]
        for s, e in ev:  # the input (>= 26 GB) is far larger than L2: no flush needed
            s.record(); fourier_ilt(Fc, t, out=out); e.record()
        torch.cuda.synchronize()
        ms = sum(s.elapsed_time(e) for s, e in ev) / len(ev)
        nbytes = N * n_t * (8 * S + 8)
        idx = torch.randint(0, N, (64,), device=ctx.dev)
        Fs = Fc[idx].cpu()
        t64 = t.cpu().double().expand(64, n_t)
        ref = ilt.fourier_line_integrate(Fs.real.double(), Fs.imag.double(), t64, ilt.SCALE * (t64 + ilt.EPS))
        err = float((ref - out[idx].cpu().double()).abs().max() / ref.abs().max())
        Ns = 10000
        Fcpu = Fc[:Ns].cpu()
        tc = t.cpu().double().expand(Ns, n_t)
        torch.set_num_threads(os.cpu_count() or 1)
        t0 = time.perf_counter()
        ilt.fourier_line_integrate(Fcpu.real.double(), Fcpu.imag.double(), tc, ilt.SCALE * (tc + ilt.EPS))
        cpu_s = time.perf_counter() - t0
        gbs = nbytes / (ms * 1e-3) / 1e9
        out_rows.append({"S": S, "ms": ms, "points_per_s": N * n_t / (ms * 1e-3),
                         "roofline": {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                      "frac": gbs / peaks["hbm_gbs"], "bytes_per_point": 8 * S + 8},
                         "relerr_vs_oracle_sample": err,
                         "cpu_baseline": {"points_per_s": Ns * n_t / cpu_s, "cores": os.cpu_count(), "kind": "port",
                                          "sample": f"{Ns} trajectories, fp64"}})
        del F, Fc, out
        torch.cuda.empty_cache()
    return {"workload": f"ILT microbench: Fourier-series inverse Laplace, {N} trajectories x {n_t} time points, complex64", "kernel": "ilt_rows_kernel",
            "rows": out_rows}


def extra_cfg5(ctx, instances=32, K=4096, H=30, steps=10, warmup=3, delay=1):
    """BASELINE config 5, one GPU's share: ``instances`` env x seed instances in closed loop, instance-batched per env."""
    import numpy as np

    import neurallaplacecontrol_b200 as nlc
    from _util import DT, S_TERMS, weights
    from oracle import costs

    torch, dev = ctx.torch, ctx.dev
    envs = ["oderl-pendulum", "oderl-cartpole", "oderl-acrobot"]
    batches = []
    for ei, e in enumerate(envs):
        ids = [i for i in range(instances) if i % 3 == ei]
        if not ids:
            continue
        nx, nu = costs.ENV_DIMS[e]
        ah = costs.ENV_ACT_HIGH[e]
        m = nlc.NeuralLaplaceModel(nx, nu, nx, hidden_units=128, s_recon_terms=S_TERMS, state_mean=np.zeros(nx), state_std=np.ones(nx),
                                   action_mean=np.array([0] * nu), action_std=np.array([1.0]), normalize=True, normalize_time=True,
                                   dt=DT, device=dev, math_mode=ctx.args.math).double()
        m.load_state_dict(weights(e, calibrated=True))
        bp = nlc.BatchedMPPIDelay(nlc.NLDynamics(m, DT), nlc.EnvRunningCost(e), nx, nlc.noise_sigma_for(nu), len(ids), seeds=ids,
                                  num_samples=K, horizon=H, device=dev, u_min=torch.tensor(-ah), u_max=torch.tensor(ah), u_scale=ah,
                                  math_mode=ctx.args.math)
        st = torch.stack([torch.tensor(np.array(START_STATE[e]) + np.random.default_rng(gi).uniform(-0.05, 0.05, nx), dtype=torch.float32)
                          for gi in ids]).to(dev).contiguous()
        batches.append({"env": e, "planner": bp, "states": st, "bufs": torch.zeros(len(ids), 4, nu, device=dev),
                        "reward": torch.zeros(len(ids), device=dev), "stream": torch.cuda.Stream(device=dev)})

    def control_step():
        for b in batches:
            with torch.cuda.stream(b["stream"]):
                a = b["planner"].command(b["states"], b["bufs"])
                nlc.env_step(b["env"], b["states"], b["bufs"], a.float().contiguous(), delay, DT, b["reward"])
        for b in batches:
            b["stream"].synchronize()

    for _ in range(warmup):
        control_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        control_step()
    torch.cuda.synchronize()
    dt_ = (time.perf_counter() - t0) / steps
    ok = all(bool(torch.isfinite(b["states"]).all()) for b in batches)
    return {"workload": f"batched closed-loop eval, one GPU's share: {instances} env x seed instances x MPPI K={K} H={H} (256 over 8 GPUs, "
                        "instance-sharded, no collective)", "ms_per_control_step_all_instances": 1e3 * dt_,
            "value": instances * K * H / dt_, "unit": UNIT, "instances": instances, "closed_loop": True, "states_finite": ok,
            "timing": "wall clock around command + env_step of all instances, synchronised", "math": ctx.args.math}


def run_gpu(args, env, K, H, desc):
    ctx = Ctx(args)
    torch = ctx.torch
    torch.set_grad_enabled(False)
    world, rank = ctx.world, ctx.rank
    K_head = K if args.scaling == "strong" else K * world
    sampler = ClockSampler(ctx.local)
    if rank == 0:
        sampler.start()
    head = time_plan(ctx, env, K_head, H, ctx.group, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, head["planner"])  # before kernels_alone reuses the planner's buffers
    ms_enc, ms_roll = kernels_alone(ctx, head, env, H, args.steps)
    split = in_step_split(ctx, head, args.steps)
    other = None
    check = None
    if world > 1:
        # the other scaling mode in the same run, and the equivalence of the sharded plan with the unsharded one
        K_other = K * world if args.scaling == "strong" else K
        o = time_plan(ctx, env, K_other, H, ctx.group, args.steps, args.warmup)
        other = {"scaling": "weak" if args.scaling == "strong" else "strong", "K_total": K_other, "K_per_gpu": K_other // world,
                 "ms_per_step": o["ms_dev"], "value": K_other * H / (o["ms_dev"] * 1e-3), "unit": UNIT,
                 "e2e_value": K_other * H / (o["ms_e2e"] * 1e-3)}
        del o
        check = sharded_vs_unsharded(ctx, env, K, H)
    if rank == 0:
        peaks = load_peaks()
        inp, planner = head["inp"], head["planner"]
        nx, nu = inp["nx"], inp["nu"]
        Kl = planner.K_local
        steps_per_plan = K_head * H
        value = steps_per_plan / (head["ms_dev"] * 1e-3)
        e2e = steps_per_plan / (head["ms_e2e"] * 1e-3)
        pp = (Kl + 127) // 128 > N_SM
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": head["ms_dev"], "plan_latency_ms": head["ms_dev"], "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": desc if K_head == K else desc.replace(f"K={K}", f"K={K_head} ({K} per GPU x {world})"),
                       "env": env, "K": K_head, "H": H, "S": inp["S"], "hidden": 128, "history_window": 4,
                       "parallelism": f"K-sharded x{world}", "K_per_gpu": Kl, "tiles_per_gpu": (Kl + 127) // 128,
                       "sm_fill": min(1.0, ((Kl + 127) // 128) / N_SM),
                       "rollout_form": "ping-pong, 2 tiles per CTA" if pp else "1 tile per CTA", "math": args.math,
                       "noise": "on-device Philox4x32-10", "l2": "flushed between timed steps (256 MiB fill)", "keep_states": True,
                       "idle_before_each_timed_region_s": args.idle},
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": UNIT, "ms_per_step": head["ms_e2e"], "h2d_bytes_per_step": 4 * (nx + 4 * nu) * world,
                    "d2h_bytes_per_step": 4 * nu * world},
            "gpu_launches": head["launches"] * world,
            "roofline": roofline_block(ctx, env, Kl, H, ms_enc, ms_roll, split, head["ms_dev"], clocks, peaks, args.workload),
        }
        if other:
            line[other["scaling"]] = other
        if check:
            line["sharded_vs_unsharded"] = check
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(env, K, H, args.cpu_samples)
    del head
    torch.cuda.empty_cache()
    if world == 1 and not args.no_extra:
        peaks = load_peaks()
        extra = []
        for fn in (lambda: extra_plan(ctx, "cfg3", peaks), lambda: extra_plan(ctx, "cfg1", peaks), lambda: extra_cfg5(ctx),
                   lambda: extra_ilt(ctx, peaks), lambda: extra_plan(ctx, "cfg4", peaks, S=33)) + \
                  (() if args.math == "tc_fp16" else (lambda: extra_plan(ctx, "cfg4", peaks, math="tc_fp16"),)):
            try:
                extra.append(fn())
            except Exception as exc:  # an extra must never take the headline line down
                extra.append({"error": f"{type(exc).__name__}: {exc}"})
            torch.cuda.empty_cache()
        line["extra"] = extra
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        ctx.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg4", choices=sorted(WORKLOADS))
    ap.add_argument("--math", default="tc_split3", choices=["fp32", "tc_split3", "tc_fp16"])
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"],
                    help="strong (default): the named K sharded N ways - north_star's config 4; weak: every GPU plans the named K")
    ap.add_argument("--cpu-samples", type=int, default=8192, help="samples per CPU step when the whole K does not fit the time box")
    ap.add_argument("--idle", type=float, default=1.0, help="seconds of idle before every timed region (equal power state for every number of the line)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the config 1/2/3/5 extras (N = 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the headline's last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU arm's outputs (--impl b200)")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    env, K, H, desc = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, env, K, H, desc)
    else:
        run_gpu(args, env, K, H, desc)


if __name__ == "__main__":
    main()

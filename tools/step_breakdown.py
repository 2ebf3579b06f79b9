#!/usr/bin/env python
"""Where one control step's time goes IN SITU: CUDA events between the stage-level C-ABI calls of a config-4 step
(perturb -> encode -> rollout -> softmax -> combine), L2 flushed before each step as bench.py does."""
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
    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    env, K, H, B = "oderl-acrobot", 65536, 50, 4
    nx, nu = costs.ENV_DIMS[env]
    ah = float(costs.ENV_ACT_HIGH[env])
    model = nlc.NeuralLaplaceModel(nx, nu, nx, hidden_units=128, s_recon_terms=S_TERMS, state_mean=np.zeros(nx), state_std=np.ones(nx),
                                   action_mean=np.array([0] * nu), action_std=np.array([1.0]), normalize=True, normalize_time=True,
                                   dt=DT, device=dev).double()
    model.load_state_dict(weights(env, calibrated=True))
    planner = nlc.MPPIDelay(nlc.NLDynamics(model, DT), nlc.EnvRunningCost(env), nx, nlc.noise_sigma_for(nu), num_samples=K, horizon=H,
                            device=dev, u_min=torch.tensor(-ah), u_max=torch.tensor(ah), u_scale=ah,
                            U_init=torch.zeros(H, nu, dtype=torch.float64), seed=1, math_mode="tc_split3")
    state = torch.tensor([1.0, 0, 1, 0, 0, 0], dtype=torch.float64, device=dev)
    buf = torch.zeros(B, nu, dtype=torch.float64, device=dev)
    planner.command(state, buf)  # creates the handle and buffers
    lib, h = _lib.load(), planner._handle
    d, mh = planner._desc(B, K, 0, K, 1, 0), planner._model_handle()
    mp, ro, mode = d.mppi, d.rollout, d.math_mode
    g = lambda which, shape: planner._buf(which, shape)  # noqa: E731
    U, noise, pert, hist = g(_lib.BUF_U, (H, nu)), g(_lib.BUF_NOISE, (K, H, nu)), g(_lib.BUF_PERTURBED, (K, H, nu)), g(_lib.BUF_HIST, (K, B - 1 + H, nu))
    acts, p, cost, w, states = g(_lib.BUF_ACTIONS, (K, H, nu)), g(_lib.BUF_P, (K, H, 2)), g(_lib.BUF_COST_TOTAL, (K,)), g(_lib.BUF_WEIGHTS, (K,)), g(_lib.BUF_STATES, (K, H, nx))
    triple, action, stats = g(_lib.BUF_TRIPLE, (2 + H * nu,)), g(_lib.BUF_ACTION, (nu,)), g(_lib.BUF_STATS, (2,))
    U2 = torch.zeros_like(U)
    pc = torch.zeros(K, device=dev)
    ws = torch.zeros(int(lib.nlc_softmax_workspace_bytes(K, H * nu)) // 4 + 64, device=dev)
    st32, ab32 = state.float().contiguous(), buf.float().contiguous()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    s = _lib.current_stream_ptr()
    names = ["perturb", "encode", "rollout", "softmax_partial", "combine"]
    acc = {n: [] for n in names}
    for it in range(8):
        flush.fill_(1)
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
        ev[0].record()
        _lib.check(lib.nlc_perturb(C.byref(mp), U.data_ptr(), U2.data_ptr(), 1, None, 1, it, ab32.data_ptr(), pert.data_ptr(), noise.data_ptr(),
                                   hist.data_ptr(), acts.data_ptr(), pc.data_ptr(), s)); ev[1].record()
        _lib.check(lib.nlc_encode_history(mh, hist.data_ptr(), K, H, B, p.data_ptr(), mode, s)); ev[2].record()
        _lib.check(lib.nlc_rollout_cost(mh, C.byref(ro), st32.data_ptr(), 0, p.data_ptr(), hist.data_ptr(), pc.data_ptr(), K, H, B, nu,
                                        cost.data_ptr(), states.data_ptr(), mode, s)); ev[3].record()
        _lib.check(lib.nlc_softmax_partial(cost.data_ptr(), noise.data_ptr(), K, H, nu, 1.0, triple.data_ptr(), w.data_ptr(), ws.data_ptr(), s)); ev[4].record()
        _lib.check(lib.nlc_softmax_combine(triple.data_ptr(), 1, H, nu, 1.0, ah, U2.data_ptr(), action.data_ptr(), stats.data_ptr(), s)); ev[5].record()
        torch.cuda.synchronize()
        if it >= 3:
            for i, n in enumerate(names):
                acc[n].append(ev[i].elapsed_time(ev[i + 1]))
    out = {n: round(float(np.median(v)), 4) for n, v in acc.items()}
    out["sum_ms"] = round(sum(out.values()), 4)
    print(json.dumps(out))


if __name__ == "__main__":
    main()

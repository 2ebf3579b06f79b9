#!/usr/bin/env python
"""Timeline of the rollout kernel's first CTA (clock64 per warp at the phase boundaries), the one-tile form of
rollout_tc2.cu (forced here with NLC_ROLLOUT_TILES=1); the ping-pong form has its own tool, trace_rollout_pp.py.
Measurement tool only."""
import ctypes as C
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

EV = ["A1 written", "M1 done", "E1 done", "M2 done", "E2 done", "M3(a) done", "E3a done", "M3b done"]


def main():
    os.environ["NLC_ROLLOUT_TILES"] = "1"
    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    env = "oderl-acrobot"
    nx, nu = costs.ENV_DIMS[env]
    model = nlc.NeuralLaplaceModel(nx, nu, nx, hidden_units=128, s_recon_terms=S_TERMS, state_mean=np.zeros(nx), state_std=np.ones(nx),
                                   action_mean=np.array([0] * nu), action_std=np.array([1.0]), normalize=True, normalize_time=True,
                                   dt=DT, device=dev).double()
    model.load_state_dict(weights(env, calibrated=True))
    mh = model.set_prediction_time(DT)
    lib = _lib.load()
    lib.nlc_debug_set_rollout_trace.argtypes = [C.c_void_p]
    lib.nlc_debug_set_rollout_trace.restype = None
    K, H, B = int(os.environ.get("K", 65536)), 50, 4
    hist = torch.randn(K, B - 1 + H, nu, device=dev, dtype=torch.float32)
    p = torch.empty(K, H, 2, device=dev, dtype=torch.float32)
    mode = _lib.MATH_MODES["tc_split3"]
    _lib.check(lib.nlc_encode_history(mh, hist.data_ptr(), K, H, B, p.data_ptr(), mode, _lib.current_stream_ptr()))
    st = torch.tensor([1.0, 0.0, 1.0, 0.0, 0.0, 0.0], dtype=torch.float32, device=dev)
    ro = _lib.RolloutOpts()
    ro.env, ro.state_constraint, ro.goal_x, ro.dynamics, ro.delay, ro.dt = _lib.ENV_IDS[env], 0, 0.0, 0, 0, DT
    cost = torch.empty(K, device=dev, dtype=torch.float32)
    states = torch.empty(K, H, nx, device=dev, dtype=torch.float32)
    trace = torch.zeros(104 * 16 * 8, dtype=torch.int64, device=dev)
    lib.nlc_debug_set_rollout_trace(trace.data_ptr())
    for _ in range(2):
        _lib.check(lib.nlc_rollout_cost(mh, C.byref(ro), st.data_ptr(), 0, p.data_ptr(), hist.data_ptr(), None, K, H, B, nu,
                                        cost.data_ptr(), states.data_ptr(), mode, _lib.current_stream_ptr()))
    torch.cuda.synchronize()
    tr = trace.cpu().numpy().reshape(104, 16, 8).astype(np.int64)
    print("per event min/median/max over the 16 warps, clocks relative to the step's first A1")
    for s in (4, 5, 6, 7, 24, 25, 26, 27, 28):
        row = []
        for e in range(8):
            v = tr[s, :, e]
            v = v[v > 0]
            row.append("-" if len(v) == 0 else f"{v.min() - tr[s, :, 0].min():6d}/{int(np.median(v)) - tr[s, :, 0].min():6d}/{v.max() - tr[s, :, 0].min():6d}")
        print(f" step {s:2d} | " + " | ".join(row))
    last = max(e for e in range(8) if (tr[:, :, e] > 0).any())  # the step's last product: M3 (resident W3) or M3b (streamed)
    st = [int(tr[s_, :, 0].min()) for s_ in range(104)]
    tails = [int(np.median(tr[s_ + 1, :, 0])) - int(np.median(tr[s_, :, last])) for s_ in range(103)]
    print("tail (last product done -> next A1 written) (k clk):", [round(x / 1e3, 1) for x in tails])
    print("step durations (k clk):", [round((st[i + 1] - st[i]) / 1e3, 1) for i in range(103)])
    print("events:", ", ".join(f"{i}={n}" for i, n in enumerate(EV)))


if __name__ == "__main__":
    main()

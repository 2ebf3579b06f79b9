"""ctypes binding of ``libnlc_b200.so`` (C ABI declared in ``include/nlc_b200.h``).

There is no CPU fallback: if the shared library is missing, ``load()`` raises, and every compute
entry point of the library returns ``NLC_ERR_ARCH`` (raised here as ``RuntimeError``) when no
sm_100 device is present.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC_DIR = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libnlc_b200.so")

NLC_OK = 0
ENV_IDS = {"oderl-pendulum": 0, "oderl-cartpole": 1, "oderl-acrobot": 2}
ENV_DIMS = {"oderl-pendulum": (3, 1), "oderl-cartpole": (5, 1), "oderl-acrobot": (6, 2)}
DYN_NEURAL_LAPLACE, DYN_ANALYTIC_DELAY = 0, 1
MATH_MODES = {"fp32": 0, "tc_split3": 1, "tc_fp16": 2}

(BUF_U, BUF_NOISE, BUF_PERTURBED, BUF_COST_TOTAL, BUF_WEIGHTS, BUF_STATES, BUF_ACTIONS, BUF_TRIPLE, BUF_ALL_TRIPLES,
 BUF_ACTION, BUF_STATS, BUF_HIST, BUF_P, BUF_STATE, BUF_ACTION_BUFFER) = range(15)

_dp = C.POINTER(C.c_double)
_fp = C.c_void_p  # device float pointers travel as integers


class ModelDesc(C.Structure):
    _fields_ = [
        ("state_dim", C.c_int32), ("action_dim", C.c_int32), ("hidden_units", C.c_int32), ("s_terms", C.c_int32),
        ("encode_obs_time", C.c_int32), ("normalize", C.c_int32), ("normalize_time", C.c_int32),
        ("action_std_len", C.c_int32), ("dt", C.c_double),
        ("state_mean", _dp), ("state_std", _dp), ("action_mean", _dp), ("action_std", _dp),
        ("gru_w_ih_l0", _dp), ("gru_w_hh_l0", _dp), ("gru_b_ih_l0", _dp), ("gru_b_hh_l0", _dp),
        ("gru_w_ih_l1", _dp), ("gru_w_hh_l1", _dp), ("gru_b_ih_l1", _dp), ("gru_b_hh_l1", _dp),
        ("enc_out_w", _dp), ("enc_out_b", _dp),
        ("mlp_w0", _dp), ("mlp_b0", _dp), ("mlp_w2", _dp), ("mlp_b2", _dp), ("mlp_w4", _dp), ("mlp_b4", _dp),
    ]


class MppiParams(C.Structure):
    _fields_ = [
        ("K", C.c_int32), ("T", C.c_int32), ("nu", C.c_int32), ("B", C.c_int32),
        ("k_offset", C.c_int64), ("k_total", C.c_int64),
        ("lambda_", C.c_float), ("u_scale", C.c_float),
        ("has_bounds", C.c_int32), ("u_min", C.c_float * 4), ("u_max", C.c_float * 4),
        ("sample_null_action", C.c_int32), ("noise_abs_cost", C.c_int32),
        ("sigma_inv", C.c_float * 16), ("sigma_chol", C.c_float * 16), ("noise_mu", C.c_float * 4),
        ("u_init", C.c_float * 4),
    ]


class RolloutOpts(C.Structure):
    _fields_ = [("env", C.c_int32), ("state_constraint", C.c_int32), ("goal_x", C.c_float), ("dynamics", C.c_int32),
                ("delay", C.c_int32), ("dt", C.c_float)]


class PlannerDesc(C.Structure):
    _fields_ = [("mppi", MppiParams), ("rollout", RolloutOpts), ("nx", C.c_int32), ("n_shards", C.c_int32),
                ("shard_index", C.c_int32), ("math_mode", C.c_int32), ("keep_states", C.c_int32), ("seed", C.c_uint64)]


class PlannerF64Desc(C.Structure):
    """``nlc_planner_f64_desc``: the fp32 planner's descriptor for shapes and flags, and the fp64 values beside it."""
    _fields_ = [("base", PlannerDesc), ("lambda_", C.c_double), ("u_scale", C.c_double), ("dt", C.c_double), ("goal_x", C.c_double),
                ("u_min", C.c_double * 4), ("u_max", C.c_double * 4), ("sigma_inv", C.c_double * 16),
                ("sigma_chol", C.c_double * 16), ("noise_mu", C.c_double * 4), ("u_init", C.c_double * 4)]


# name -> (restype, argtypes); also the list the CPU test checks against include/nlc_b200.h
SIGNATURES = {
    "nlc_last_error": (C.c_char_p, []),
    "nlc_version": (C.c_int, []),
    "nlc_device_check": (C.c_int, [C.c_int]),
    "nlc_launch_count": (C.c_uint64, []),
    "nlc_model_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(ModelDesc), C.c_int]),
    "nlc_model_destroy": (C.c_int, [C.c_void_p]),
    "nlc_model_set_prediction_time": (C.c_int, [C.c_void_p, C.c_double]),
    "nlc_model_forward": (C.c_int, [C.c_void_p, _fp, _fp, C.c_int, C.c_int, _fp, _fp, C.c_int, C.c_void_p]),
    "nlc_model_forward_ts": (C.c_int, [C.c_void_p, _fp, _fp, _fp, C.c_int, C.c_int, _fp, _fp, C.c_int, C.c_void_p]),
    "nlc_model_grad_floats": (C.c_int64, [C.POINTER(ModelDesc)]),
    "nlc_model_backward_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_int, C.c_int]),
    "nlc_model_backward_ts": (C.c_int, [C.c_void_p, _fp, _fp, _fp, C.c_int, C.c_int, _fp, _fp, _fp, _fp, C.c_void_p, C.c_void_p]),
    "nlc_model_forward_multi_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "nlc_model_forward_multi": (C.c_int, [C.c_void_p, _fp, _fp, _fp, C.c_int, C.c_int, C.c_int, _fp, _fp, C.c_void_p, C.c_int,
                                          C.c_void_p]),
    "nlc_model_backward_multi_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "nlc_model_backward_multi": (C.c_int, [C.c_void_p, _fp, _fp, _fp, C.c_int, C.c_int, C.c_int, _fp, _fp, _fp, _fp, C.c_void_p,
                                           C.c_void_p]),
    "nlc_model_forward_f64_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "nlc_model_forward_f64": (C.c_int, [C.c_void_p, _fp, _fp, _fp, _fp, C.c_int, C.c_int, C.c_int, _fp, _fp, C.c_void_p, C.c_void_p]),
    "nlc_model_backward_f64_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "nlc_model_backward_f64": (C.c_int, [C.c_void_p, _fp, _fp, _fp, _fp, C.c_int, C.c_int, C.c_int, _fp, _fp, _fp, _fp, C.c_void_p,
                                         C.c_void_p]),
    "nlc_encode_history": (C.c_int, [C.c_void_p, _fp, C.c_int, C.c_int, C.c_int, _fp, C.c_int, C.c_void_p]),
    "nlc_perturb": (C.c_int, [C.POINTER(MppiParams), _fp, _fp, C.c_int, _fp, C.c_uint64, C.c_uint64, _fp, _fp, _fp,
                              _fp, _fp, _fp, C.c_void_p]),
    "nlc_rollout_cost": (C.c_int, [C.c_void_p, C.POINTER(RolloutOpts), _fp, C.c_int, _fp, _fp, _fp, C.c_int, C.c_int,
                                   C.c_int, C.c_int, _fp, _fp, C.c_int, C.c_void_p]),
    "nlc_softmax_workspace_bytes": (C.c_int64, [C.c_int, C.c_int]),
    "nlc_softmax_partial": (C.c_int, [_fp, _fp, C.c_int, C.c_int, C.c_int, C.c_float, _fp, _fp, C.c_void_p,
                                      C.c_void_p]),
    "nlc_softmax_combine": (C.c_int, [_fp, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, _fp, _fp, _fp,
                                      C.c_void_p]),
    "nlc_planner_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.POINTER(PlannerDesc), C.c_int]),
    "nlc_planner_destroy": (C.c_int, [C.c_void_p]),
    "nlc_planner_set_U": (C.c_int, [C.c_void_p, _dp]),
    "nlc_planner_get_U": (C.c_int, [C.c_void_p, _dp]),
    "nlc_planner_buffer": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "nlc_planner_rollout": (C.c_int, [C.c_void_p, _fp, C.c_int, _fp, _fp, C.c_void_p]),
    "nlc_planner_finish": (C.c_int, [C.c_void_p, C.c_void_p]),
    "nlc_planner_step": (C.c_int, [C.c_void_p, C.c_void_p]),
    "nlc_planner_step_profile": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.c_void_p]),
    "nlc_planner_overlap_status": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "nlc_debug_overlap_plan": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_longlong)]),
    "nlc_planner_exchange_export": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "nlc_planner_exchange_connect": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "nlc_planner_exchange_status": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "nlc_planner_command_host": (C.c_int, [C.c_void_p, _dp, _dp, _fp, _dp, C.c_void_p]),
    "nlc_planner_f64_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.POINTER(PlannerF64Desc), C.c_int]),
    "nlc_planner_f64_destroy": (C.c_int, [C.c_void_p]),
    "nlc_planner_f64_set_params": (C.c_int, [C.c_void_p, _fp, C.c_void_p]),
    "nlc_planner_f64_set_U": (C.c_int, [C.c_void_p, _dp]),
    "nlc_planner_f64_get_U": (C.c_int, [C.c_void_p, _dp]),
    "nlc_planner_f64_buffer": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "nlc_planner_f64_command": (C.c_int, [C.c_void_p, _fp, C.c_int, _fp, _fp, C.c_void_p]),
    "nlc_planner_f64_command_host": (C.c_int, [C.c_void_p, _dp, _dp, _dp, C.c_void_p]),
    "nlc_batch_planner_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.POINTER(PlannerDesc), C.c_int,
                                           C.POINTER(C.c_uint64), C.c_int]),
    "nlc_batch_planner_destroy": (C.c_int, [C.c_void_p]),
    "nlc_batch_planner_set_U": (C.c_int, [C.c_void_p, _dp]),
    "nlc_batch_planner_buffer": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "nlc_batch_planner_command": (C.c_int, [C.c_void_p, _fp, _fp, _fp, _fp, C.c_void_p]),
    "nlc_env_step": (C.c_int, [C.POINTER(RolloutOpts), _fp, _fp, _fp, C.c_int, C.c_int, C.c_int, _fp, C.c_void_p]),
    "nlc_ilt_fourier": (C.c_int, [_fp, _fp, C.c_int, C.c_int64, C.c_int, C.c_int, _fp, C.c_void_p]),
    "nlc_selftest_umma_gemm_ts": (C.c_int, [_fp, _fp, C.c_int, C.c_int, C.c_int, C.c_int, _fp, C.c_void_p]),
    "nlc_selftest_umma_gemm": (C.c_int, [_fp, _fp, C.c_int, C.c_int, C.c_int, C.c_int, _fp, C.c_void_p]),
}

_lib = None


def build(verbose: bool = False) -> str:
    """Compile ``libnlc_b200.so`` in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
    proc = subprocess.run(["make", "-C", CSRC_DIR, "-j", str(os.cpu_count() or 4)], capture_output=True, text=True)
    if verbose or proc.returncode != 0:
        print(proc.stdout[-4000:])
        print(proc.stderr[-4000:])
    if proc.returncode != 0:
        raise RuntimeError("building libnlc_b200.so failed (see output above)")
    return LIB_PATH


def load():
    """Load the shared library (once) and declare every prototype of ``include/nlc_b200.h``."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` or "
            f"`make -C {CSRC_DIR}`.  neurallaplacecontrol_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != NLC_OK:
        msg = load().nlc_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libnlc_b200 {what} failed ({rc}): {msg}")


def ptr(t):
    """Device (or host) address of a torch tensor, 0 for None.  Tensors must be contiguous."""
    if t is None:
        return None
    if not t.is_contiguous():
        raise ValueError("libnlc_b200 needs contiguous tensors")
    return t.data_ptr()


def current_stream_ptr():
    """cudaStream_t of torch's current stream on the current device, as an integer."""
    import torch

    raw = getattr(torch._C, "_cuda_getCurrentRawStream", None)  # one C call (torch.cuda.current_stream builds a Stream object: ~6 us)
    if raw is not None:
        return raw(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


def as_double_array(x):
    """numpy/torch/sequence -> (ctypes double array, keep-alive ndarray)."""
    import numpy as np

    arr = np.ascontiguousarray(np.asarray(x, dtype=np.float64).reshape(-1))
    return arr.ctypes.data_as(_dp), arr

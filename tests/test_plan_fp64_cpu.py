"""CPU-side checks of the fp64 planner (``nlc_planner_f64_*``): the descriptor's ctypes mirror, no CPU fallback, and the
numpy statement of its on-device sampler (the transform stated in ``include/nlc_b200.h``), which the GPU tests compare the
kernel's noise against."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle.philox import philox4x32_10

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def uniform53(hi, lo):
    """(2 ((hi >> 6) 2^26 + (lo >> 6)) + 1) 2^-53: odd multiples of 2^-53 in (0, 1), exact in fp64."""
    m = (hi.astype(np.uint64) >> np.uint64(6)) << np.uint64(26) | (lo.astype(np.uint64) >> np.uint64(6))
    return (2 * m + 1).astype(np.float64) * 2.0 ** -53


def f64_noise(K, T, nu, seed, call_index, chol, mu):
    """noise (K, T, nu) of the fp64 planner's sampler for (seed, call index)."""
    idx = np.arange(K, dtype=np.uint64)[:, None] * np.uint64(T) + np.arange(T, dtype=np.uint64)[None, :]
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32)
    z = np.zeros((K, T, 4))
    for b in range(2 if nu > 2 else 1):
        ctr = np.zeros((K, T, 4), dtype=np.uint32)
        ctr[..., 0] = (idx & np.uint64(0xFFFFFFFF)).astype(np.uint32)
        ctr[..., 1] = (idx >> np.uint64(32)).astype(np.uint32)
        ctr[..., 2] = np.uint32(call_index & 0xFFFFFFFF)
        ctr[..., 3] = np.uint32(((call_index >> 32) & 0xFFFFFFFF) ^ (0x80000000 if b else 0))
        x = philox4x32_10(ctr, key)
        u1, u2 = uniform53(x[..., 0], x[..., 1]), uniform53(x[..., 2], x[..., 3])
        r = np.sqrt(-2.0 * np.log(u1))
        z[..., 2 * b], z[..., 2 * b + 1] = r * np.cos(2 * np.pi * u2), r * np.sin(2 * np.pi * u2)
    return np.asarray(mu, dtype=np.float64) + z[..., :nu] @ np.asarray(chol, dtype=np.float64).T


def test_desc_layout_matches_header():
    from neurallaplacecontrol_b200 import _lib

    prog = '#include <stdio.h>\n#include "nlc_b200.h"\nint main(){printf("%zu\\n", sizeof(nlc_planner_f64_desc));return 0;}\n'
    exe = os.path.join(ROOT, "tests", "_sizes_f64.out")
    try:
        subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.join(ROOT, "include"), "-o", exe], input=prog.encode(), check=True)
        got = int(subprocess.run([exe], capture_output=True, check=True).stdout)
    finally:
        if os.path.exists(exe):
            os.remove(exe)
    assert got == C.sizeof(_lib.PlannerF64Desc)


def test_uniforms_stay_inside_the_open_interval():
    ext = np.array([0, 1, 63, 64, 0xFFFFFFC0, 0xFFFFFFFF], dtype=np.uint32)
    hi, lo = np.meshgrid(ext, ext)
    u = uniform53(hi.ravel(), lo.ravel())
    assert u.min() == 2.0 ** -53 and u.max() == 1.0 - 2.0 ** -53
    assert np.isfinite(np.log(u)).all() and (np.log(u) < 0).all()
    z = f64_noise(64, 16, 2, seed=3, call_index=0, chol=np.linalg.cholesky([[1.0, 0.5], [0.5, 1.0]]), mu=[0.0, 0.0])
    assert np.isfinite(z).all() and abs(z.mean()) < 0.2 and abs(z.std() - 1.0) < 0.1


def test_sampler_statement_draws_fresh_blocks():
    chol, mu = np.eye(4), np.zeros(4)
    a = f64_noise(8, 5, 4, seed=1, call_index=0, chol=chol, mu=mu)
    b = f64_noise(8, 5, 4, seed=1, call_index=1, chol=chol, mu=mu)
    assert not np.array_equal(a, b) and not np.array_equal(a[..., :2], a[..., 2:])
    np.testing.assert_array_equal(f64_noise(8, 5, 2, seed=1, call_index=0, chol=np.eye(2), mu=np.zeros(2)), a[..., :2])


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_f64_entry_points_have_no_cpu_path():
    import neurallaplacecontrol_b200 as nlc
    from neurallaplacecontrol_b200 import _lib

    lib = _lib.load()
    h = C.c_void_p()
    d = _lib.PlannerF64Desc()
    assert lib.nlc_planner_f64_create(C.byref(h), None, C.byref(d), 0) == -3  # NLC_ERR_ARCH
    assert lib.nlc_planner_f64_destroy(None) == 0
    m = nlc.NeuralLaplaceModel(3, 1, 3, hidden_units=128, s_recon_terms=17, state_mean=np.zeros(3), state_std=np.ones(3),
                               action_mean=np.zeros(1), action_std=np.ones(1), normalize=True, normalize_time=True).double()
    with pytest.raises(RuntimeError):
        nlc.MPPIDelay(nlc.NLDynamics(m), nlc.EnvRunningCost("oderl-pendulum"), 3, nlc.noise_sigma_for(1), math_mode="fp64")


def test_null_arguments_are_rejected():
    from neurallaplacecontrol_b200 import _lib

    lib = _lib.load()
    assert lib.nlc_planner_f64_create(None, None, None, 0) == -1
    assert lib.nlc_planner_f64_set_params(None, None, None) == -1
    assert lib.nlc_planner_f64_command(None, None, 0, None, None, None) == -1
    assert lib.nlc_planner_f64_command_host(None, None, None, None, None) == -1

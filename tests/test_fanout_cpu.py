"""Host-side argument checks of the many-model batch planner and the per-instance-delay env steps
(``nlc_batch_planner_create_multi``, ``nlc_env_step_delays``, ``nlc_env_step_f64_delays``) and of ``BatchedMPPIDelay``'s
sequence of dynamics handles: all run before any CUDA call, so they are checked without a device."""
import ctypes as C

import numpy as np
import pytest
import torch

NLC_ERR_ARG, NLC_ERR_SHAPE, NLC_ERR_ARCH, NLC_ERR_CUDA = -1, -2, -3, -4
# stand-in device addresses: every call below is refused by its host-side checks before anything is dereferenced
FAKE = 0x10000


def _load():
    from neurallaplacecontrol_b200 import _lib

    return _lib, _lib.load()


def _desc(_lib, dynamics, delay=0, B=4):
    d = _lib.PlannerDesc()
    d.mppi.K, d.mppi.T, d.mppi.nu, d.mppi.B, d.mppi.lambda_ = 64, 5, 1, B, 1.0
    d.rollout.env, d.rollout.dynamics, d.rollout.delay, d.rollout.dt = 0, dynamics, delay, 0.05
    d.nx, d.n_shards = 3, 1
    return d


def _create(lib, _lib, models, delays, d, I):
    h = C.c_void_p()
    seeds = (C.c_uint64 * I)(*range(I))
    m = None if models is None else (C.c_void_p * I)(*models)
    dl = None if delays is None else (C.c_int32 * I)(*delays)
    return lib.nlc_batch_planner_create_multi(C.byref(h), m, dl, C.byref(d), I, seeds, 0)


def test_batch_planner_create_multi_argument_checks():
    _lib, lib = _load()
    an, nl = _desc(_lib, _lib.DYN_ANALYTIC_DELAY), _desc(_lib, _lib.DYN_NEURAL_LAPLACE)
    h = C.c_void_p()
    seeds = (C.c_uint64 * 2)(0, 1)
    assert lib.nlc_batch_planner_create_multi(None, None, None, C.byref(an), 2, seeds, 0) == NLC_ERR_ARG
    assert lib.nlc_batch_planner_create_multi(C.byref(h), None, None, C.byref(an), 2, None, 0) == NLC_ERR_ARG
    assert lib.nlc_batch_planner_create_multi(C.byref(h), None, None, C.byref(an), 0, seeds, 0) == NLC_ERR_ARG
    assert _create(lib, _lib, None, [0, 4, 1, 2], an, 4) == NLC_ERR_ARG             # delay outside the 4-entry buffer
    assert b"instance 1 has delay 4" in lib.nlc_last_error()
    assert _create(lib, _lib, None, [0, 1, -1, 2], an, 4) == NLC_ERR_ARG
    assert _create(lib, _lib, None, None, _desc(_lib, _lib.DYN_ANALYTIC_DELAY, delay=5), 4) == NLC_ERR_ARG
    assert _create(lib, _lib, None, None, nl, 4) == NLC_ERR_ARG                      # Neural Laplace without models
    assert _create(lib, _lib, [FAKE, FAKE, None, FAKE], None, nl, 4) == NLC_ERR_ARG  # mixed: instance 2 has no model
    assert b"instance 2" in lib.nlc_last_error()
    assert _create(lib, _lib, [None, FAKE, None, None], [0, 1, 2, 3], an, 4) == NLC_ERR_ARG  # mixed: analytic with a model
    bad_shape = _desc(_lib, _lib.DYN_ANALYTIC_DELAY, B=9)
    assert _create(lib, _lib, None, None, bad_shape, 4) == NLC_ERR_SHAPE
    odd_k = _desc(_lib, _lib.DYN_ANALYTIC_DELAY)
    odd_k.mppi.K = 63
    assert _create(lib, _lib, None, None, odd_k, 4) == NLC_ERR_SHAPE
    # the single-model entry point is this call: its checks are the same
    assert lib.nlc_batch_planner_create(C.byref(h), None, C.byref(nl), 2, seeds, 0) == NLC_ERR_ARG
    assert lib.nlc_batch_planner_create(C.byref(h), None, C.byref(an), 0, seeds, 0) == NLC_ERR_ARG


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_batch_planner_create_multi_valid_arguments_need_a_device():
    _lib, lib = _load()
    an = _desc(_lib, _lib.DYN_ANALYTIC_DELAY)
    assert _create(lib, _lib, None, [0, 1, 2, 3], an, 4) == NLC_ERR_ARCH
    assert _create(lib, _lib, [None] * 4, [3, 3, 0, 0], an, 4) == NLC_ERR_ARCH


def test_env_step_delays_argument_checks():
    _lib, lib = _load()
    ro = _lib.RolloutOpts()
    ro.env, ro.dynamics, ro.dt = 0, _lib.DYN_ANALYTIC_DELAY, 0.05

    def f32(o=C.byref(ro), delays=FAKE, status=FAKE, I=2, B=4, nu=1, state=FAKE):
        return lib.nlc_env_step_delays(o, delays, state, FAKE, FAKE, I, B, nu, None, status, None)

    def f64(env=0, delays=FAKE, status=FAKE, I=2, B=4, nu=1, state=FAKE):
        return lib.nlc_env_step_f64_delays(env, delays, 0.05, state, FAKE, FAKE, I, B, nu, None, status, None)

    for fn in (f32, f64):
        assert fn(delays=None) == NLC_ERR_ARG
        assert fn(status=None) == NLC_ERR_ARG  # per-instance delays are checked on the device: the status word is required
        assert fn(state=None) == NLC_ERR_ARG
        assert fn(I=0) == NLC_ERR_ARG
        assert fn(B=9) == NLC_ERR_ARG
        assert fn(nu=2) == NLC_ERR_SHAPE
    assert f32(o=None) == NLC_ERR_ARG
    assert f64(env=3) == NLC_ERR_ARG
    ro.env = 7
    assert f32() == NLC_ERR_ARG


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_env_step_delays_valid_arguments_need_a_device():
    _lib, lib = _load()
    ro = _lib.RolloutOpts()
    ro.env, ro.dynamics, ro.delay, ro.dt = 2, _lib.DYN_ANALYTIC_DELAY, 99, 0.05  # o->delay is not read with per-instance delays
    # past the argument checks the first CUDA call (the current device) fails without a device
    assert lib.nlc_env_step_delays(C.byref(ro), FAKE, FAKE, FAKE, FAKE, 2, 4, 2, None, FAKE, None) in (NLC_ERR_ARCH, NLC_ERR_CUDA)
    assert lib.nlc_env_step_f64_delays(1, FAKE, 0.05, FAKE, FAKE, FAKE, 2, 4, 1, None, FAKE, None) in (NLC_ERR_ARCH, NLC_ERR_CUDA)


def test_batched_planner_rejects_bad_dynamics_sequences():
    """BatchedMPPIDelay's checks of a sequence of dynamics handles run before any planner object or device handle exists."""
    import neurallaplacecontrol_b200 as nlc

    def model(nx, nu):
        return nlc.NeuralLaplaceModel(nx, nu, nx, hidden_units=128, s_recon_terms=17, state_mean=np.zeros(nx), state_std=np.ones(nx),
                                      action_mean=np.zeros(nu), action_std=np.ones(1), normalize=True, normalize_time=True)

    env, nx, nu, I = "oderl-pendulum", 3, 1, 4
    m = model(nx, nu)
    nl, an = nlc.NLDynamics(m, 0.05), nlc.AnalyticDelayDynamics(env, 1, 0.05)
    cost, sig = nlc.EnvRunningCost(env), nlc.noise_sigma_for(nu)
    cases = [
        (ValueError, [nl] * (I + 1)),
        (TypeError, [nl, an, nl, nl]),
        (ValueError, [nl, nlc.NLDynamics(model(6, 2), 0.05), nl, nl]),
        (ValueError, [nl, nlc.NLDynamics(m, 0.02), nl, nl]),
        (ValueError, [an, an, nlc.AnalyticDelayDynamics(env, 4, 0.05), an]),
        (ValueError, [an, nlc.AnalyticDelayDynamics("oderl-acrobot", 1, 0.05), an, an]),
    ]
    for exc, dyns in cases:
        with pytest.raises(exc):
            nlc.BatchedMPPIDelay(dyns, cost, nx, sig, I, num_samples=64, horizon=5)
    with pytest.raises(ValueError):  # a delay inside a larger action buffer is fine; outside the given size it is not
        nlc.BatchedMPPIDelay([an, an, nlc.AnalyticDelayDynamics(env, 2, 0.05), an], cost, nx, sig, I, num_samples=64, horizon=5,
                             action_buffer_size=2)

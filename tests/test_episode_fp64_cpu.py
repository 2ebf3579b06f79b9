"""CPU-side checks of the fp64 environment step: ``nlc_env_step_f64`` checks its arguments before any CUDA call, and
``env_step`` rejects tensors it has no kernel for before it reaches the library."""
import ctypes as C

import pytest
import torch


def test_env_step_f64_rejects_bad_arguments():
    from neurallaplacecontrol_b200 import _lib

    lib = _lib.load()
    host = (C.c_double * 64)()  # never read: every call below fails its argument checks first
    p = C.addressof(host)

    def call(env=0, delay=1, I=2, B=4, nu=1, state=p, buf=p, action=p):
        return lib.nlc_env_step_f64(env, delay, 0.05, state, buf, action, I, B, nu, None, None)

    for kw in ({"state": None}, {"buf": None}, {"action": None}, {"I": 0}, {"B": 0}, {"B": 9}, {"env": -1}, {"env": 3},
               {"delay": -1}, {"delay": 4}, {"B": 1, "delay": 1}):
        assert call(**kw) == -1, kw  # NLC_ERR_ARG
    assert b"delay" in lib.nlc_last_error()
    assert call(env=2, nu=1) == -2  # NLC_ERR_SHAPE: the acrobot takes two actions
    assert call(env=1, nu=2) == -2
    assert b"nu=" in lib.nlc_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_env_step_f64_has_no_cpu_fallback():
    from neurallaplacecontrol_b200 import _lib

    host = (C.c_double * 64)()
    p = C.addressof(host)
    assert _lib.load().nlc_env_step_f64(0, 1, 0.05, p, p, p, 2, 4, 1, None, None) != 0


def test_env_step_rejects_cpu_and_mixed_tensors():
    import neurallaplacecontrol_b200 as nlc

    s, b, a = torch.zeros(2, 3, dtype=torch.float64), torch.zeros(2, 4, 1, dtype=torch.float64), torch.zeros(2, 1, dtype=torch.float64)
    with pytest.raises(TypeError):
        nlc.env_step("oderl-pendulum", s, b, a, 1)  # no CPU path in either precision
    with pytest.raises(TypeError):
        nlc.env_step("oderl-pendulum", s.float(), b.float(), a.float(), 1)
    with pytest.raises(TypeError):
        nlc.env_step("oderl-pendulum", s.half(), b.half(), a.half(), 1)

"""CPU-side checks of the fp64 entry points: argument checks that need no device, and no CPU fallback in fp64 mode."""
import numpy as np
import pytest
import torch


def test_workspace_functions_reject_bad_arguments():
    from neurallaplacecontrol_b200 import _lib

    lib = _lib.load()
    for fn in (lib.nlc_model_forward_f64_workspace_bytes, lib.nlc_model_backward_f64_workspace_bytes):
        assert fn(None, 8, 1, 4) == -1  # NLC_ERR_ARG: no handle
    assert lib.nlc_model_forward_f64(None, None, None, None, None, 8, 1, 4, None, None, None, None) == -1
    assert lib.nlc_model_backward_f64(None, None, None, None, None, 8, 1, 4, None, None, None, None, None, None) == -1


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_fp64_mode_has_no_cpu_fallback():
    import neurallaplacecontrol_b200 as nlc

    m = nlc.NeuralLaplaceModel(3, 1, 3, hidden_units=128, s_recon_terms=17, state_mean=np.zeros(3), state_std=np.ones(3),
                               action_mean=np.zeros(1), action_std=np.ones(1), normalize=True, normalize_time=True,
                               math_mode="fp64").double()
    with pytest.raises(RuntimeError):
        m(torch.zeros(2, 3, dtype=torch.float64), torch.zeros(2, 4, 1, dtype=torch.float64), torch.full((2, 3), 0.05))

"""The oracle's forward with several prediction times per sample, ``ts`` (K, n_t), is n_t single-time forwards side by side:
column j of the (K, n_t, nx) result equals ``nl_forward`` at ``ts[:, j]`` (fp64).  The GPU tests of
``NeuralLaplaceModel.forward`` with (K, n_t) times (tests/test_gpu_multi_time.py) rest on these semantics."""
import pytest
import torch

from _util import DT, ENVS, weights
from oracle.costs import ENV_DIMS
from oracle.nl_model import nl_forward


@pytest.mark.parametrize("env", ENVS)
@pytest.mark.parametrize("n_t", [2, 7])
def test_oracle_multi_time_equals_single_time_columns(env, n_t):
    nx, nu = ENV_DIMS[env]
    sd = weights(env, calibrated=True)
    g = torch.Generator().manual_seed(n_t)
    K = 9
    obs = torch.randn(K, nx, generator=g, dtype=torch.float64)
    act = torch.randn(K, 4, nu, generator=g, dtype=torch.float64)
    inc = 0.2 + torch.empty(K, n_t, dtype=torch.float64).exponential_(1.0, generator=g)
    ts = DT * torch.cumsum(inc, dim=1)
    ts = ts[:, torch.randperm(n_t, generator=g)]  # not sorted
    multi = nl_forward(sd, obs, act, ts)
    assert multi.shape == (K, n_t, nx)
    for j in range(n_t):
        col = nl_forward(sd, obs, act, ts[:, j:j + 1])
        torch.testing.assert_close(multi[:, j], col, rtol=1e-12, atol=1e-14)

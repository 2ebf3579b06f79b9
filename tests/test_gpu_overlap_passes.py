"""Plans whose ping-pong rollout takes two passes per CTA run their encoder partly beside the rollout: the first pass's
samples are encoded before the fork, the last pass's samples in step-major order, their last steps beside the rollout,
which rolls out pass-major and polls only in its last pass.  Same kernels, same per-sample arithmetic: bit-identical
actions, costs, states and U as the plain sequence."""
import numpy as np
import pytest
import torch

from _util import DT, S_TERMS, START_STATE, weights

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)


def _model(env):
    import neurallaplacecontrol_b200 as nlc
    from oracle import costs

    nx, nu = costs.ENV_DIMS[env]
    m = nlc.NeuralLaplaceModel(nx, nu, nx, hidden_units=128, s_recon_terms=S_TERMS, ilt_algorithm="fourier",
                               encode_obs_time=False, state_mean=np.zeros(nx), state_std=np.ones(nx),
                               action_mean=np.array([0] * nu), action_std=np.array([1.0]), normalize=True,
                               normalize_time=True, dt=DT, math_mode="tc_split3").double()
    missing = m.load_state_dict(weights(env, calibrated=True))
    assert not missing.missing_keys and not missing.unexpected_keys
    return m


def _planner(env, model, K, T):
    import neurallaplacecontrol_b200 as nlc
    from oracle import costs

    nx, nu = costs.ENV_DIMS[env]
    ah = np.float32(costs.ENV_ACT_HIGH[env])
    return nlc.MPPIDelay(nlc.NLDynamics(model, DT), nlc.EnvRunningCost(env), nx, nlc.noise_sigma_for(nu), num_samples=K,
                         horizon=T, device="cuda:0", lambda_=1.0, u_min=torch.tensor(-ah), u_max=torch.tensor(ah), u_scale=ah,
                         U_init=torch.zeros(T, nu, dtype=torch.float64), math_mode="tc_split3", seed=5)


# config 4 on one GPU (512 tiles on 128 CTAs); a ragged plan (313 tiles on 79 CTAs: the last CTAs of the last pass hold one
# live tile or none); a short cartpole horizon (391 tiles on 98 CTAs)
@pytest.mark.parametrize("env,K,T", [("oderl-acrobot", 65536, 50), ("oderl-acrobot", 40001, 20), ("oderl-cartpole", 50000, 9)])
def test_two_pass_overlapped_step_equals_sequential_step(env, K, T, monkeypatch):
    from oracle import costs

    nx, nu = costs.ENV_DIMS[env]
    res = {}
    for name in ("overlap", "plain"):
        if name == "plain":  # a forced rollout form keeps the plain launch sequence
            monkeypatch.setenv("NLC_ROLLOUT_TILES", "3")
        p = _planner(env, _model(env), K, T)
        acts = []
        buf = torch.zeros(4, nu, dtype=torch.float64)
        for it in range(3):  # the third step runs from the captured graph
            acts.append(p.command(np.array(START_STATE[env]), buf).clone())
        ov, status = p.overlap_status()
        assert ov == (name == "overlap") and status == 0, (name, ov, status)
        res[name] = (torch.stack(acts), p.cost_total.clone(), p.states.clone(), p.U.clone())
    for a, b in zip(res["overlap"], res["plain"]):
        assert torch.equal(a, b)

"""Instance-batched planning and the closed control loop (BASELINE config 5; SURVEY 8 f2).

The reference evaluates one (env, delay, model, seed) instance per process: ``loop()`` of
``mppi_with_model.py:244-317`` alternates ``MPPIDelay.command`` (``:258``) with ``step_env`` (``:193-216``: ``get_action``,
one Euler step of the true dynamics, reward) and a host round trip per control step (``:254,267``).  Here ``I`` instances
of one environment share every kernel launch and nothing leaves the device inside the loop:

* :class:`BatchedMPPIDelay` - ``I`` independent ``MPPIDelay`` objects (own control sequence, action buffer, sampler seed):
  stage 1 and stage 4 per instance, ONE encoder launch and ONE rollout launch over all ``I*K`` samples
  (``nlc_batch_planner_*``).  Instance ``i`` reproduces a stand-alone ``MPPIDelay(..., seed=seeds[i])``.
* :func:`env_step` - ``step_env`` for ``I`` instances on the device (``nlc_env_step``; dynamics as stated by the
  reference's ``oracle.py:11-224``, golden-pinned in ``tests/golden/env_step_*.npz``).
* :func:`run_closed_loop` - ``loop()`` for ``I`` instances; returns the reference's result keys per instance.

Everything computes in ``libnlc_b200.so``; there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import time

import numpy as np
import torch

from . import _lib
from .closures import NLDynamics
from .planners.mppi_delay import MPPIDelay, _DevView


class BatchedMPPIDelay:
    """``n_instances`` planners of one environment / model behind one set of kernel launches.

    Constructor arguments are ``MPPIDelay``'s (``planners/mppi_delay.py:64-90``) plus ``n_instances``, ``seeds``
    (one sampler seed per instance, default ``range(n_instances)``) and ``U_init`` of shape ``(T, nu)`` (shared) or
    ``(I, T, nu)``.  ``process_group`` is not accepted: a batch is sharded by instance, never by sample (SURVEY 8e)."""

    def __init__(self, dynamics, running_cost, nx, noise_sigma, n_instances, seeds=None, U_init=None, **kw):
        if "process_group" in kw and kw["process_group"] is not None:
            raise NotImplementedError("BatchedMPPIDelay shards by instance: give each rank its own instances")
        if kw.get("math_mode") == "fp64":
            raise NotImplementedError("BatchedMPPIDelay has no fp64 mode: plan each instance with MPPIDelay(math_mode='fp64')")
        self.I = int(n_instances)
        self.seeds = list(range(self.I)) if seeds is None else [int(s) for s in seeds]
        if len(self.seeds) != self.I:
            raise ValueError("seeds must have one entry per instance")
        kw.setdefault("keep_states", False)
        T = kw.get("horizon", 15)
        self._tpl = MPPIDelay(dynamics, running_cost, nx, noise_sigma, U_init=torch.zeros(T, 1 if torch.as_tensor(noise_sigma).dim() == 0
                                                                                         else torch.as_tensor(noise_sigma).shape[0]), **kw)
        t = self._tpl
        self.K, self.T, self.nx, self.nu, self.B, self.d, self.dtype = t.K, t.T, t.nx, t.nu, t.B, t.d, t.dtype
        self.keep_states = t.keep_states
        self.noise_dist = t.noise_dist
        if U_init is None:
            U = torch.zeros(self.I, self.T, self.nu, dtype=torch.float64)
        else:
            U = torch.as_tensor(U_init).detach().to("cpu", torch.float64)
            U = U.reshape(1, self.T, self.nu).repeat(self.I, 1, 1) if U.numel() == self.T * self.nu else U.reshape(self.I, self.T, self.nu)
        self._U_host = U.contiguous()
        self._lib = _lib.load()
        self._handle, self._handle_B, self._handle_model, self._views, self._calls = None, None, None, {}, 0

    def _ensure(self, B):
        # the packed model is re-fetched on every call (see MPPIDelay._ensure): a rebuilt or re-folded model handle
        # must never be planned on silently
        model_h = None
        if isinstance(self._tpl.F, NLDynamics):
            if self._tpl.F.model._cuda_device is None:
                self._tpl.F.model._cuda_device = self.d
            model_h = self._tpl.F.model.set_prediction_time(self._tpl.F.dt)
        key = None if model_h is None else model_h.value
        if self._handle is not None and self._handle_B == B and self._handle_model == key:
            return self._handle
        self._destroy()
        self._handle_model = key
        d, model_h = self._tpl._desc(B, self.K, 0, self.K, 1, 0)
        seeds = (C.c_uint64 * self.I)(*self.seeds)
        h = C.c_void_p()
        _lib.check(self._lib.nlc_batch_planner_create(C.byref(h), model_h, C.byref(d), self.I, seeds, self.d.index), "nlc_batch_planner_create")
        ptr, keep = _lib.as_double_array(self._U_host.numpy())
        _lib.check(self._lib.nlc_batch_planner_set_U(h, ptr), "nlc_batch_planner_set_U")
        self._handle, self._handle_B, self._views = h, B, {}
        return h

    def _destroy(self):
        if self._handle is not None:
            # keep the planned control sequences: a new handle (another buffer length, a rebuilt model) starts from them
            self._U_host = self._buf(_lib.BUF_U, (self.I, self.T, self.nu)).detach().to("cpu", torch.float64).contiguous()
            self._lib.nlc_batch_planner_destroy(self._handle)
            self._handle, self._views = None, {}

    def _set_U(self, value):
        U = torch.as_tensor(value).detach().to("cpu", torch.float64)
        U = U.reshape(1, self.T, self.nu).repeat(self.I, 1, 1) if U.numel() == self.T * self.nu else U.reshape(self.I, self.T, self.nu)
        self._U_host = U.contiguous()
        if self._handle is not None:
            ptr, keep = _lib.as_double_array(self._U_host.numpy())
            _lib.check(self._lib.nlc_batch_planner_set_U(self._handle, ptr), "nlc_batch_planner_set_U")

    def reset(self):
        """``MPPIDelay.reset`` (``mppi_delay.py:226-230``) for every instance: resample each control sequence."""
        self._set_U(self.noise_dist.sample((self.I, self.T)))

    def __del__(self):
        try:
            self._destroy()
        except Exception:
            pass

    def _buf(self, which, shape):
        key = (which, tuple(shape))
        if key not in self._views:
            p, n = C.c_void_p(), C.c_int64()
            _lib.check(self._lib.nlc_batch_planner_buffer(self._handle, which, C.byref(p), C.byref(n)), "nlc_batch_planner_buffer")
            if p.value is None or n.value == 0:
                return None
            assert int(np.prod(shape)) == n.value, (which, shape, n.value)
            self._views[key] = torch.as_tensor(_DevView(p.value, shape), device=self.d)
        return self._views[key]

    def _after(self, which, shape):
        return None if self._handle is None or self._calls == 0 else self._buf(which, shape)

    # the single planner's attributes, with a leading instance axis
    U = property(lambda self: self._U_host.to(self.dtype) if self._handle is None else self._buf(_lib.BUF_U, (self.I, self.T, self.nu)),
                 lambda self, value: self._set_U(value))
    noise = property(lambda self: self._after(_lib.BUF_NOISE, (self.I, self.K, self.T, self.nu)))
    perturbed_action = property(lambda self: self._after(_lib.BUF_PERTURBED, (self.I, self.K, self.T, self.nu)))
    cost_total = property(lambda self: self._after(_lib.BUF_COST_TOTAL, (self.I, self.K)))
    actions = property(lambda self: self._after(_lib.BUF_ACTIONS, (self.I, self.K, self.T, self.nu)))
    states = property(lambda self: self._after(_lib.BUF_STATES, (self.I, self.K, self.T, self.nx)) if self.keep_states else None)

    @property
    def omega(self):
        if self._handle is None or self._calls == 0:
            return None
        w = self._buf(_lib.BUF_WEIGHTS, (self.I, self.K))
        return w / self._buf(_lib.BUF_STATS, (self.I, 2))[:, 1:2]

    def command(self, states, action_buffers, noise=None):
        """``MPPIDelay.command`` for every instance.  ``states`` (I, nx), ``action_buffers`` (I, B, nu) env units,
        ``noise`` optional injected samples (I, K, T, nu).  Returns the actions (I, nu), env units, on the device."""
        action_buffers = torch.as_tensor(action_buffers)
        B = action_buffers.shape[1]
        h = self._ensure(B)
        st = torch.as_tensor(states).to(device=self.d, dtype=torch.float32).reshape(self.I, self.nx).contiguous()
        ab = action_buffers.to(device=self.d, dtype=torch.float32).reshape(self.I, B, self.nu).contiguous()
        nz = None
        if noise is not None:
            nz = torch.as_tensor(noise).to(device=self.d, dtype=torch.float32).reshape(self.I, self.K, self.T, self.nu).contiguous()
        out = torch.empty(self.I, self.nu, dtype=torch.float32, device=self.d)
        with torch.cuda.device(self.d):
            _lib.check(self._lib.nlc_batch_planner_command(h, st.data_ptr(), ab.data_ptr(), _lib.ptr(nz), out.data_ptr(),
                                                           _lib.current_stream_ptr()), "nlc_batch_planner_command")
        self._calls += 1
        return out.to(self.dtype)


def env_step(env_name, states, action_buffers, actions, action_delay, dt=0.05, rewards=None):
    """``step_env`` (``mppi_with_model.py:193-216``) for I instances, in place on fp32 CUDA tensors: ``action_buffers``
    (I, B, nu) is rolled and receives ``actions`` (I, nu) (``get_action``, ``:25-28``), ``states`` (I, nx) advances by
    one Euler step of the true dynamics driven by the delayed action, ``rewards`` (I) receives the step reward."""
    for t in (states, action_buffers, actions):
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
            raise TypeError("env_step works in place on contiguous fp32 CUDA tensors (no CPU fallback)")
    I, B, nu = action_buffers.shape
    ro = _lib.RolloutOpts()
    ro.env, ro.state_constraint, ro.goal_x, ro.dynamics, ro.delay, ro.dt = _lib.ENV_IDS[env_name], 0, 0.0, _lib.DYN_ANALYTIC_DELAY, int(action_delay), float(dt)
    with torch.cuda.device(states.device):
        _lib.check(_lib.load().nlc_env_step(C.byref(ro), states.data_ptr(), action_buffers.data_ptr(), actions.data_ptr(), I, B, nu,
                                            _lib.ptr(rewards), _lib.current_stream_ptr()), "nlc_env_step")


def run_closed_loop(planner: BatchedMPPIDelay, env_name, states0, action_delay, n_steps, dt=0.05, noise_fn=None):
    """``loop()`` of ``mppi_with_model.py:244-317`` for ``planner.I`` instances: zero action buffers (``:245``), then
    ``n_steps`` x (command, step_env); rewards accumulate on the device.

    NOT the reference environment's integrator: ``env_step`` takes ONE EXPLICIT EULER step of the dynamics as the
    reference's ``oracle.py`` states them (what its "oracle" planner model uses), whereas the reference's gym envs
    integrate the same right-hand side with ``torchdiffeq.odeint`` (``base_env.py:136-173``, dopri5 by default).
    Closed-loop rewards are therefore those of the Euler-discretised plant, not the reference environment's.  ``noise_fn(it)`` may return injected noise for
    step ``it`` (parity tests).  Returns the reference's result keys (``:289-302``) with per-instance arrays."""
    I, B, nu, dev = planner.I, planner.B, planner.nu, planner.d
    states = torch.as_tensor(states0).to(device=dev, dtype=torch.float32).reshape(I, planner.nx).clone()
    bufs = torch.zeros(I, B, nu, dtype=torch.float32, device=dev)
    total = torch.zeros(I, dtype=torch.float32, device=dev)
    reward = torch.zeros(I, dtype=torch.float32, device=dev)
    elapsed = 0.0
    for it in range(int(n_steps)):
        t0 = time.perf_counter()
        actions = planner.command(states, bufs, None if noise_fn is None else noise_fn(it))
        torch.cuda.synchronize(dev)
        elapsed += time.perf_counter() - t0  # the reference's bracket (:255-264) around command()
        env_step(env_name, states, bufs, actions.to(torch.float32).contiguous(), action_delay, dt, reward)
        total += reward
    torch.cuda.synchronize(dev)
    tot = total.double().cpu().numpy()
    return {"env_name": env_name, "roll_outs": planner.K, "time_steps": planner.T, "episode_elapsed_time": elapsed,
            "episode_elapsed_time_per_it": elapsed / max(int(n_steps), 1), "dt": dt, "delay": action_delay, "planner": "mpc",
            "total_reward_raw": tot, "total_reward": tot * (200.0 / max(int(n_steps), 1)), "final_states": states.double().cpu().numpy(),
            "n_instances": I}

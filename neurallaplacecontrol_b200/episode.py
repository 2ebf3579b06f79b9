"""Instance-batched planning and the closed control loop (BASELINE config 5; SURVEY 8 f2).

The reference evaluates one (env, delay, model, seed) instance per process: ``loop()`` of
``mppi_with_model.py:244-317`` alternates ``MPPIDelay.command`` (``:258``) with ``step_env`` (``:193-216``: ``get_action``,
one Euler step of the true dynamics, reward) and a host round trip per control step (``:254,267``).  Here ``I`` instances
of one environment share every kernel launch and nothing leaves the device inside the loop:

* :class:`BatchedMPPIDelay` - ``I`` independent ``MPPIDelay`` objects (own control sequence, action buffer, sampler seed,
  and optionally own model or analytic delay): stage 1 and stage 4 per instance, ONE encoder launch and ONE rollout launch
  per run of consecutive instances sharing a model (``nlc_batch_planner_*``), the runs side by side on the GPU.  Instance
  ``i`` reproduces a stand-alone ``MPPIDelay(dynamics_i, ..., seed=seeds[i])``.
* :func:`env_step` - ``step_env`` for ``I`` instances on the device (``nlc_env_step``, or ``nlc_env_step_f64`` on fp64
  tensors, ``*_delays`` with one action delay per instance; dynamics as stated by the reference's ``oracle.py:11-224``,
  golden-pinned in ``tests/golden/env_step_*.npz``).
* :func:`run_closed_loop` - ``loop()`` for ``I`` instances of a ``BatchedMPPIDelay``, or in fp64 over one
  ``MPPIDelay(math_mode="fp64")`` per instance; returns the reference's result keys per instance.

Everything computes in ``libnlc_b200.so``; there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import time

import torch

from . import _lib
from .closures import AnalyticDelayDynamics, NLDynamics
from .planners.mppi_delay import MPPIDelay, _MPPIDelayF64, _buffer_view


class BatchedMPPIDelay:
    """``n_instances`` planners of one environment behind one set of kernel launches.

    Constructor arguments are ``MPPIDelay``'s (``planners/mppi_delay.py:64-90``) plus ``n_instances``, ``seeds``
    (one sampler seed per instance, default ``range(n_instances)``) and ``U_init`` of shape ``(T, nu)`` (shared) or
    ``(I, T, nu)``.  ``process_group`` is not accepted: a batch is sharded by instance, never by sample (SURVEY 8e).

    ``dynamics`` is one handle for every instance, or a sequence of ``n_instances`` handles - all ``NLDynamics`` (each
    instance plans with its own model; instances holding the same model object share its device handle) or all
    ``AnalyticDelayDynamics`` (each with its own delay), with one ``dt``.  The reference's grid of one checkpoint per
    (delay, seed) then plans as one batch: consecutive instances with the same model (or analytic delay) form a run, one
    encoder and one rollout launch per run, the runs side by side on the GPU.  Keep instances of one model adjacent."""
    _c_buffer, _typestr = "nlc_batch_planner_buffer", "<f4"

    def __init__(self, dynamics, running_cost, nx, noise_sigma, n_instances, seeds=None, U_init=None, **kw):
        if "process_group" in kw and kw["process_group"] is not None:
            raise NotImplementedError("BatchedMPPIDelay shards by instance: give each rank its own instances")
        if kw.get("math_mode") == "fp64":
            raise NotImplementedError("BatchedMPPIDelay has no fp64 mode: plan each instance with MPPIDelay(math_mode='fp64') "
                                      "and drive them with run_closed_loop([planner_0, planner_1, ...], ...)")
        self.I = int(n_instances)
        self.seeds = list(range(self.I)) if seeds is None else [int(s) for s in seeds]
        if len(self.seeds) != self.I:
            raise ValueError("seeds must have one entry per instance")
        self._dyns = self._check_dynamics(dynamics, nx, running_cost, kw.get("action_buffer_size", 4))
        kw.setdefault("keep_states", False)
        T = kw.get("horizon", 15)
        self._tpl = MPPIDelay(self._dyns[0], running_cost, nx, noise_sigma, U_init=torch.zeros(T, 1 if torch.as_tensor(noise_sigma).dim() == 0
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

    def _check_dynamics(self, dynamics, nx, running_cost, B):
        """One dynamics handle per instance, checked before anything reaches the device."""
        if not isinstance(dynamics, (list, tuple)):
            return [dynamics] * self.I
        dyns = list(dynamics)
        if len(dyns) != self.I:
            raise ValueError(f"dynamics must be one handle or one per instance ({self.I}), got {len(dyns)}")
        if not (all(isinstance(d, NLDynamics) for d in dyns) or all(isinstance(d, AnalyticDelayDynamics) for d in dyns)):
            raise TypeError("the dynamics of one batch must be all NLDynamics or all AnalyticDelayDynamics handles")
        if len({d.dt for d in dyns}) != 1:
            raise ValueError("the dynamics of one batch must share dt")
        nu = _lib.ENV_DIMS[running_cost.env_name][1]
        for i, d in enumerate(dyns):
            if isinstance(d, NLDynamics) and (d.model.output_dim, d.model.action_dim) != (nx, nu):
                raise ValueError(f"instance {i}: the model's (state_dim, action_dim) = {(d.model.output_dim, d.model.action_dim)}, "
                                 f"the batch plans ({nx}, {nu})")
            if isinstance(d, AnalyticDelayDynamics):
                if d.env_name != running_cost.env_name:
                    raise ValueError(f"instance {i}: analytic dynamics of {d.env_name} in a batch of {running_cost.env_name}")
                if not 0 <= d.delay < int(B):
                    raise ValueError(f"instance {i}: delay {d.delay} outside the {int(B)}-entry action buffer")
        return dyns

    def _model_handles(self):
        """The device handle of every instance's model (None for the analytic dynamics).  Each distinct model is re-fetched
        on every call (see MPPIDelay._ensure): a rebuilt or re-folded model handle must never be planned on silently."""
        if not isinstance(self._dyns[0], NLDynamics):
            return None
        by_model = {}
        for d in self._dyns:
            if id(d.model) not in by_model:
                if d.model._cuda_device is None:
                    d.model._cuda_device = self.d
                by_model[id(d.model)] = self._tpl._fetch_handle(d.model)
        return [by_model[id(d.model)] for d in self._dyns]

    def _ensure(self, B):
        handles = self._model_handles()
        delays = [int(d.delay) for d in self._dyns]
        key = (None if handles is None else tuple(h.value for h in handles), tuple(delays))
        if self._handle is not None and self._handle_B == B and self._handle_model == key:
            return self._handle
        self._destroy()
        self._handle_model = key
        d = self._tpl._desc(B, self.K, 0, self.K, 1, 0)
        seeds = (C.c_uint64 * self.I)(*self.seeds)
        models = None if handles is None else (C.c_void_p * self.I)(*key[0])
        dl = (C.c_int32 * self.I)(*delays)
        h = C.c_void_p()
        _lib.check(self._lib.nlc_batch_planner_create_multi(C.byref(h), models, dl, C.byref(d), self.I, seeds, self.d.index),
                   "nlc_batch_planner_create_multi")
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

    _buf = _buffer_view

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


def _delays(action_delay, I, B, device):
    """``action_delay`` as the env step takes it: an int (returned as is), or one delay per instance (a sequence or an integer
    tensor of ``I`` entries, each in ``[0, B)``, checked here on the host) returned as an int32 CUDA tensor."""
    d = torch.as_tensor(action_delay).detach().cpu()
    if d.dim() == 0:
        return int(action_delay)
    if d.is_floating_point() or d.is_complex() or d.dtype == torch.bool:
        raise TypeError("per-instance delays must be integers")
    d = d.reshape(-1)
    if d.numel() != I:
        raise ValueError(f"action_delay must be an int or hold one delay per instance ({I}), got {d.numel()}")
    if bool(((d < 0) | (d >= B)).any()):
        raise ValueError(f"action delays {d.tolist()} must lie in [0, {B}) (the action buffer has {B} entries)")
    return d.to(device=device, dtype=torch.int32)


def _env_step(env_name, states, action_buffers, actions, delay, dt, rewards, status):
    """The launch of :func:`env_step` on checked arguments: ``delay`` an int or the int32 CUDA tensor of ``_delays``,
    ``status`` an int32 CUDA word (per-instance delays only; set to 1 by the kernel for an entry out of range)."""
    I, B, nu = action_buffers.shape
    lib, env, stream = _lib.load(), _lib.ENV_IDS[env_name], _lib.current_stream_ptr()
    per_instance = torch.is_tensor(delay)
    if states.dtype == torch.float64:
        if per_instance:
            _lib.check(lib.nlc_env_step_f64_delays(env, delay.data_ptr(), float(dt), states.data_ptr(), action_buffers.data_ptr(),
                                                   actions.data_ptr(), I, B, nu, _lib.ptr(rewards), status.data_ptr(), stream),
                       "nlc_env_step_f64_delays")
        else:
            _lib.check(lib.nlc_env_step_f64(env, delay, float(dt), states.data_ptr(), action_buffers.data_ptr(), actions.data_ptr(),
                                            I, B, nu, _lib.ptr(rewards), stream), "nlc_env_step_f64")
        return
    ro = _lib.RolloutOpts()
    ro.env, ro.state_constraint, ro.goal_x, ro.dynamics, ro.delay, ro.dt = env, 0, 0.0, _lib.DYN_ANALYTIC_DELAY, 0 if per_instance else delay, float(dt)
    if per_instance:
        _lib.check(lib.nlc_env_step_delays(C.byref(ro), delay.data_ptr(), states.data_ptr(), action_buffers.data_ptr(), actions.data_ptr(),
                                           I, B, nu, _lib.ptr(rewards), status.data_ptr(), stream), "nlc_env_step_delays")
    else:
        _lib.check(lib.nlc_env_step(C.byref(ro), states.data_ptr(), action_buffers.data_ptr(), actions.data_ptr(), I, B, nu,
                                    _lib.ptr(rewards), stream), "nlc_env_step")


def env_step(env_name, states, action_buffers, actions, action_delay, dt=0.05, rewards=None):
    """``step_env`` (``mppi_with_model.py:193-216``) for I instances, in place on CUDA tensors: ``action_buffers``
    (I, B, nu) is rolled and receives ``actions`` (I, nu) (``get_action``, ``:25-28``), ``states`` (I, nx) advances by
    one Euler step of the true dynamics driven by the delayed action, ``rewards`` (I) receives the step reward.
    ``action_delay`` is one int for every instance, or one delay per instance (a sequence or an integer tensor of I entries,
    each in ``[0, B)``; checked on the host before the launch) - the reference's delay grid in one call.

    All tensors (``rewards`` if given) are contiguous and either all fp32 (``nlc_env_step``) or all fp64
    (``nlc_env_step_f64``: the reference's own precision and evaluation order, ``dt`` kept in fp64); anything else raises
    ``TypeError``.  In both precisions this is the Euler step of the reference's ``oracle.py``, NOT the reference
    environment's integrator (see :func:`run_closed_loop`)."""
    tensors = [t for t in (states, action_buffers, actions, rewards) if t is not None]
    dtype = states.dtype
    if dtype not in (torch.float32, torch.float64) or not all(t.is_cuda and t.dtype == dtype and t.is_contiguous() for t in tensors):
        raise TypeError("env_step works in place on contiguous CUDA tensors, all fp32 or all fp64 (no CPU fallback)")
    I, B, nu = action_buffers.shape
    with torch.cuda.device(states.device):
        delay = _delays(action_delay, I, B, states.device)
        status = torch.zeros(1, dtype=torch.int32, device=states.device) if torch.is_tensor(delay) else None
        _env_step(env_name, states, action_buffers, actions, delay, dt, rewards, status)


class _F64Instances:
    """One ``MPPIDelay(math_mode="fp64")`` per instance behind the ``command`` of :class:`BatchedMPPIDelay`: a control step
    plans every instance in turn on the device (``nlc_planner_f64_command``) and stacks the actions."""

    def __init__(self, planners):
        self.planners = list(planners)
        if not self.planners:
            raise ValueError("run_closed_loop needs at least one planner")
        for p in self.planners:
            if not isinstance(p, _MPPIDelayF64):
                raise TypeError("a list of planners must hold MPPIDelay(math_mode='fp64') objects, one per instance "
                                "(fp32 instances are batched by BatchedMPPIDelay)")
        p0 = self.planners[0]
        for p in self.planners:
            if (p.nx, p.nu, p.B, p.d) != (p0.nx, p0.nu, p0.B, p0.d):
                raise ValueError("the planners of one closed loop must share nx, nu, the action buffer size and the device")
            if p.u_per_command != 1:
                raise ValueError("the closed loop applies one action per command: u_per_command must be 1")
        self.I, self.nx, self.nu, self.B, self.d, self.K, self.T = len(self.planners), p0.nx, p0.nu, p0.B, p0.d, p0.K, p0.T

    def command(self, states, action_buffers, noise=None):
        """``states`` (I, nx), ``action_buffers`` (I, B, nu) fp64 on the device; ``noise`` optional (I, K, T, nu): instance
        i's slice goes in through its planner's ``noise_dist.sample`` for this call only.  Returns the actions (I, nu)."""
        actions = []
        for i, p in enumerate(self.planners):
            if noise is None:
                actions.append(p.command(states[i], action_buffers[i]))
                continue
            saved = p.noise_dist.__dict__.get("sample")
            p.noise_dist.sample = lambda shape, nz=noise[i]: nz
            try:
                actions.append(p.command(states[i], action_buffers[i]))
            finally:
                if saved is None:
                    del p.noise_dist.sample
                else:
                    p.noise_dist.sample = saved
        return torch.stack(actions)


def run_closed_loop(planner, env_name, states0, action_delay, n_steps, dt=0.05, noise_fn=None):
    """``loop()`` of ``mppi_with_model.py:244-317`` for I instances: zero action buffers (``:245``), then
    ``n_steps`` x (command, step_env); rewards accumulate on the device.

    ``planner`` is a :class:`BatchedMPPIDelay` (``I = planner.I``; fp32 state, buffers and rewards), or a list / tuple of
    ``MPPIDelay(math_mode="fp64")`` objects, one per instance (``I = len(planner)``; they share ``nx``, ``nu``, the action
    buffer size and the device, and take ``u_per_command == 1``): then the state, the buffers and the rewards are fp64 like
    the reference's loop, each instance plans on its own planner and one fp64 ``env_step`` advances them all.
    ``roll_outs`` / ``time_steps`` of the result are those of the first planner.  ``action_delay`` is one int or one delay per
    instance (as :func:`env_step` takes it, checked before the first control step); the result's ``"delay"`` is then an
    array of the I delays.

    NOT the reference environment's integrator: ``env_step`` takes ONE EXPLICIT EULER step of the dynamics as the
    reference's ``oracle.py`` states them (what its "oracle" planner model uses), whereas the reference's gym envs
    integrate the same right-hand side with ``torchdiffeq.odeint`` (``base_env.py:136-173``, dopri5 by default).
    Closed-loop rewards are therefore those of the Euler-discretised plant, not the reference environment's.  ``noise_fn(it)`` may return injected noise
    (I, K, T, nu) for step ``it`` (parity tests).  Returns the reference's result keys (``:289-302``) with per-instance arrays."""
    if isinstance(planner, (list, tuple)):
        planner, dtype = _F64Instances(planner), torch.float64
    else:
        dtype = torch.float32
    I, B, nu, dev = planner.I, planner.B, planner.nu, planner.d
    with torch.cuda.device(dev):
        delay = _delays(action_delay, I, B, dev)  # checked once, before the first launch
        status = torch.zeros(1, dtype=torch.int32, device=dev) if torch.is_tensor(delay) else None
    states = torch.as_tensor(states0).to(device=dev, dtype=dtype).reshape(I, planner.nx).clone()
    bufs = torch.zeros(I, B, nu, dtype=dtype, device=dev)
    total = torch.zeros(I, dtype=dtype, device=dev)
    reward = torch.zeros(I, dtype=dtype, device=dev)
    elapsed = 0.0
    for it in range(int(n_steps)):
        t0 = time.perf_counter()
        actions = planner.command(states, bufs, None if noise_fn is None else noise_fn(it))
        torch.cuda.synchronize(dev)
        elapsed += time.perf_counter() - t0  # the reference's bracket (:255-264) around command()
        with torch.cuda.device(dev):
            _env_step(env_name, states, bufs, actions.to(dtype).contiguous(), delay, dt, reward, status)
        total += reward
    torch.cuda.synchronize(dev)
    tot = total.double().cpu().numpy()
    return {"env_name": env_name, "roll_outs": planner.K, "time_steps": planner.T, "episode_elapsed_time": elapsed,
            "episode_elapsed_time_per_it": elapsed / max(int(n_steps), 1), "dt": dt,
            "delay": delay.cpu().numpy() if torch.is_tensor(delay) else action_delay, "planner": "mpc",
            "total_reward_raw": tot, "total_reward": tot * (200.0 / max(int(n_steps), 1)), "final_states": states.double().cpu().numpy(),
            "n_instances": I}

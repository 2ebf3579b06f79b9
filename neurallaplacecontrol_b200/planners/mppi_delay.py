"""``MPPIDelay`` with the reference's constructor, ``command(state, action_buffer)`` / ``reset`` /
``get_rollouts`` signatures and post-call attributes (``planners/mppi_delay.py:52-381``), executed as a fixed
sequence of sm_100a kernels behind ``libnlc_b200.so``.

Differences a caller can see, all deliberate:

* ``dynamics`` / ``running_cost`` must be the declarative handles of :mod:`neurallaplacecontrol_b200.closures`
  (a fused kernel cannot call opaque Python; there is no CPU fallback, so anything else raises ``TypeError``).
* Arithmetic is fp32 on the device; tensors left on the object (``noise``, ``perturbed_action``, ``cost_total``,
  ``cost_total_non_zero``, ``omega``, ``states``, ``actions``, ``U``) are fp32 CUDA tensors (zero-copy views of the
  planner's buffers); the returned action is cast to ``noise_sigma.dtype`` like the reference's.
* Options the reference's callers never use and this path does not implement raise ``NotImplementedError``
  instead of being silently ignored: ``terminal_state_cost`` (an opaque callable), ``step_dependent_dynamics``, ``rollout_samples > 1``
  (legacy variance branch, ``:291-292,310``), planner-level ``encode_obs_time`` with a Neural Laplace model (a model built
  with ``encode_obs_time=True`` is supported: the closure-level time channel of ``mppi_with_model.py:110-119`` is
  synthesised inside the encoder kernels).
* Extra keyword arguments (not in the reference): ``process_group`` shards the K samples over the ranks of a
  ``torch.distributed`` group (one exchange of the (beta, eta, W) triple per control step), ``seed`` keys the
  on-device Philox sampler, ``math_mode`` selects the contraction arithmetic (default ``"tc_split3"``: tcgen05 tensor
  cores, fp16 hi/lo split operands, fp32 accumulate - fp32-class, the 1e-4 bound; ``"fp32"`` = CUDA-core FFMA anchor;
  ``"tc_fp16"`` = single pass, 2e-2 bound; ``"fp64"`` = the whole control step in fp64, see below), ``keep_states`` can
  drop the ``states`` trajectory output.

``math_mode="fp64"`` plans at the reference's own precision (its model is ``.double()``, ``train_utils.py:267``, and its
``noise_sigma`` fp64): the object is an fp64 planner (``nlc_planner_f64_*``) whose kernels compute every stage in fp64 -
stage 1 bit-identical to the reference for the same noise, the model as ``NeuralLaplaceModel(math_mode="fp64")`` computes it,
fixed-order softmax sums.  It works whatever the model's own ``math_mode``: before every control step the model's parameters
go to the device as one flat fp64 tensor when they changed (``_fingerprint``), so an optimizer step between two commands is
planned with.  Post-call attributes are fp64 CUDA tensors (zero-copy views), injected noise is kept in fp64.  It plans on one
GPU: ``process_group`` / ``shard``, ``get_rollouts``, ``set_inputs`` / ``step`` and ``BatchedMPPIDelay`` raise
``NotImplementedError``.

Noise injection for parity tests works as on the reference: replace ``planner.noise_dist.sample`` with a callable
returning the ``(K, T, nu)`` tensor (it is called once per ``command`` with ``(K, T)``, ``mppi_delay.py:319``).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
from torch.distributions.multivariate_normal import MultivariateNormal

from .. import _lib, sharding
from ..closures import AnalyticDelayDynamics, EnvRunningCost, NLDynamics


import contextlib

_NULL_CTX = contextlib.nullcontext()


class _DevView:
    """Zero-copy torch view of a raw device buffer through ``__cuda_array_interface__``."""

    def __init__(self, ptr, shape, typestr="<f4"):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}


def _bound_vector(x, nu, name):
    """Bound per action dimension: a scalar (what the reference's callers pass, mppi_with_model.py:227-228) or ``nu`` values.
    With a ``(nu,)`` tensor the reference's ``_bound_action`` (``mppi_delay.py:347-356``: slices of the T axis, ``torch.min``
    broadcasting over the last axis) clamps every ``(k, t, u)`` entry to ``[u_min[u], u_max[u]]``."""
    if x is None:
        return None
    t = torch.as_tensor(x, dtype=torch.float64).reshape(-1)
    if t.numel() == 1:
        t = t.repeat(nu)
    if t.numel() != nu:
        raise ValueError(f"{name} must be a scalar or have one entry per action dimension ({nu})")
    return t


class MPPIDelay:
    def __new__(cls, *args, **kw):
        if cls is MPPIDelay and kw.get("math_mode") == "fp64":
            cls = _MPPIDelayF64  # a planner object of its own (nlc_planner_f64_*): see its docstring
        return super().__new__(cls)

    def __init__(self, dynamics, running_cost, nx, noise_sigma, num_samples=100, horizon=15, device="cpu",
                 terminal_state_cost=None, lambda_=1.0, noise_mu=None, u_min=None, u_max=None, u_init=None,
                 U_init=None, u_scale=1, u_per_command=1, step_dependent_dynamics=False, rollout_samples=1,
                 rollout_var_cost=0, rollout_var_discount=0.95, dt=0.05, sample_null_action=False,
                 noise_abs_cost=False, encode_obs_time=False, *, process_group=None, seed=0, math_mode="tc_split3",
                 keep_states=True, action_buffer_size=4, shard=None):
        if not isinstance(dynamics, (NLDynamics, AnalyticDelayDynamics)):
            raise TypeError("dynamics must be an NLDynamics or AnalyticDelayDynamics handle: the fused rollout kernel "
                            "cannot call an opaque Python callable and this package has no CPU fallback")
        if not isinstance(running_cost, EnvRunningCost):
            raise TypeError("running_cost must be an EnvRunningCost handle (see neurallaplacecontrol_b200.closures)")
        if terminal_state_cost is not None:
            raise NotImplementedError("terminal_state_cost is not used on the reference path and is not implemented")
        if step_dependent_dynamics:
            raise NotImplementedError("step_dependent_dynamics is not implemented")
        if rollout_samples != 1:
            raise NotImplementedError("rollout_samples > 1 (legacy variance branch) is not implemented")
        if encode_obs_time and not isinstance(dynamics, AnalyticDelayDynamics):
            # mppi_delay.py:261-287 appends a running time channel to the window it hands to `dynamics`; the reference
            # only uses that with the analytic dynamics (mppi_dataset_collector.py:166-180), which ignore the channel.
            # A Neural Laplace model with encode_obs_time gets its channel from the closure instead (NLDynamics).
            raise NotImplementedError("planner-level encode_obs_time is implemented for AnalyticDelayDynamics only")
        if not 1 <= int(u_per_command) <= int(horizon):
            raise ValueError("u_per_command must lie in [1, horizon]")
        dev = torch.device(device)
        if dev.type != "cuda":
            if not torch.cuda.is_available():
                raise RuntimeError("MPPIDelay (B200) needs a CUDA device; there is no CPU fallback")
            dev = torch.device("cuda", torch.cuda.current_device())
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.d = dev
        noise_sigma = torch.as_tensor(noise_sigma)
        self.dtype = noise_sigma.dtype
        self.K = num_samples
        self.T = horizon
        self.encode_obs_time = encode_obs_time
        self.dt = dt
        self.nx = nx
        self.nu = 1 if noise_sigma.dim() == 0 else noise_sigma.shape[0]
        self.lambda_ = lambda_
        if noise_mu is None:
            noise_mu = torch.zeros(self.nu, dtype=self.dtype)
        if u_init is None:
            u_init = torch.zeros_like(noise_mu)
        if self.nu == 1:
            noise_mu = noise_mu.view(-1)
            noise_sigma = noise_sigma.view(-1, 1)
        self.u_scale = u_scale
        self.u_per_command = u_per_command
        # mppi_delay.py:143-150: if one bound is given the other is its negative
        lo, hi = _bound_vector(u_min, self.nu, "u_min"), _bound_vector(u_max, self.nu, "u_max")
        if hi is not None and lo is None:
            lo = -hi
        if lo is not None and hi is None:
            hi = -lo
        scalar = lo is not None and bool((lo == lo[0]).all()) and bool((hi == hi[0]).all())
        self.u_min = None if lo is None else (lo[0] if scalar else lo).to(device=self.d, dtype=torch.float32)
        self.u_max = None if hi is None else (hi[0] if scalar else hi).to(device=self.d, dtype=torch.float32)
        self._bounds = None if lo is None else (lo.tolist(), hi.tolist())
        self.noise_mu = noise_mu
        self.noise_sigma = noise_sigma
        self.noise_sigma_inv = torch.inverse(noise_sigma)
        self.noise_dist = MultivariateNormal(noise_mu, covariance_matrix=noise_sigma)
        self.u_init = u_init
        self.F = dynamics
        self.running_cost = running_cost
        self.terminal_state_cost = None
        self.sample_null_action = sample_null_action
        self.noise_abs_cost = noise_abs_cost
        self.state = None
        self.M = rollout_samples
        self.rollout_var_cost = rollout_var_cost
        self.rollout_var_discount = rollout_var_discount
        self.B = int(action_buffer_size)
        self.math_mode = math_mode
        self.keep_states = bool(keep_states)
        self.seed = int(seed)

        # ---- sharding of the K samples (SURVEY 8e) -------------------------------------------------------------
        self.process_group = process_group
        if process_group is not None:
            import torch.distributed as dist

            self.G = dist.get_world_size(process_group)
            self.rank = dist.get_rank(process_group)
        elif shard is not None:
            # (rank, G) without a process group: the caller moves the triples between the shards itself and drives the
            # control step through _rollout_phase / _finish_phase (single-GPU tests of the sharded arithmetic)
            self.rank, self.G = int(shard[0]), int(shard[1])
        else:
            self.G, self.rank = 1, 0
        self.k_offset, self.K_local = sharding.shard_range(self.K, self.G, self.rank)

        self._lib = _lib.load()
        self._handle = None
        self._handle_B = None
        self._handle_model = None
        self._exchange = False
        self.last_action_host = None
        self._views = {}
        if U_init is None:
            U_init = self._replicated(self.noise_dist.sample((self.T,)))  # mppi_delay.py:163-164
        self._U_host = torch.as_tensor(U_init).detach().to("cpu", torch.float64).reshape(self.T, self.nu).clone()
        self._U_dirty = True

    def _replicated(self, t):
        """A tensor drawn from this rank's own RNG, made identical on every rank of the shard group (rank 0's draw wins):
        U must start replicated for the sharded plan to equal the unsharded one."""
        if self.G == 1:
            return t
        import torch.distributed as dist

        backend = dist.get_backend(self.process_group)
        buf = t.detach().to(self.d if backend == "nccl" else "cpu", torch.float64).contiguous()
        dist.broadcast(buf, src=dist.get_global_rank(self.process_group, 0), group=self.process_group)
        return buf.cpu()

    # ---- device handle ---------------------------------------------------------------------------------------
    def _desc(self, B, K_local, k_offset, k_total, n_shards, shard_index):
        """``nlc_planner_desc`` of this planner's options (shared with the instance-batched planner)."""
        d = _lib.PlannerDesc()
        mp = d.mppi
        mp.K, mp.T, mp.nu, mp.B = K_local, self.T, self.nu, B
        mp.k_offset, mp.k_total = k_offset, k_total
        mp.lambda_, mp.u_scale = float(self.lambda_), float(self.u_scale)
        mp.has_bounds = int(self.u_max is not None)
        if self._bounds is not None:
            for i in range(self.nu):
                mp.u_min[i], mp.u_max[i] = self._bounds[0][i], self._bounds[1][i]
        mp.sample_null_action, mp.noise_abs_cost = int(self.sample_null_action), int(self.noise_abs_cost)
        sinv = self.noise_sigma_inv.to(torch.float64).reshape(self.nu, self.nu)
        chol = torch.linalg.cholesky(self.noise_sigma.to(torch.float64).reshape(self.nu, self.nu))
        for i in range(self.nu):
            mp.noise_mu[i] = float(self.noise_mu.reshape(-1)[i])
            mp.u_init[i] = float(torch.as_tensor(self.u_init).reshape(-1)[i])
            for j in range(self.nu):
                mp.sigma_inv[i * self.nu + j] = float(sinv[i, j])
                mp.sigma_chol[i * self.nu + j] = float(chol[i, j])
        ro = d.rollout
        ro.env = _lib.ENV_IDS[self.running_cost.env_name]
        ro.state_constraint = int(self.running_cost.state_constraint)
        ro.goal_x = float(self.running_cost.goal_x)
        ro.dynamics = self.F.kind
        ro.delay = int(self.F.delay)
        ro.dt = float(self.F.dt)
        d.nx, d.n_shards, d.shard_index = self.nx, n_shards, shard_index
        d.math_mode = _lib.MATH_MODES[self.math_mode]
        d.keep_states = int(self.keep_states)
        d.seed = self.seed
        model_h = None
        if isinstance(self.F, NLDynamics):
            if self.F.model._cuda_device is None:
                self.F.model._cuda_device = self.d
            model_h = self.F.model.set_prediction_time(self.F.dt)
        return d, model_h

    def _ensure(self, B):
        """The device planner for a B-entry action buffer.  The packed model is re-fetched on EVERY call: the model
        rebuilds its handle when a parameter changed (``load_state_dict``, an optimizer step) and re-folds its
        constants when ``forward`` ran at another prediction time, and the planner must never roll out on a stale
        or re-folded handle - so the prediction time is folded back to this planner's ``dt`` and the planner handle
        is recreated when the model handle is a new one."""
        model_h = None
        if isinstance(self.F, NLDynamics):
            if self.F.model._cuda_device is None:
                self.F.model._cuda_device = self.d
            model_h = self.F.model.set_prediction_time(self.F.dt)
        key = None if model_h is None else model_h.value
        if self._handle is not None and self._handle_B == B and self._handle_model == key:
            return self._handle
        self._destroy()
        d, model_h = self._desc(B, self.K_local, self.k_offset, self.K, self.G, self.rank)
        h = C.c_void_p()
        _lib.check(self._lib.nlc_planner_create(C.byref(h), model_h, C.byref(d), self.d.index), "nlc_planner_create")
        self._handle, self._handle_B, self._views = h, B, {}
        self._handle_model = None if model_h is None else model_h.value
        self._U_dirty = True
        self._exchange = False
        if self.G > 1 and self.process_group is not None:
            self._connect_exchange(h)
        return self._handle

    # ---- device-side exchange of the shard triples (include/nlc_b200.h: nlc_planner_exchange_*) ----------------------------
    def _connect_exchange(self, h):
        """Map every rank's mailbox into this process through CUDA IPC (one all-gather of the 64-byte handles, at handle
        creation only).  From then on a control step exchanges the triples on the device and is ONE graph launch.  If any
        rank cannot map a peer (no P2P between the GPUs, ``NLC_NO_DEVICE_EXCHANGE=1``) every rank falls back to the
        all-gather of ``sharding.gather_triples``.  Collective: every rank of the group creates its handle at the same call."""
        import os

        import torch.distributed as dist

        backend = dist.get_backend(self.process_group)
        cdev = self.d if backend == "nccl" else torch.device("cpu")
        mine = (C.c_char * 64)()
        want = os.environ.get("NLC_NO_DEVICE_EXCHANGE", "0") != "1"
        if want:
            want = self._lib.nlc_planner_exchange_export(h, mine, None) == _lib.NLC_OK
        allh = torch.zeros(self.G * 64, dtype=torch.uint8, device=cdev)
        dist.all_gather_into_tensor(allh, torch.frombuffer(bytearray(bytes(mine)), dtype=torch.uint8).to(cdev), group=self.process_group)
        ok = torch.tensor([1 if want else 0], dtype=torch.int32, device=cdev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.process_group)
        if int(ok) == 1:
            buf = allh.cpu().numpy().tobytes()
            ok[0] = 1 if self._lib.nlc_planner_exchange_connect(h, 0, buf) == _lib.NLC_OK else 0
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.process_group)
        if int(ok) == 1:
            self._exchange = True
        else:
            # a half-connected group would deadlock in the device-side poll: drop the handle and keep the collective path
            # (a connected handle cannot be disconnected, so it is rebuilt; nothing has been planned with it yet)
            d, model_h = self._desc(self._handle_B, self.K_local, self.k_offset, self.K, self.G, self.rank)
            self._lib.nlc_planner_destroy(h)
            h2 = C.c_void_p()
            _lib.check(self._lib.nlc_planner_create(C.byref(h2), model_h, C.byref(d), self.d.index), "nlc_planner_create")
            self._handle = h2
        return self._exchange

    @staticmethod
    def connect_local_shards(planners, action_buffer_size=4):
        """Shards of one plan living in ONE process (``shard=(rank, G)``; single-GPU tests of the sharded step): connect their
        mailboxes by device pointer.  The caller then drives ``_begin`` on every shard before any ``_finish``."""
        ptrs = []
        for p in planners:
            h = p._ensure(action_buffer_size)
            ptr = C.c_void_p()
            _lib.check(p._lib.nlc_planner_exchange_export(h, None, C.byref(ptr)), "nlc_planner_exchange_export")
            ptrs.append(ptr.value)
        arr = (C.c_void_p * len(ptrs))(*ptrs)
        for p in planners:
            _lib.check(p._lib.nlc_planner_exchange_connect(p._handle, 1, arr), "nlc_planner_exchange_connect")
            p._exchange = True

    def exchange_status(self):
        """(connected, status): device-side exchange in use, and 2 if a poll for a peer's triple gave up."""
        if self._handle is None:
            return False, 0
        a, b = C.c_int(), C.c_int()
        _lib.check(self._lib.nlc_planner_exchange_status(self._handle, C.byref(a), C.byref(b)), "nlc_planner_exchange_status")
        return bool(a.value), int(b.value)

    def _destroy(self):
        if self._handle is not None:
            self._sync_U_to_host()
            self._lib.nlc_planner_destroy(self._handle)
            self._handle = None
            self._views = {}

    def __del__(self):
        try:
            if self._handle is not None:
                self._lib.nlc_planner_destroy(self._handle)
        except Exception:
            pass

    def _buf(self, which, shape):
        """fp32 CUDA tensor aliasing one of the planner's device buffers."""
        key = (which, tuple(shape))
        if key not in self._views:
            p, n = C.c_void_p(), C.c_int64()
            _lib.check(self._lib.nlc_planner_buffer(self._handle, which, C.byref(p), C.byref(n)), "nlc_planner_buffer")
            if p.value is None or n.value == 0:
                return None
            assert int(np.prod(shape)) == n.value, (which, shape, n.value)
            self._views[key] = torch.as_tensor(_DevView(p.value, shape), device=self.d)
        return self._views[key]

    def _sync_U_to_host(self):
        if self._handle is not None and not self._U_dirty:
            arr = np.empty(self.T * self.nu, dtype=np.float64)
            _lib.check(self._lib.nlc_planner_get_U(self._handle, arr.ctypes.data_as(C.POINTER(C.c_double))), "nlc_planner_get_U")
            self._U_host = torch.from_numpy(arr).reshape(self.T, self.nu).clone()

    def _push_U(self):
        if self._U_dirty:
            ptr, keep = _lib.as_double_array(self._U_host.numpy())
            _lib.check(self._lib.nlc_planner_set_U(self._handle, ptr), "nlc_planner_set_U")
            self._U_dirty = False

    # ---- the reference's attributes ------------------------------------------------------------------------------
    @property
    def U(self):
        if self._handle is None or self._U_dirty:
            return self._U_host.to(self.dtype)
        return self._buf(_lib.BUF_U, (self.T, self.nu))

    @U.setter
    def U(self, value):
        self._U_host = torch.as_tensor(value).detach().to("cpu", torch.float64).reshape(self.T, self.nu).clone()
        self._U_dirty = True

    def _after(self, which, shape):
        if self._handle is None or self._calls == 0:
            return None
        return self._buf(which, shape)

    _calls = 0
    noise = property(lambda self: self._after(_lib.BUF_NOISE, (self.K_local, self.T, self.nu)))
    perturbed_action = property(lambda self: self._after(_lib.BUF_PERTURBED, (self.K_local, self.T, self.nu)))
    cost_total = property(lambda self: self._after(_lib.BUF_COST_TOTAL, (self.K_local,)))
    states = property(lambda self: self._after(_lib.BUF_STATES, (self.K_local, self.T, self.nx)) if self.keep_states else None)
    actions = property(lambda self: self._after(_lib.BUF_ACTIONS, (self.K_local, self.T, self.nu)))

    @property
    def cost_total_non_zero(self):
        """exp(-(c - beta)/lambda) with the GLOBAL beta (mppi_delay.py:210-211) for this shard's samples."""
        if self._handle is None or self._calls == 0:
            return None
        w = self._buf(_lib.BUF_WEIGHTS, (self.K_local,))
        beta_local = self._buf(_lib.BUF_TRIPLE, (2 + self.T * self.nu,))[0]
        beta = self._buf(_lib.BUF_STATS, (2,))[0]
        return w * torch.exp(-(beta_local - beta) / self.lambda_)

    @property
    def omega(self):
        nz = self.cost_total_non_zero
        return None if nz is None else nz / self._buf(_lib.BUF_STATS, (2,))[1]

    # ---- MPPIDelay.command ---------------------------------------------------------------------------------------
    def _injected_noise(self):
        """The reference's tests inject noise by replacing ``noise_dist.sample`` (instance attribute)."""
        fn = self.noise_dist.__dict__.get("sample")
        if fn is None:
            return None
        nz = torch.as_tensor(fn((self.K, self.T)))
        if tuple(nz.shape) != (self.K, self.T, self.nu):
            raise ValueError(f"injected noise must have shape {(self.K, self.T, self.nu)}, got {tuple(nz.shape)}")
        nz = nz[self.k_offset:self.k_offset + self.K_local]  # bit-exact sample indexing: global k = offset + local k
        return nz.to(device=self.d, dtype=torch.float32).contiguous()

    def command(self, state, action_buffer):
        """:param state: (nx) or (K x nx) current state; :param action_buffer: (B x nu) past actions, env units.
        :returns action: (nu) best action (``mppi_delay.py:193-224``)."""
        action = self._begin(state, action_buffer)
        if action is not None:  # single shard, host or planner-owned inputs: the whole step was one graph launch
            return self._first_actions(action)
        if self.G > 1 and not self._exchange:
            if self.process_group is None:
                raise RuntimeError("a planner built with shard=(rank, G) has no process group to exchange the triples: "
                                   "drive it through _begin / all_triples / _finish")
            sharding.gather_triples(self.shard_triple, self.all_triples, group=self.process_group)
        return self._first_actions(self._finish())

    def _first_actions(self, action):
        """``U[:u_per_command] * u_scale`` (``mppi_delay.py:217-224``): the head action for ``u_per_command == 1``, else the first
        ``u_per_command`` planned actions as a ``(u_per_command, nu)`` tensor."""
        if self.u_per_command == 1:
            return action
        n = int(self.u_per_command)
        return (self._buf(_lib.BUF_U, (self.T, self.nu))[:n] * float(self.u_scale)).to(self.dtype)

    # The control step of a shard in its two halves; the exchange of the triples sits between them (the parity tests
    # drive the G shards of one plan through these on a single GPU).
    def _begin(self, state, action_buffer):
        """Stages 1-3 and the shard-local half of stage 4: fills ``shard_triple`` = (beta_g, eta_g, W_g[T][nu]).
        Returns the action when the fused single-shard path ran the whole step, else None."""
        action_buffer = torch.as_tensor(action_buffer)
        if self.encode_obs_time:
            action_buffer = action_buffer[:, :self.nu]  # the time column is not read by the analytic dynamics (oracle.py:23)
        B = action_buffer.shape[0]
        h = self._ensure(B)
        self._push_U()
        if not torch.is_tensor(state):
            state = torch.tensor(np.asarray(state))
        self.state = state.to(dtype=self.dtype)
        noise = self._injected_noise()
        stream = _lib.current_stream_ptr()
        per_sample = state.dim() == 2 and state.shape[0] != 1
        self.last_action_host = None
        with self._on_device():
            if (not per_sample and noise is None and (self.G == 1 or (self._exchange and self.process_group is not None))
                    and not state.is_cuda and not action_buffer.is_cuda):
                # lowest-latency path: host buffers straight through the C ABI
                sp, k1 = _lib.as_double_array(state.detach().reshape(-1).numpy())
                bp, k2 = _lib.as_double_array(action_buffer.detach().reshape(-1).numpy())
                out = np.empty(self.nu, dtype=np.float64)
                _lib.check(self._lib.nlc_planner_command_host(h, sp, bp, None, out.ctypes.data_as(C.POINTER(C.c_double)), stream),
                           "nlc_planner_command_host")
                self._calls += 1
                # the action already crossed PCIe inside the call: it is kept on the object for callers that want the host
                # value (mppi_with_model.py:262 moves it to numpy at once); the returned tensor is the planner's own
                # device-resident copy, cast like the reference's - no second transfer either way
                self.last_action_host = out
                return self._buf(_lib.BUF_ACTION, (self.nu,)).to(self.dtype)
            st = self._buf(_lib.BUF_STATE, (self.K_local, self.nx))
            if per_sample:
                if state.shape[0] != self.K:
                    raise ValueError("per-sample states must have K rows")
                st.copy_(state[self.k_offset:self.k_offset + self.K_local].to(device=self.d, dtype=torch.float32))
            else:
                st[0].copy_(state.reshape(-1).to(device=self.d, dtype=torch.float32))
            ab = self._buf(_lib.BUF_ACTION_BUFFER, (B, self.nu))
            ab.copy_(action_buffer.reshape(B, self.nu).to(device=self.d, dtype=torch.float32))
            if (self.G == 1 or (self._exchange and self.process_group is not None)) and noise is None and not per_sample:
                # fixed launch sequence on the planner's own buffers: one CUDA-graph launch (nlc_planner_step); with
                # connected shards the exchange of the triples is part of the graph
                _lib.check(self._lib.nlc_planner_step(h, stream), "nlc_planner_step")
                self._calls += 1
                return self._buf(_lib.BUF_ACTION, (self.nu,)).to(self.dtype)
            _lib.check(self._lib.nlc_planner_rollout(h, st.data_ptr(), int(per_sample), ab.data_ptr(), _lib.ptr(noise), stream),
                       "nlc_planner_rollout")
        return None

    # ---- device-resident inputs: the control loop of a caller that keeps the state on the GPU ---------------------------------
    def set_inputs(self, state, action_buffer):
        """Copy ``state`` (nx) and ``action_buffer`` (B x nu, env units) into the planner's own device buffers; :meth:`step`
        then plans on them.  (The batched closed loop and the benchmarks keep both on the device between control steps.)"""
        action_buffer = torch.as_tensor(action_buffer)
        if self.encode_obs_time:
            action_buffer = action_buffer[:, :self.nu]
        B = action_buffer.shape[0]
        self._ensure(B)
        self._push_U()
        state = torch.as_tensor(np.asarray(state)) if not torch.is_tensor(state) else state
        self.state = state.to(dtype=self.dtype)
        self._buf(_lib.BUF_STATE, (self.K_local, self.nx))[0].copy_(state.reshape(-1).to(device=self.d, dtype=torch.float32))
        self._buf(_lib.BUF_ACTION_BUFFER, (B, self.nu)).copy_(action_buffer.reshape(B, self.nu).to(device=self.d, dtype=torch.float32))

    def step(self):
        """One control step on the inputs resident in the planner's buffers (``set_inputs``), on-device sampler: ONE CUDA-graph
        launch (``nlc_planner_step``), nothing else on the host.  Returns the planner's own device-resident action (fp32
        view, valid until the next step).  Single shard, or shards connected by the device-side exchange."""
        if self._handle is None:
            raise RuntimeError("call set_inputs first")
        if self.G > 1 and not self._exchange:
            raise RuntimeError("step() needs a single shard or device-connected shards")
        with self._on_device():
            _lib.check(self._lib.nlc_planner_step(self._handle, _lib.current_stream_ptr()), "nlc_planner_step")
        self._calls += 1
        return self._buf(_lib.BUF_ACTION, (self.nu,))

    def _on_device(self):
        """Context that makes the planner's device current - a no-op object when it already is (the torch context manager
        costs ~10 us per control step)."""
        return _NULL_CTX if torch.cuda.current_device() == self.d.index else torch.cuda.device(self.d)

    def _finish(self):
        """Log-sum-exp combine of ``all_triples`` (G > 1) or of the own triple, ``U`` update, action."""
        with self._on_device():
            _lib.check(self._lib.nlc_planner_finish(self._handle, _lib.current_stream_ptr()), "nlc_planner_finish")
        self._calls += 1
        return self._buf(_lib.BUF_ACTION, (self.nu,)).to(self.dtype)

    def overlap_status(self):
        """(overlapped, status): whether this planner runs its history encoder beside the rollout kernel (plans within
        half a wave of 128-sample tiles), and 1 if the last control step's rollout timed out waiting for the encoder."""
        if self._handle is None:
            return False, 0
        a, b = C.c_int(), C.c_int()
        _lib.check(self._lib.nlc_planner_overlap_status(self._handle, C.byref(a), C.byref(b)), "nlc_planner_overlap_status")
        return bool(a.value), int(b.value)

    @property
    def shard_triple(self):
        return self._buf(_lib.BUF_TRIPLE, (2 + self.T * self.nu,))

    @property
    def all_triples(self):
        return self._buf(_lib.BUF_ALL_TRIPLES, (self.G, 2 + self.T * self.nu))

    def reset(self):
        """Clear controller state after finishing a trial (``mppi_delay.py:226-230``)."""
        self.U = self._replicated(self.noise_dist.sample((self.T,)))

    def get_rollouts(self, state, num_rollouts=1):
        """Nominal rollout of the planned sequence ``U`` (``mppi_delay.py:358-381``): ``states[:, t+1] =
        F(states[:, t], u_scale * U[t])``, returns ``(num_rollouts, T, nx)``.

        As in the reference, the dynamics receive a single ``(n, nu)`` action here, not a B-entry history window;
        ``NeuralLaplaceModel.forward`` turns that into a window of length one (``w_nl.py:131-132``), so the encoder
        sees the current action only.  The analytic delay dynamics index ``action[:, -(delay+1)]`` on that 2-D tensor
        in the reference (``oracle.py:23``) - an action component, not a time step - so they raise here.
        ``U[t].view(num_rollouts, -1)`` (``:377``) only has a meaning for ``num_rollouts == 1``; for more rollouts every
        row gets the same action (what the reference's docstring describes)."""
        if not isinstance(self.F, NLDynamics):
            raise NotImplementedError("get_rollouts passes one action, not a history window: only the Neural Laplace "
                                      "closure can consume it (oracle.py:23 indexes a window)")
        n = int(num_rollouts)
        state = torch.as_tensor(state).reshape(-1, self.nx)
        if state.shape[0] == 1:
            state = state.repeat(n, 1)
        if state.shape[0] != n:
            raise ValueError("state must be (nx) or (num_rollouts, nx)")
        model = self.F.model
        if model._cuda_device is None:
            model._cuda_device = self.d
        mh = model.set_prediction_time(self.F.dt)
        U = self.U.to(device=self.d, dtype=torch.float32).reshape(self.T, self.nu)
        hist = (float(self.u_scale) * U).reshape(1, self.T, self.nu).repeat(n, 1, 1).contiguous()  # B = 1: L = T
        st = state.to(device=self.d, dtype=torch.float32).contiguous()
        p = torch.empty((n, self.T, 2), dtype=torch.float32, device=self.d)
        cost = torch.empty((n,), dtype=torch.float32, device=self.d)
        states = torch.empty((n, self.T, self.nx), dtype=torch.float32, device=self.d)
        ro = _lib.RolloutOpts()
        ro.env, ro.state_constraint, ro.goal_x = _lib.ENV_IDS[self.running_cost.env_name], 0, 0.0
        ro.dynamics, ro.delay, ro.dt = self.F.kind, 0, float(self.F.dt)
        fp32 = _lib.MATH_MODES["fp32"]  # a handful of rows: the CUDA-core kernels (the tensor-core encoder needs B >= 2)
        with torch.cuda.device(self.d):
            stream = _lib.current_stream_ptr()
            _lib.check(self._lib.nlc_encode_history(mh, hist.data_ptr(), n, self.T, 1, p.data_ptr(), fp32, stream), "nlc_encode_history")
            _lib.check(self._lib.nlc_rollout_cost(mh, C.byref(ro), st.data_ptr(), 1, p.data_ptr(), hist.data_ptr(), None, n, self.T, 1,
                                                  self.nu, cost.data_ptr(), states.data_ptr(), fp32, stream), "nlc_rollout_cost")
        return states.to(self.dtype)


class _MPPIDelayF64(MPPIDelay):
    """``MPPIDelay(..., math_mode="fp64")``: the control step on the fp64 planner handle (``nlc_planner_f64_*``), single shard,
    direct launches on the current stream (host inputs: one C call that copies in, plans and copies the action back)."""

    def __init__(self, *args, process_group=None, shard=None, **kw):
        if process_group is not None or shard is not None:
            raise NotImplementedError("math_mode='fp64' plans on one GPU: K sharding (process_group / shard) is not implemented")
        super().__init__(*args, **kw)
        self._params_key = None
        self._params_dev = None

    def _desc_f64(self, B):
        d = _lib.PlannerF64Desc()
        b = d.base
        mp = b.mppi
        mp.K, mp.T, mp.nu, mp.B, mp.k_offset, mp.k_total = self.K, self.T, self.nu, B, 0, self.K
        mp.has_bounds = int(self._bounds is not None)
        mp.sample_null_action, mp.noise_abs_cost = int(self.sample_null_action), int(self.noise_abs_cost)
        ro = b.rollout
        ro.env = _lib.ENV_IDS[self.running_cost.env_name]
        ro.state_constraint, ro.dynamics, ro.delay = int(self.running_cost.state_constraint), self.F.kind, int(self.F.delay)
        b.nx, b.n_shards, b.shard_index, b.keep_states, b.seed = self.nx, 1, 0, int(self.keep_states), self.seed
        d.lambda_, d.u_scale, d.dt, d.goal_x = float(self.lambda_), float(self.u_scale), float(self.F.dt), float(self.running_cost.goal_x)
        if self._bounds is not None:
            for i in range(self.nu):
                d.u_min[i], d.u_max[i] = self._bounds[0][i], self._bounds[1][i]
        sinv = self.noise_sigma_inv.to(torch.float64).reshape(self.nu, self.nu)
        chol = torch.linalg.cholesky(self.noise_sigma.to(torch.float64).reshape(self.nu, self.nu))
        for i in range(self.nu):
            d.noise_mu[i] = float(self.noise_mu.reshape(-1)[i])
            d.u_init[i] = float(torch.as_tensor(self.u_init).reshape(-1)[i])
            for j in range(self.nu):
                d.sigma_inv[i * self.nu + j], d.sigma_chol[i * self.nu + j] = float(sinv[i, j]), float(chol[i, j])
        return d

    def _ensure(self, B):
        """The fp64 planner for a B-entry action buffer, rebuilt when the model's handle is a new one (its buffers or device
        changed); its weights come separately (``_push_params``)."""
        model_h = None
        if isinstance(self.F, NLDynamics):
            if self.F.model._cuda_device is None:
                self.F.model._cuda_device = self.d
            with self._on_device():
                model_h = self.F.model._handle_f64()
        key = None if model_h is None else model_h.value
        if self._handle is not None and self._handle_B == B and self._handle_model == key:
            return self._handle
        self._destroy()
        h = C.c_void_p()
        _lib.check(self._lib.nlc_planner_f64_create(C.byref(h), model_h, C.byref(self._desc_f64(B)), self.d.index), "nlc_planner_f64_create")
        self._handle, self._handle_B, self._handle_model, self._views = h, B, key, {}
        self._U_dirty = True
        self._params_key = None
        return h

    def _push_params(self, h, stream):
        """The model's parameters as one flat fp64 tensor (named_parameters() order, the ``_forward_f64`` layout), sent only
        when they changed since the last control step."""
        if not isinstance(self.F, NLDynamics):
            return
        model = self.F.model
        key = model._fingerprint()
        if key == self._params_key:
            return
        params = torch.cat([p.detach().reshape(-1) for p in model.parameters()]).to(device=self.d, dtype=torch.float64)
        _lib.check(self._lib.nlc_planner_f64_set_params(h, params.data_ptr(), stream), "nlc_planner_f64_set_params")
        self._params_dev, self._params_key = params, key

    def _destroy(self):
        if self._handle is not None:
            self._sync_U_to_host()
            self._lib.nlc_planner_f64_destroy(self._handle)
            self._handle = None
            self._views = {}

    def __del__(self):
        try:
            if self._handle is not None:
                self._lib.nlc_planner_f64_destroy(self._handle)
        except Exception:
            pass

    def _buf(self, which, shape):
        """fp64 CUDA tensor aliasing one of the fp64 planner's device buffers."""
        key = (which, tuple(shape))
        if key not in self._views:
            p, n = C.c_void_p(), C.c_int64()
            _lib.check(self._lib.nlc_planner_f64_buffer(self._handle, which, C.byref(p), C.byref(n)), "nlc_planner_f64_buffer")
            if p.value is None or n.value == 0:
                return None
            assert int(np.prod(shape)) == n.value, (which, shape, n.value)
            self._views[key] = torch.as_tensor(_DevView(p.value, shape, "<f8"), device=self.d)
        return self._views[key]

    def _sync_U_to_host(self):
        if self._handle is not None and not self._U_dirty:
            arr = np.empty(self.T * self.nu, dtype=np.float64)
            _lib.check(self._lib.nlc_planner_f64_get_U(self._handle, arr.ctypes.data_as(C.POINTER(C.c_double))), "nlc_planner_f64_get_U")
            self._U_host = torch.from_numpy(arr).reshape(self.T, self.nu).clone()

    def _push_U(self):
        if self._U_dirty:
            ptr, keep = _lib.as_double_array(self._U_host.numpy())
            _lib.check(self._lib.nlc_planner_f64_set_U(self._handle, ptr), "nlc_planner_f64_set_U")
            self._U_dirty = False

    @property
    def cost_total_non_zero(self):
        """exp(-(1/lambda)(c - beta)) (mppi_delay.py:210-211)."""
        return self._after(_lib.BUF_WEIGHTS, (self.K,))

    @property
    def omega(self):
        nz = self.cost_total_non_zero
        return None if nz is None else (1.0 / self._buf(_lib.BUF_STATS, (2,))[1]) * nz

    def _injected_noise(self):
        fn = self.noise_dist.__dict__.get("sample")
        if fn is None:
            return None
        nz = torch.as_tensor(fn((self.K, self.T)))
        if tuple(nz.shape) != (self.K, self.T, self.nu):
            raise ValueError(f"injected noise must have shape {(self.K, self.T, self.nu)}, got {tuple(nz.shape)}")
        return nz.to(device=self.d, dtype=torch.float64).contiguous()

    def command(self, state, action_buffer):
        """:param state: (nx) or (K x nx) current state; :param action_buffer: (B x nu) past actions, env units.
        :returns action: (nu) best action (``mppi_delay.py:193-224``), ``(u_per_command, nu)`` for ``u_per_command > 1``."""
        action_buffer = torch.as_tensor(action_buffer)
        if self.encode_obs_time:
            action_buffer = action_buffer[:, :self.nu]  # the time column is not read by the analytic dynamics (oracle.py:23)
        B = action_buffer.shape[0]
        h = self._ensure(B)
        self._push_U()
        if not torch.is_tensor(state):
            state = torch.tensor(np.asarray(state))
        self.state = state.to(dtype=self.dtype)
        noise = self._injected_noise()
        per_sample = state.dim() == 2 and state.shape[0] != 1
        with self._on_device():
            stream = _lib.current_stream_ptr()
            self._push_params(h, stream)
            if not per_sample and noise is None and not state.is_cuda and not action_buffer.is_cuda:
                sp, k1 = _lib.as_double_array(state.detach().reshape(-1).numpy())
                bp, k2 = _lib.as_double_array(action_buffer.detach().reshape(-1).numpy())
                out = np.empty(self.nu, dtype=np.float64)
                _lib.check(self._lib.nlc_planner_f64_command_host(h, sp, bp, out.ctypes.data_as(C.POINTER(C.c_double)), stream),
                           "nlc_planner_f64_command_host")
                self.last_action_host = out
            else:
                if per_sample and state.shape[0] != self.K:
                    raise ValueError("per-sample states must have K rows")
                st = (state if per_sample else state.reshape(-1)).to(device=self.d, dtype=torch.float64).contiguous()
                ab = action_buffer.reshape(B, self.nu).to(device=self.d, dtype=torch.float64).contiguous()
                _lib.check(self._lib.nlc_planner_f64_command(h, st.data_ptr(), int(per_sample), ab.data_ptr(), _lib.ptr(noise), stream),
                           "nlc_planner_f64_command")
                self.last_action_host = None
        self._calls += 1
        return self._first_actions(self._buf(_lib.BUF_ACTION, (self.nu,)).to(self.dtype, copy=True))

    def _unsupported(self, what):
        raise NotImplementedError(f"{what} is not implemented for math_mode='fp64' (single-GPU command() only)")

    def set_inputs(self, state, action_buffer):
        self._unsupported("set_inputs / step (the resident-input graph step)")

    def step(self):
        self._unsupported("set_inputs / step (the resident-input graph step)")

    def get_rollouts(self, state, num_rollouts=1):
        self._unsupported("get_rollouts")

    def _begin(self, state, action_buffer):
        self._unsupported("the sharded control step")

    def _finish(self):
        self._unsupported("the sharded control step")

    def overlap_status(self):
        return False, 0

    def exchange_status(self):
        return False, 0

    shard_triple = property(lambda self: self._unsupported("the sharded control step"))
    all_triples = property(lambda self: self._unsupported("the sharded control step"))

"""``NeuralLaplaceModel`` with the reference's constructor, ``state_dict`` layout and ``forward`` signature
(``w_nl.py:66-145``), evaluated by the CUDA kernels of ``libnlc_b200.so``.

The ``torch.nn`` sub-modules below only HOLD parameters under the reference's key names
(``action_encoder.gru.*``, ``action_encoder.linear_out.*``, ``laplace_rep_func.linear_tanh_stack.{0,2,4}.*``),
so reference checkpoints load unchanged and random init under a seed matches the reference module's.
They are never called: ``forward`` packs the weights into a device handle and launches the kernels.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from . import _lib


class _EncoderParams(nn.Module):
    """Parameter container for ReverseGRUEncoder (w_nl.py:14-23)."""

    def __init__(self, dimension_in, latent_dim, hidden_units, encode_obs_time):
        super().__init__()
        if encode_obs_time:
            dimension_in += 1
        self.gru = nn.GRU(dimension_in, hidden_units, 2, batch_first=True)
        self.linear_out = nn.Linear(hidden_units, latent_dim)
        nn.init.xavier_uniform_(self.linear_out.weight)


class _RepFuncParams(nn.Module):
    """Parameter container for LaplaceRepresentationFunc (w_nl.py:35-53)."""

    def __init__(self, s_dim, output_dim, latent_dim, hidden_units):
        super().__init__()
        self.linear_tanh_stack = nn.Sequential(
            nn.Linear(s_dim * 2 + latent_dim, hidden_units), nn.Tanh(),
            nn.Linear(hidden_units, hidden_units), nn.Tanh(),
            nn.Linear(hidden_units, s_dim * 2 * output_dim),
        )
        for m in self.linear_tanh_stack.modules():
            if isinstance(m, nn.Linear):
                nn.init.xavier_uniform_(m.weight)


class NeuralLaplaceModel(nn.Module):
    def __init__(self, state_dim, action_dim, latent_dim, hidden_units=64, s_recon_terms=33, ilt_algorithm="fourier",
                 encode_obs_time=False, state_mean=None, state_std=None, action_mean=None, action_std=None,
                 normalize=False, normalize_time=False, dt=0.05, device=None, math_mode="tc_split3"):
        super().__init__()
        if ilt_algorithm != "fourier":
            raise NotImplementedError("only ilt_algorithm='fourier' is on this path (w_nl.py:86-88 'cme' is not)")
        if hidden_units not in (64, 128):
            raise NotImplementedError("the kernels are built for hidden_units = 128 (config.py:37) and 64 (the class default, "
                                      "w_nl.py:71; fp32 CUDA-core kernels only)")
        self.ilt_algorithm = ilt_algorithm
        self.latent_dim = latent_dim
        self.action_encoder = _EncoderParams(action_dim, 2, hidden_units // 2, encode_obs_time)
        self.laplace_rep_func = _RepFuncParams(s_recon_terms, state_dim, state_dim + 2, hidden_units)
        self.encode_obs_time = encode_obs_time
        self.output_dim = state_dim
        self.action_dim = action_dim
        self.hidden_units = hidden_units
        self.normalize = normalize
        self.normalize_time = normalize_time
        self.s_recon_terms = s_recon_terms
        self.math_mode = math_mode
        for name, val in (("state_mean", state_mean), ("state_std", state_std), ("action_mean", action_mean),
                          ("action_std", action_std), ("dt", dt)):
            # torch.tensor(...) exactly as w_nl.py:107-111 (dt becomes an fp32 buffer there; .double() keeps that value)
            self.register_buffer(name, torch.tensor(val if val is not None else 0.0))
        self._cuda_device = torch.device(device) if device is not None else None
        self._handle = None
        self._handle_key = None
        self._handle_bkey = None
        self._handle_ts = None

    # ---- device handle -------------------------------------------------------------------------------------------
    def _fingerprint(self):
        """(version, address) of every parameter and buffer: changes on ``load_state_dict``, optimizer steps, ``.double()`` ...
        The tensor list is cached (walking the module tree costs ~60 us, this runs once per control step) and dropped whenever
        a tensor attribute is (re)assigned or ``_apply`` (``.to`` / ``.double`` / ``.cuda``) runs."""
        ts = self.__dict__.get("_fp_tensors")
        if ts is None:
            ts = [v for _, v in self.state_dict(keep_vars=True).items()]
            self.__dict__["_fp_tensors"] = ts
        return tuple((v._version, v.data_ptr()) for v in ts)

    def _buffer_key(self):
        """(version, address) of the buffers (state_mean, state_std, action_mean, action_std, dt) and the device: all of the
        handle that math_mode="fp64" reads, whose weights come per call."""
        bs = self.__dict__.get("_fp_buffers")
        if bs is None:
            bs = list(self.buffers())
            self.__dict__["_fp_buffers"] = bs
        return tuple((v._version, v.data_ptr()) for v in bs), str(self._device())

    def _apply(self, fn, *a, **k):
        self.__dict__["_fp_buffers"] = None
        self.__dict__["_fp_tensors"] = None
        for m in self.modules():
            m.__dict__["_fp_tensors"] = None
        return super()._apply(fn, *a, **k)

    def __setattr__(self, name, value):
        if isinstance(value, (torch.Tensor, nn.Module)):
            self.__dict__["_fp_tensors"] = None
            self.__dict__["_fp_buffers"] = None
        super().__setattr__(name, value)

    def _device(self):
        if self._cuda_device is not None:
            return self._cuda_device
        p = next(self.parameters())
        if p.is_cuda:
            return p.device
        if not torch.cuda.is_available():
            raise RuntimeError("neurallaplacecontrol_b200 needs a CUDA device (sm_100); there is no CPU fallback")
        return torch.device("cuda", torch.cuda.current_device())

    def handle(self):
        """The packed device model (rebuilt when any parameter or buffer changed)."""
        key = (self._fingerprint(), str(self._device()))
        if self._handle is not None and key == self._handle_key:
            return self._handle
        self._free()
        lib = _lib.load()
        sd = {k: v.detach().to("cpu", torch.float64).contiguous().numpy() for k, v in self.state_dict().items()}
        keep = []

        def dp(name):
            a = np.ascontiguousarray(sd[name].reshape(-1))
            keep.append(a)
            return a.ctypes.data_as(C.POINTER(C.c_double))

        d = _lib.ModelDesc()
        d.state_dim, d.action_dim, d.hidden_units, d.s_terms = self.output_dim, self.action_dim, self.hidden_units, self.s_recon_terms
        d.encode_obs_time, d.normalize, d.normalize_time = int(self.encode_obs_time), int(self.normalize), int(self.normalize_time)
        d.action_std_len = int(sd["action_std"].size)
        d.dt = float(sd["dt"])
        d.state_mean, d.state_std = dp("state_mean"), dp("state_std")
        d.action_mean, d.action_std = dp("action_mean"), dp("action_std")
        g = "action_encoder.gru."
        d.gru_w_ih_l0, d.gru_w_hh_l0, d.gru_b_ih_l0, d.gru_b_hh_l0 = dp(g + "weight_ih_l0"), dp(g + "weight_hh_l0"), dp(g + "bias_ih_l0"), dp(g + "bias_hh_l0")
        d.gru_w_ih_l1, d.gru_w_hh_l1, d.gru_b_ih_l1, d.gru_b_hh_l1 = dp(g + "weight_ih_l1"), dp(g + "weight_hh_l1"), dp(g + "bias_ih_l1"), dp(g + "bias_hh_l1")
        d.enc_out_w, d.enc_out_b = dp("action_encoder.linear_out.weight"), dp("action_encoder.linear_out.bias")
        s = "laplace_rep_func.linear_tanh_stack."
        d.mlp_w0, d.mlp_b0, d.mlp_w2, d.mlp_b2, d.mlp_w4, d.mlp_b4 = (dp(s + "0.weight"), dp(s + "0.bias"), dp(s + "2.weight"),
                                                                      dp(s + "2.bias"), dp(s + "4.weight"), dp(s + "4.bias"))
        if sd["action_mean"].size != self.action_dim:
            raise ValueError("action_mean must have action_dim entries")
        h = C.c_void_p()
        dev = self._device()
        _lib.check(lib.nlc_model_create(C.byref(h), C.byref(d), dev.index if dev.index is not None else 0), "nlc_model_create")
        self._handle, self._handle_key, self._handle_ts = h, key, float(sd["dt"])
        self._handle_bkey = self._buffer_key()
        return h

    def _handle_f64(self):
        """The handle for math_mode="fp64": any live handle built with the current buffers and device serves, however the
        parameters changed since (an optimizer step does not rebuild it); otherwise ``handle()``."""
        if self._handle is not None and self._handle_bkey == self._buffer_key():
            return self._handle
        return self.handle()

    def _free(self):
        if self._handle is not None:
            _lib.load().nlc_model_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self._free()
        except Exception:
            pass

    def set_prediction_time(self, ts: float):
        """Fold the constants of a fixed prediction time (the planner passes dt, mppi_with_model.py:74)."""
        h = self.handle()
        if self._handle_ts != float(ts):
            _lib.check(_lib.load().nlc_model_set_prediction_time(h, float(ts)), "nlc_model_set_prediction_time")
            self._handle_ts = float(ts)
        return h

    # ---- forward -------------------------------------------------------------------------------------------------
    def forward(self, in_batch_obs, in_batch_action, ts_pred):
        """Predicted state difference, ``w_nl.py:117-145``.  ``in_batch_obs`` (K,nx), ``in_batch_action`` (K,B,nu)
        or (K,nu), ``ts_pred`` (K,1) seconds.  CUDA tensors in, tensor of the input dtype out.

        ``ts_pred`` (K, n_t) with n_t >= 2 predicts at every (sample, time) pair, as the reference's ``laplace_reconstruct``
        does: ``torch.squeeze`` of a (K, n_t, nx) result, each sample's history encoded once (``nlc_model_forward_multi``).

        In grad mode, when a parameter or an input requires grad, the output carries a ``grad_fn`` like the reference
        module's: its backward runs ``nlc_model_backward_ts`` (``nlc_model_backward_multi`` for (K, n_t) times; fp32 CUDA cores).  The forward values are the same either way.

        ``math_mode="fp64"`` runs every form, forward and backward, in fp64 (``nlc_model_forward_f64`` /
        ``nlc_model_backward_f64``), the precision the reference trains in: the parameters go to the kernels per call as one
        flat fp64 tensor, so an optimizer step needs no repacking of the device handle."""
        if torch.is_grad_enabled():
            if torch.is_tensor(ts_pred) and ts_pred.requires_grad:
                raise NotImplementedError("NeuralLaplaceModel: gradients with respect to ts_pred are not provided")
            params = list(self.parameters())
            if in_batch_obs.requires_grad or in_batch_action.requires_grad or any(p.requires_grad for p in params):
                out = _ForwardWithGrad.apply(self, in_batch_obs, in_batch_action, ts_pred, *params)
                return torch.squeeze(out.to(in_batch_obs.dtype))
        out, _ = self._forward_kernels(in_batch_obs, in_batch_action, ts_pred)
        return torch.squeeze(out.to(in_batch_obs.dtype))

    def _inputs(self, in_batch_obs, in_batch_action, ts_pred, dtype=torch.float32):
        dev = self._device()
        obs = in_batch_obs.detach().to(device=dev, dtype=dtype).contiguous()
        act = in_batch_action.detach().to(device=dev, dtype=dtype)
        if act.dim() == 2:
            act = act.unsqueeze(1)
        act = act.contiguous()
        if dtype == torch.float64 and not torch.is_tensor(ts_pred):
            ts_pred = torch.as_tensor(ts_pred, dtype=torch.float64)  # a Python float keeps its fp64 value
        ts = torch.as_tensor(ts_pred).detach().to(device=dev, dtype=torch.float64)
        if ts.dim() == 2 and ts.shape[1] >= 2:  # several times per sample: (K, n_t), a 2-D tensor of its own
            if ts.shape[0] != act.shape[0]:
                raise ValueError(f"ts_pred of shape {tuple(ts.shape)} needs one row of times per sample ({act.shape[0]})")
            return dev, obs, act, ts.contiguous()
        ts = ts.reshape(-1)
        if ts.numel() not in (1, act.shape[0]):
            raise ValueError("ts_pred must hold one time per sample")
        return dev, obs, act, ts

    def _forward_kernels(self, in_batch_obs, in_batch_action, ts_pred):
        """(K, nx) or, for (K, n_t) times, (K, n_t, nx) fp32 output of the forward kernels and the prepared inputs
        (device, obs, act, ts); fp64, and the prepared inputs with the flat parameters, in math_mode="fp64"."""
        if self.math_mode == "fp64":
            return self._forward_f64(in_batch_obs, in_batch_action, ts_pred)
        dev, obs, act, ts = self._inputs(in_batch_obs, in_batch_action, ts_pred)
        K, B = act.shape[0], act.shape[1]
        lib = _lib.load()
        if ts.dim() == 2:
            n_t = ts.shape[1]
            out = torch.empty((K, n_t, self.output_dim), dtype=torch.float32, device=dev)
            p_action = torch.empty((K, 2), dtype=torch.float32, device=dev)
            ts32 = ts.to(torch.float32).contiguous()
            with torch.cuda.device(dev):
                h = self.handle()
                ws = torch.empty(int(lib.nlc_model_forward_multi_workspace_bytes(h, K, n_t, B)), dtype=torch.uint8, device=dev)
                _lib.check(lib.nlc_model_forward_multi(h, obs.data_ptr(), act.data_ptr(), ts32.data_ptr(), K, n_t, B, out.data_ptr(),
                                                       p_action.data_ptr(), ws.data_ptr(), _lib.MATH_MODES[self.math_mode],
                                                       _lib.current_stream_ptr()), "nlc_model_forward_multi")
            self.last_p_action = p_action
            return out, (dev, obs, act, ts)
        out = torch.empty((K, self.output_dim), dtype=torch.float32, device=dev)
        t0 = float(ts[0])
        with torch.cuda.device(dev):
            if bool((ts == ts[0]).all()):
                h = self.set_prediction_time(t0)
                p_action = torch.empty((K, 2), dtype=torch.float32, device=dev)
                _lib.check(lib.nlc_model_forward(h, obs.data_ptr(), act.data_ptr(), K, B, out.data_ptr(), p_action.data_ptr(),
                                                 _lib.MATH_MODES[self.math_mode], _lib.current_stream_ptr()), "nlc_model_forward")
                self.last_p_action = p_action
            else:
                h = self.handle()
                ts32 = ts.to(torch.float32).contiguous()
                scratch = torch.empty((K, 4 + self.hidden_units), dtype=torch.float32, device=dev)
                _lib.check(lib.nlc_model_forward_ts(h, obs.data_ptr(), act.data_ptr(), ts32.data_ptr(), K, B, out.data_ptr(),
                                                    scratch.data_ptr(), _lib.MATH_MODES[self.math_mode], _lib.current_stream_ptr()),
                           "nlc_model_forward_ts")
                self.last_p_action = scratch.view(-1)[:2 * K].view(K, 2)
        return out, (dev, obs, act, ts)

    def _forward_f64(self, in_batch_obs, in_batch_action, ts_pred):
        """``nlc_model_forward_f64``: (K, nx) or (K, n_t, nx) fp64 output and (device, obs, act, ts (K, n_t), flat parameters,
        n_t given) for the backward."""
        dev, obs, act, ts = self._inputs(in_batch_obs, in_batch_action, ts_pred, torch.float64)
        K, B = act.shape[0], act.shape[1]
        multi = ts.dim() == 2
        ts2 = (ts if multi else ts.expand(K).reshape(K, 1)).to(torch.float64).contiguous()  # a uniform time becomes per sample
        n_t = ts2.shape[1]
        # one flat fp64 tensor in named_parameters() order (one host-to-device copy for CPU parameters)
        params = torch.cat([p.detach().reshape(-1) for p in self.parameters()]).to(device=dev, dtype=torch.float64)
        lib = _lib.load()
        out = torch.empty((K, n_t, self.output_dim), dtype=torch.float64, device=dev)
        p_action = torch.empty((K, 2), dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            h = self._handle_f64()
            ws = torch.empty(int(lib.nlc_model_forward_f64_workspace_bytes(h, K, n_t, B)), dtype=torch.uint8, device=dev)
            _lib.check(lib.nlc_model_forward_f64(h, params.data_ptr(), obs.data_ptr(), act.data_ptr(), ts2.data_ptr(), K, n_t, B,
                                                 out.data_ptr(), p_action.data_ptr(), ws.data_ptr(), _lib.current_stream_ptr()),
                       "nlc_model_forward_f64")
        self.last_p_action = p_action
        return (out if multi else out.view(K, self.output_dim)), (dev, obs, act, ts2, params, multi)

    def _backward_f64(self, prepared, grad_out, need_obs, need_act):
        dev, obs, act, ts, params, multi = prepared
        K, B, n_t = act.shape[0], act.shape[1], ts.shape[1]
        lib = _lib.load()
        g = grad_out.detach().to(device=dev, dtype=torch.float64).reshape(K, n_t, self.output_dim).contiguous()
        grad_params = torch.empty_like(params)
        g_obs = torch.empty_like(obs) if need_obs else None
        g_act = torch.empty_like(act) if need_act else None
        with torch.cuda.device(dev):
            h = self._handle_f64()
            ws = torch.empty(int(lib.nlc_model_backward_f64_workspace_bytes(h, K, n_t, B)), dtype=torch.uint8, device=dev)
            _lib.check(lib.nlc_model_backward_f64(h, params.data_ptr(), obs.data_ptr(), act.data_ptr(), ts.data_ptr(), K, n_t, B,
                                                  g.data_ptr(), grad_params.data_ptr(), _lib.ptr(g_obs), _lib.ptr(g_act),
                                                  ws.data_ptr(), _lib.current_stream_ptr()), "nlc_model_backward_f64")
        return grad_params, g_obs, g_act

    def _backward_kernels(self, prepared, grad_out, need_obs, need_act):
        """fp32 gradients from ``nlc_model_backward_ts`` (``nlc_model_backward_multi`` for (K, n_t) times), fp64 ones from
        ``nlc_model_backward_f64`` when the forward ran in math_mode="fp64": (flat parameter gradients in named_parameters()
        order, each in its state_dict layout; d obs (K, nx) or None; d act (K, B, gin) or None)."""
        if len(prepared) == 6:
            return self._backward_f64(prepared, grad_out, need_obs, need_act)
        dev, obs, act, ts = prepared
        K, B = act.shape[0], act.shape[1]
        lib = _lib.load()
        multi = ts.dim() == 2
        ts32 = (ts if multi else ts.expand(K)).to(torch.float32).contiguous()  # one uniform time becomes a per-sample time
        g = grad_out.detach().to(device=dev, dtype=torch.float32)
        g = (g.reshape(K, ts.shape[1], self.output_dim) if multi else g.reshape(K, self.output_dim)).contiguous()
        with torch.cuda.device(dev):
            h = self.handle()
            n = sum(p.numel() for p in self.parameters())
            grad_params = torch.empty(n, dtype=torch.float32, device=dev)
            g_obs = torch.empty_like(obs) if need_obs else None
            g_act = torch.empty_like(act) if need_act else None
            if multi:
                n_t = ts.shape[1]
                ws = torch.empty(int(lib.nlc_model_backward_multi_workspace_bytes(h, K, n_t, B)), dtype=torch.uint8, device=dev)
                _lib.check(lib.nlc_model_backward_multi(h, obs.data_ptr(), act.data_ptr(), ts32.data_ptr(), K, n_t, B, g.data_ptr(),
                                                        grad_params.data_ptr(), _lib.ptr(g_obs), _lib.ptr(g_act), ws.data_ptr(),
                                                        _lib.current_stream_ptr()), "nlc_model_backward_multi")
            else:
                ws = torch.empty(int(lib.nlc_model_backward_workspace_bytes(h, K, B)), dtype=torch.uint8, device=dev)
                _lib.check(lib.nlc_model_backward_ts(h, obs.data_ptr(), act.data_ptr(), ts32.data_ptr(), K, B, g.data_ptr(),
                                                     grad_params.data_ptr(), _lib.ptr(g_obs), _lib.ptr(g_act), ws.data_ptr(),
                                                     _lib.current_stream_ptr()), "nlc_model_backward_ts")
        return grad_params, g_obs, g_act


class _ForwardWithGrad(torch.autograd.Function):
    """``NeuralLaplaceModel.forward`` as one autograd node: inputs ``(model, obs, act, ts, *parameters)``; the forward
    launches exactly the kernels of the no-grad path, the backward ``nlc_model_backward_ts`` (``nlc_model_backward_multi``
    for (K, n_t) times, whose output and ``grad_out`` are (K, n_t, nx))."""

    @staticmethod
    def forward(ctx, model, obs, act, ts, *params):
        out, prepared = model._forward_kernels(obs, act, ts)
        ctx.model, ctx.prepared = model, prepared
        ctx.obs_meta = (obs.shape, obs.dtype, obs.device)
        ctx.act_meta = (act.shape, act.dtype, act.device)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        model = ctx.model
        need = ctx.needs_input_grad
        grad_params, g_obs, g_act = model._backward_kernels(ctx.prepared, grad_out, need[1], need[2])
        out = [None, None, None, None]
        if g_obs is not None:
            shape, dtype, device = ctx.obs_meta
            out[1] = g_obs.reshape(shape).to(device=device, dtype=dtype)
        if g_act is not None:
            shape, dtype, device = ctx.act_meta
            out[2] = g_act.reshape(shape).to(device=device, dtype=dtype)
        off = 0
        for p, needs in zip(model.parameters(), need[4:]):
            n = p.numel()
            out.append(grad_params[off:off + n].view(p.shape).to(device=p.device, dtype=p.dtype) if needs else None)
            off += n
        return tuple(out)

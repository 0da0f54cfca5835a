"""`DiffNet` -- drop-in for network/diff/net.py:86-135 backed by libdsvc (sm_100a kernels).

Same constructor, same `forward(spec [B,1,M,T], diffusion_step [B], cond [B,H,T]) -> [B,1,M,T]`, same
parameter names / shapes (so `utils.load_ckpt(..., strict=True)`, `.cuda()`, `state_dict()` round-trip).
The torch sub-modules below only *hold* the fp32 master parameters; no torch op runs in `forward`.
"""
import ctypes as C
import math

import torch
import torch.nn as nn

from . import _lib
from .hparams import hparams


class AttrDict(dict):
    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.__dict__ = self


class Mish(nn.Module):  # placeholder keeping `mlp.0` / `mlp.2` key numbering (net.py:99-103)
    def forward(self, x):
        return x * torch.tanh(torch.nn.functional.softplus(x))


class SinusoidalPosEmb(nn.Module):
    """net.py:32-44.  Evaluated on the HOST with the same float ops as the reference to tabulate the
    weight-free basis for every integer step (dsvc.h: dsvc_diffnet_weights.step_basis)."""

    def __init__(self, dim):
        super().__init__()
        self.dim = dim

    def forward(self, x):
        half_dim = self.dim // 2
        emb = math.log(10000) / (half_dim - 1)
        emb = torch.exp(torch.arange(half_dim, device=x.device) * -emb)
        emb = x[:, None] * emb[None, :]
        return torch.cat((emb.sin(), emb.cos()), dim=-1)


def Conv1d(*args, **kwargs):
    layer = nn.Conv1d(*args, **kwargs)
    nn.init.kaiming_normal_(layer.weight)
    return layer


class ResidualBlock(nn.Module):
    """Parameter container of net.py:58-64 (the math lives in the fused wavenet-layer kernels)."""

    def __init__(self, encoder_hidden, residual_channels, dilation):
        super().__init__()
        self.dilation = dilation
        self.dilated_conv = Conv1d(residual_channels, 2 * residual_channels, 3, padding=dilation, dilation=dilation)
        self.diffusion_projection = nn.Linear(residual_channels, residual_channels)
        self.conditioner_projection = Conv1d(encoder_hidden, 2 * residual_channels, 1)
        self.output_projection = Conv1d(residual_channels, 2 * residual_channels, 1)


class DiffNet(nn.Module):
    MATH = {"tc3f16": _lib.DSVC_MATH_TC3F16, "fp32": _lib.DSVC_MATH_FP32, "tc1f16": _lib.DSVC_MATH_TC1F16}

    def __init__(self, in_dims=80, math_mode=None, num_timesteps=None):
        super().__init__()
        self.params = params = AttrDict(
            encoder_hidden=hparams["hidden_size"], residual_layers=hparams["residual_layers"],
            residual_channels=hparams["residual_channels"], dilation_cycle_length=hparams["dilation_cycle_length"])
        self.in_dims = in_dims
        dim = params.residual_channels
        self.input_projection = Conv1d(in_dims, dim, 1)
        self.diffusion_embedding = SinusoidalPosEmb(dim)
        self.mlp = nn.Sequential(nn.Linear(dim, dim * 4), Mish(), nn.Linear(dim * 4, dim))
        self.residual_layers = nn.ModuleList([
            ResidualBlock(params.encoder_hidden, dim, 2 ** (i % params.dilation_cycle_length))
            for i in range(params.residual_layers)])
        self.skip_projection = Conv1d(dim, dim, 1)
        self.output_projection = Conv1d(dim, in_dims, 1)
        nn.init.zeros_(self.output_projection.weight)
        # --- native state (not part of state_dict) ---
        self.num_timesteps = int(num_timesteps or hparams.get("timesteps", 1000))
        if math_mode is None:
            tc_ok = in_dims % 4 == 0 and dim % 128 == 0     # the library pads the mel axis to whole tiles
            math_mode = hparams.get("dsvc_math", "tc3f16" if tc_ok else "fp32")
        self.math_mode = math_mode
        self._h = None
        self._h_key = None
        self._cond_key = None
        self._keep = None

    # ---- native handle management ----
    def _weights_key(self):
        return tuple((p.data_ptr(), p._version) for p in self.parameters()) + (self.math_mode, self.num_timesteps)

    def release(self):
        if self._h is not None:
            _lib.load().dsvc_diffnet_destroy(self._h)
        self._h = None
        self._h_key = None
        self._cond_key = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass

    def handle(self):
        """Build (or rebuild after a weight change) the libdsvc handle from the fp32 master parameters."""
        key = self._weights_key()
        if self._h is not None and key == self._h_key:
            return self._h
        self.release()
        lib = _lib.load()
        if not torch.cuda.is_available() or lib.dsvc_device_count() == 0:
            raise _lib.DsvcError("diffsvc_b200.DiffNet needs an sm_100 (B200) device: there is no CPU fallback")
        p = self.params
        cpu = lambda t: t.detach().to("cpu", torch.float32).contiguous()
        keep = []

        def f(t):
            t = cpu(t)
            keep.append(t)
            return _lib.fptr(t)

        def fa(ts):
            ts = [cpu(t) for t in ts]
            keep.extend(ts)
            arr = _lib.fptr_array(ts)
            keep.append(arr)
            return arr

        L = self.residual_layers
        w = _lib.DiffnetWeights()
        w.input_projection_w, w.input_projection_b = f(self.input_projection.weight), f(self.input_projection.bias)
        w.mlp0_w, w.mlp0_b = f(self.mlp[0].weight), f(self.mlp[0].bias)
        w.mlp2_w, w.mlp2_b = f(self.mlp[2].weight), f(self.mlp[2].bias)
        w.dilated_conv_w, w.dilated_conv_b = fa([l.dilated_conv.weight for l in L]), fa([l.dilated_conv.bias for l in L])
        w.diffusion_proj_w = fa([l.diffusion_projection.weight for l in L])
        w.diffusion_proj_b = fa([l.diffusion_projection.bias for l in L])
        w.conditioner_proj_w = fa([l.conditioner_projection.weight for l in L])
        w.conditioner_proj_b = fa([l.conditioner_projection.bias for l in L])
        w.output_proj_w, w.output_proj_b = fa([l.output_projection.weight for l in L]), fa([l.output_projection.bias for l in L])
        w.skip_projection_w, w.skip_projection_b = f(self.skip_projection.weight), f(self.skip_projection.bias)
        w.output_projection_w, w.output_projection_b = f(self.output_projection.weight), f(self.output_projection.bias)
        # weight-free sinusoid basis for t = 0..Tn-1, with the reference's own float ops (net.py:37-44)
        w.step_basis = f(self.diffusion_embedding(torch.arange(self.num_timesteps, dtype=torch.long)).to(torch.float32))
        cfg = _lib.DiffnetConfig(self.in_dims, p.residual_channels, p.encoder_hidden, p.residual_layers,
                                 p.dilation_cycle_length, self.num_timesteps, self.MATH[self.math_mode])
        h = C.c_void_p()
        with torch.cuda.device(self.input_projection.weight.device if self.input_projection.weight.is_cuda else torch.cuda.current_device()):
            _lib.check(lib.dsvc_diffnet_create(C.byref(h), C.byref(cfg), C.byref(w), _lib.current_stream()))
        self._h, self._h_key, self._cond_key = h, key, None
        self._sched_key = None
        return h

    def prepare(self, cond, lengths=None):
        """Hoisted per-utterance work: conditioner projections of all layers (net.py:68)."""
        h = self.handle()
        cond = cond.detach().to(torch.float32).contiguous()
        assert cond.is_cuda and cond.dim() == 3 and cond.shape[1] == self.params.encoder_hidden, cond.shape
        B, _, T = cond.shape
        lens = None
        if lengths is not None:
            lens = (C.c_int32 * B)(*[int(v) for v in lengths])
        key = (cond.data_ptr(), cond._version, tuple(cond.shape), None if lengths is None else tuple(int(v) for v in lengths))
        if key != self._cond_key:
            with torch.cuda.device(cond.device):     # the handle's kernels launch on the current device: the tensors' own
                _lib.check(_lib.load().dsvc_diffnet_prepare(h, B, T, lens, _lib.dptr(cond), _lib.current_stream()))
            self._cond_key = key
            self._keep = cond
        return h

    def forward(self, spec, diffusion_step, cond):
        """:param spec: [B, 1, M, T]  :param diffusion_step: [B] (all equal)  :param cond: [B, H, T]"""
        h = self.prepare(cond)
        ts = diffusion_step.reshape(-1)
        t = int(ts[0])
        if ts.numel() > 1 and not bool((ts == ts[0]).all()):
            raise ValueError("all batch items must share the diffusion step (the reference's sampler does)")
        spec = spec.detach().to(torch.float32).contiguous()
        out = torch.empty_like(spec)
        with torch.cuda.device(spec.device):
            _lib.check(_lib.load().dsvc_diffnet_eval(h, _lib.dptr(spec), t, _lib.dptr(out), _lib.current_stream()))
        return out

"""`Generator` / `load_model` -- drop-in for modules/nsf_hifigan/models.py:14-30, :325-396 backed by
libdsvc.  Holds the weight-norm-folded fp32 weights and a native handle; `__call__(c, f0)` has the
reference's signature: c [B, num_mels, T] natural-log mel, f0 [B, T] Hz -> [B, 1, T*hop]."""
import ctypes as C
import json
import os

import numpy as np
import torch

from .. import _lib


class AttrDict(dict):
    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.__dict__ = self


def fold_weight_norm(sd):
    """remove_weight_norm (models.py:389-396): w = g * v / ||v|| over all dims but 0."""
    out = {}
    for k, v in sd.items():
        if k.endswith(".weight_g"):
            base = k[:-len(".weight_g")]
            wv = sd[base + ".weight_v"]
            norm = wv.reshape(wv.shape[0], -1).norm(dim=1).reshape(-1, *([1] * (wv.dim() - 1)))
            out[base + ".weight"] = wv * (v / norm)
        elif not k.endswith(".weight_v"):
            out[k] = v
    return out


def resblock_type(h):
    """models.py:337 / modules/hifigan/hifigan.py:119: ResBlock1 for '1', ResBlock2 for anything else.  A missing
    key or an integer 1 also mean ResBlock1."""
    return 1 if str(h.get("resblock", "1")) == "1" else 2


def resblock_dilations(h):
    """Dilations per ResBlock: ResBlock2 (models.py:73-83) builds its two convs from dilation[0] and dilation[1] and
    ignores further entries."""
    rds = [list(d) for d in h["resblock_dilation_sizes"]]
    if resblock_type(h) == 1:
        return rds
    for d in rds:
        if len(d) < 2:
            raise ValueError("ResBlock2 needs two dilations per kernel, got %r" % (d,))
    return [d[:2] for d in rds]


def resblock_keys(h):
    """ResBlock conv names per module list, in the order the native generator takes them ([stage * num_kernels + j][m]):
    {"convs1": [...], "convs2": [...]} for ResBlock1, {"convs": [...]} for ResBlock2 (resblocks.{n}.convs.{m})."""
    nk, ns = len(h["resblock_kernel_sizes"]), len(h["upsample_rates"])
    nd = len(resblock_dilations(h)[0])
    idx = [(i * nk + j, m) for i in range(ns) for j in range(nk) for m in range(nd)]
    names = ("convs1", "convs2") if resblock_type(h) == 1 else ("convs",)
    return {c: ["resblocks.%d.%s.%d" % (n, c, m) for n, m in idx] for c in names}


def state_dict_keys(h, has_source=True):
    """Every weight-norm-folded key the native generator reads."""
    ns = len(h["upsample_rates"])
    keys = ["conv_pre.weight", "conv_pre.bias", "conv_post.weight", "conv_post.bias"]
    keys += ["ups.%d.%s" % (i, p) for i in range(ns) for p in ("weight", "bias")]
    if has_source:
        keys += ["m_source.l_linear.weight", "m_source.l_linear.bias"]
        keys += ["noise_convs.%d.%s" % (i, p) for i in range(ns) for p in ("weight", "bias")]
    for names in resblock_keys(h).values():
        keys += [n + p for n in names for p in (".weight", ".bias")]
    return keys


class Generator:
    def __init__(self, h, state_dict=None, device="cuda"):
        self.h = h if isinstance(h, AttrDict) else AttrDict(h)
        self.device = torch.device(device)
        self.num_kernels = len(self.h.resblock_kernel_sizes)
        self.num_upsamples = len(self.h.upsample_rates)
        self.hop = int(np.prod(self.h.upsample_rates))
        self._h = None
        self._sd = None
        if state_dict is not None:
            self.load_state_dict(state_dict)

    # nn.Module-ish surface the reference touches (models.py:23-28)
    def to(self, device):
        self.device = torch.device(device)
        return self

    def eval(self):
        return self

    def remove_weight_norm(self):
        print("Removing weight norm...")
        if self._sd is not None and any(k.endswith("weight_g") for k in self._sd):
            self.load_state_dict(self._sd)
        return self

    def state_dict(self):
        return dict(self._sd)

    def load_state_dict(self, sd, strict=True):
        sd = {k: v.detach().to("cpu", torch.float32) for k, v in sd.items()}
        self._sd = fold_weight_norm(sd)
        self._build()

    def release(self):
        if self._h is not None:
            _lib.load().dsvc_nsf_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass

    def _build(self):
        self.release()
        h, sd = self.h, self._sd
        rb = resblock_type(h)
        if rb == 2:      # name what is missing, as the reference's load_state_dict(strict=True) would
            missing = [k for k in state_dict_keys(h, "m_source.l_linear.weight" in sd) if k not in sd]
            if missing:
                raise KeyError("Missing key(s) in state_dict: %s" % ", ".join('"%s"' % k for k in missing))
        lib = _lib.load()
        if not torch.cuda.is_available() or lib.dsvc_device_count() == 0:
            raise _lib.DsvcError("diffsvc_b200 NSF-HiFiGAN needs an sm_100 (B200) device: there is no CPU fallback")
        nk, ns = self.num_kernels, self.num_upsamples
        dil = resblock_dilations(h)
        nd = len(dil[0])
        cfg = _lib.NsfConfig()
        cfg.num_mels, cfg.sampling_rate = int(h.num_mels), int(h.sampling_rate)
        cfg.upsample_initial_channel, cfg.num_upsamples = int(h.upsample_initial_channel), ns
        for i in range(ns):
            cfg.upsample_rates[i] = int(h.upsample_rates[i])
            cfg.upsample_kernel_sizes[i] = int(h.upsample_kernel_sizes[i])
        cfg.num_kernels, cfg.num_dilations, cfg.harmonic_num = nk, nd, 8
        self.has_source = "m_source.l_linear.weight" in sd
        cfg.has_source = 1 if self.has_source else 0
        for j in range(nk):
            cfg.resblock_kernel_sizes[j] = int(h.resblock_kernel_sizes[j])
            assert len(dil[j]) == nd
            for m in range(nd):
                cfg.resblock_dilation_sizes[j][m] = int(dil[j][m])
        keep = []

        def f(k):
            t = sd[k].contiguous()
            keep.append(t)
            return _lib.fptr(t)

        def fa(keys):
            ts = [sd[k].contiguous() for k in keys]
            keep.extend(ts)
            arr = _lib.fptr_array(ts)
            keep.append(arr)
            return arr

        w = _lib.NsfWeights()
        if self.has_source:
            w.source_linear_w, w.source_linear_b = f("m_source.l_linear.weight"), f("m_source.l_linear.bias")
            w.noise_convs_w = fa(["noise_convs.%d.weight" % i for i in range(ns)])
            w.noise_convs_b = fa(["noise_convs.%d.bias" % i for i in range(ns)])
        w.conv_pre_w, w.conv_pre_b = f("conv_pre.weight"), f("conv_pre.bias")
        w.ups_w, w.ups_b = fa(["ups.%d.weight" % i for i in range(ns)]), fa(["ups.%d.bias" % i for i in range(ns)])
        # ResBlock1: convs1 / convs2; ResBlock2: resblocks.{n}.convs.{m} in the convs1 slots, convs2 stays NULL
        first, *second = resblock_keys(h).values()
        w.convs1_w, w.convs1_b = fa([n + ".weight" for n in first]), fa([n + ".bias" for n in first])
        if second:
            w.convs2_w, w.convs2_b = fa([n + ".weight" for n in second[0]]), fa([n + ".bias" for n in second[0]])
        w.conv_post_w, w.conv_post_b = f("conv_post.weight"), f("conv_post.bias")
        hd = C.c_void_p()
        dev = self.device if self.device.type == "cuda" else torch.device("cuda")
        with torch.cuda.device(dev):
            _lib.check(lib.dsvc_nsf_create_ex(C.byref(hd), C.byref(cfg), rb, C.byref(w), _lib.current_stream()))
        self._h = hd

    def forward_mel(self, mel, f0, mel_scale=1.0, rand_ini=None, sine_noise=None, seed=None):
        """mel [B, T, num_mels] channels-last (scaled by mel_scale on load), f0 [B, T] -> wav [B, T*hop]."""
        assert self._h is not None, "Generator has no weights loaded"
        mel = mel.detach().to(torch.float32).contiguous()
        B, T, M = mel.shape
        assert M == self.h.num_mels, (mel.shape, self.h.num_mels)
        if f0 is not None:
            f0 = f0.detach().to(mel.device, torch.float32).contiguous()
            assert tuple(f0.shape) == (B, T), (mel.shape, f0.shape)
        wav = torch.empty(B, T * self.hop, device=mel.device, dtype=torch.float32)
        ri = sn = None
        if rand_ini is not None:
            rand_ini = rand_ini.detach().to(mel.device, torch.float32).contiguous()
            ri = _lib.dptr(rand_ini)
        if sine_noise is not None:
            sine_noise = sine_noise.detach().to(mel.device, torch.float32).contiguous()
            assert tuple(sine_noise.shape) == (B, T * self.hop, 9), sine_noise.shape
            sn = _lib.dptr(sine_noise)
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        with torch.cuda.device(mel.device):      # the handle's kernels launch on the current device: the tensors' own
            _lib.check(_lib.load().dsvc_nsf_forward(self._h, _lib.dptr(mel), None if f0 is None else _lib.dptr(f0), ri, sn, C.c_uint64(seed),
                                                    C.c_float(mel_scale), _lib.dptr(wav), B, T, _lib.current_stream()))
        return wav

    def __call__(self, x, f0=None, **kw):
        """Generator.forward(x [B,num_mels,T], f0 [B,T]) -> [B,1,T*hop]  (models.py:361-387)."""
        return self.forward_mel(x.transpose(1, 2), f0, 1.0, **kw)[:, None, :]


def load_model(model_path, device="cuda"):
    """models.py:14-30: sibling config.json + ckpt['generator'] (weight_g / weight_v form)."""
    config_file = os.path.join(os.path.split(model_path)[0], "config.json")
    with open(config_file) as f:
        h = AttrDict(json.loads(f.read()))
    cp_dict = torch.load(model_path, map_location="cpu")
    generator = Generator(h, cp_dict["generator"], device=device)
    generator.eval()
    generator.remove_weight_norm()
    del cp_dict
    return generator, h

"""Golden vectors of ResBlock2 ("resblock": "2") vocoder generators from the UNMODIFIED reference (CPU, fp32).

Run once, with DIFFSVC_REFERENCE_ROOT pointing at a checkout of the reference:

    python tests/golden/make_golden_resblock2.py    # nsf_resblock2_small.npz, hifigan24k_resblock2_small.npz

It builds the reference's own NSF-HiFiGAN `Generator` and 24 kHz `HifiGanGenerator` with resblock "2", perturbs
their weights as make_golden.py does for the ResBlock1 fixtures, records the random draws, and writes the
weight-norm checkpoint, the folded weights, the inputs, the draws and the waveforms (tests/test_resblock2.py).
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from make_golden import HERE, DrawRecorder, _np, rh  # noqa: E402


def _perturb_generator(gen):
    """The perturbation of gen_nsf / gen_hifigan24k: the reference's init (std 0.01) gives a ~0 waveform."""
    with torch.no_grad():
        for n, p in gen.named_parameters():
            if n.endswith("weight_v") or (n.endswith(".weight") and "noise_convs" in n):
                p.mul_(1.0 / (p.std() + 1e-8)).mul_(0.35 / np.sqrt(np.prod(p.shape[1:]) / (4 if n.startswith("ups") else 1)))
            if n.endswith("weight_g"):
                p.copy_(p * (1.0 + 0.3 * torch.randn_like(p)))


def gen_nsf_resblock2():
    """The NSF Generator with resblock "2" (ResBlock2, modules/nsf_hifigan/models.py:73-94, chosen at :337).  The
    second dilation list has three entries: ResBlock2 reads only the first two.  Dilation 12 at kernel 7 reaches 36
    rows, past the narrow kernel's 192-row window, so the 32- and 16-channel stages take the 256-row one; the 8-channel
    stage stays on the FFMA GEMM."""
    models = rh.import_nsf_models()
    from modules.nsf_hifigan.env import AttrDict
    h = AttrDict(resblock="2", upsample_rates=[4, 2, 2], upsample_kernel_sizes=[8, 4, 4],
                 upsample_initial_channel=64, resblock_kernel_sizes=[3, 7],
                 resblock_dilation_sizes=[[1, 2], [3, 12, 5]], num_mels=8, sampling_rate=16000)
    torch.manual_seed(56)
    gen = models.Generator(h).eval()
    _perturb_generator(gen)
    ckpt_sd = {k: v.clone() for k, v in gen.state_dict().items()}
    g = torch.Generator().manual_seed(10)
    B, T = 2, 12
    mel = torch.randn(B, 8, T, generator=g)
    f0 = torch.rand(B, T, generator=g) * 300 + 100
    f0[0, 3:6] = 0
    f0[1, 9:] = 0
    gen.remove_weight_norm()
    with DrawRecorder() as rec, torch.no_grad():
        wav = gen(mel, f0)
    kinds = [k for k, _ in rec.log]
    assert kinds == ["rand", "randn_like", "randn_like"], kinds       # models.py:192, :271, :322
    d = _np(ckpt_sd, "ckpt/")
    d.update(_np(gen.state_dict(), "sd/"))
    d.update(mel=mel.numpy(), f0=f0.numpy(), rand_ini=rec.log[0][1].numpy(), sine_noise=rec.log[1][1].numpy(),
             wav=wav.numpy())
    for k in ("upsample_rates", "upsample_kernel_sizes", "resblock_kernel_sizes"):
        d["h/" + k] = np.asarray(h[k], dtype=np.int64)
    for j, ds in enumerate(h.resblock_dilation_sizes):              # ragged: one array per kernel
        d["dil/%d" % j] = np.asarray(ds, dtype=np.int64)
    d["h/upsample_initial_channel"] = np.int64(h.upsample_initial_channel)
    d["h/num_mels"] = np.int64(8)
    d["h/sampling_rate"] = np.int64(16000)
    np.savez_compressed(os.path.join(HERE, "nsf_resblock2_small.npz"), **d)
    print("nsf_resblock2_small: wav", tuple(wav.shape), float(wav.abs().max()), float(wav.std()))


def gen_hifigan24k_resblock2():
    """The 24 kHz generator (modules/hifigan/hifigan.py:104-169) with resblock "2" (ResBlock2 :70-91, chosen at
    :119): with the pitch source (f0 given and f0=None) and a second model built without it."""
    import modules.hifigan.hifigan as hg
    h = dict(resblock="2", upsample_rates=[4, 2], upsample_kernel_sizes=[8, 4], upsample_initial_channel=64,
             resblock_kernel_sizes=[3, 5], resblock_dilation_sizes=[[1, 3], [2, 8]], use_pitch_embed=True,
             audio_sample_rate=24000)
    torch.manual_seed(78)
    gen = hg.HifiGanGenerator(h).eval()
    _perturb_generator(gen)
    ckpt_sd = {k: v.clone() for k, v in gen.state_dict().items()}
    g = torch.Generator().manual_seed(20)
    B, T = 2, 10
    mel = torch.randn(B, 80, T, generator=g)
    f0 = torch.rand(B, T, generator=g) * 300 + 100
    f0[1, 2:5] = 0
    gen.remove_weight_norm()
    with DrawRecorder() as rec, torch.no_grad():
        wav_f0 = gen(mel, f0)
    assert [k for k, _ in rec.log] == ["rand", "randn_like", "randn_like"]
    with torch.no_grad():
        wav_plain = gen(mel)
    gen2 = hg.HifiGanGenerator(dict(h, use_pitch_embed=False)).eval()
    _perturb_generator(gen2)
    ckpt2 = {k: v.clone() for k, v in gen2.state_dict().items()}
    gen2.remove_weight_norm()
    with torch.no_grad():
        wav_nosrc = gen2(mel)
    d = _np(ckpt_sd, "ckpt/")
    d.update(_np(ckpt2, "nosrc_ckpt/"))
    d.update(mel=mel.numpy(), f0=f0.numpy(), rand_ini=rec.log[0][1].numpy(), sine_noise=rec.log[1][1].numpy(),
             wav_f0=wav_f0.numpy(), wav_plain=wav_plain.numpy(), wav_nosrc=wav_nosrc.numpy())
    for k in ("upsample_rates", "upsample_kernel_sizes", "resblock_kernel_sizes", "resblock_dilation_sizes"):
        d["h/" + k] = np.asarray(h[k], dtype=np.int64)
    d["h/upsample_initial_channel"] = np.int64(h["upsample_initial_channel"])
    d["h/audio_sample_rate"] = np.int64(24000)
    np.savez_compressed(os.path.join(HERE, "hifigan24k_resblock2_small.npz"), **d)
    print("hifigan24k_resblock2_small: wav", tuple(wav_f0.shape), float(wav_f0.std()), float(wav_plain.std()),
          float(wav_nosrc.std()))


def main():
    rh.install()
    gen_nsf_resblock2()
    gen_hifigan24k_resblock2()


if __name__ == "__main__":
    main()

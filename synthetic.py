"""Seeded synthetic checkpoints and inputs.

The reference repository ships no weights, no vocoder `config.json` and no audio fixtures for this path
(SURVEY.md section 8c: `checkpoints/` is git-ignored), so the bench, the smoke test and the parity tests all draw
their model weights and utterances from the generators below.  NEUTRAL module: it is neither the product
(`diffsvc_b200/`) nor the checker (`oracle/`), and both sides of a parity test must be fed from the same call so
that they evaluate the same function.  Pure torch-CPU tensor construction; no model arithmetic lives here.
"""
import math

import numpy as np
import torch

NSF_H_44K = dict(  # assumed openvpi 44.1 kHz topology (SURVEY.md section 8c): not in the reference repo
    resblock="1", upsample_rates=[8, 8, 2, 2, 2], upsample_kernel_sizes=[16, 16, 4, 4, 4],
    upsample_initial_channel=512, resblock_kernel_sizes=[3, 7, 11],
    resblock_dilation_sizes=[[1, 3, 5], [1, 3, 5], [1, 3, 5]], num_mels=128, sampling_rate=44100,
    n_fft=2048, win_size=2048, hop_size=512, fmin=40, fmax=16000)


NSF_H_44K_V3 = dict(  # a HiFi-GAN "V3"-style 44.1 kHz NSF generator: ResBlock2 blocks, dilations up to 12
    NSF_H_44K, resblock="2", resblock_kernel_sizes=[3, 5, 7], resblock_dilation_sizes=[[1, 2], [2, 6], [3, 12]])


HIFIGAN_H_24K = dict(  # assumed 24 kHz HiFi-GAN topology (SURVEY.md section 8c): its config.yaml is not in the reference repo
    resblock="1", upsample_rates=[8, 4, 2, 2], upsample_kernel_sizes=[16, 8, 4, 4],
    upsample_initial_channel=512, resblock_kernel_sizes=[3, 7, 11],
    resblock_dilation_sizes=[[1, 3, 5], [1, 3, 5], [1, 3, 5]], num_mels=80, sampling_rate=24000,
    audio_sample_rate=24000, hop_size=128, use_pitch_embed=True)


# The 24 kHz model of training/config.yaml (the reference's default config), as overrides of the 44.1 kHz defaults
# (diffsvc_b200.hparams.DEFAULTS_44K).  spec_min / spec_max stay scalar: the config's per-bin lists are trained statistics.
HPARAMS_24K = dict(
    audio_num_mel_bins=80, audio_sample_rate=24000, hop_size=128, fft_size=512, win_size=512, fmin=30, fmax=12000,
    hidden_size=256, residual_layers=20, residual_channels=256, dilation_cycle_length=4, keep_bins=80,
    f0_min=50.0, f0_max=1100.0, pndm_speedup=10, use_nsf=True, use_pitch_embed=True,
    vocoder="diffsvc_b200.vocoders.hifigan.HifiGAN", vocoder_ckpt="checkpoints/0109_hifigan_bigpopcs_hop128",
)


def synth_diffnet_weights(M=128, C=384, H=256, L=20, seed=1234):
    """Seeded synthetic DiffNet state dict with the reference's key names and init statistics
    (kaiming-normal convs net.py:47-50, default Linear init), and a NON-zero output_projection
    (the reference zero-inits it, net.py:110, which would make every parity test vacuous)."""
    g = torch.Generator().manual_seed(seed)

    def kaiming(co, ci, k):
        return torch.randn(co, ci, k, generator=g) * math.sqrt(2.0 / (ci * k))

    def unif(shape, fan_in):
        b = 1.0 / math.sqrt(fan_in)
        return (torch.rand(*shape, generator=g) * 2 - 1) * b

    sd = {
        "input_projection.weight": kaiming(C, M, 1), "input_projection.bias": unif((C,), M),
        "mlp.0.weight": unif((4 * C, C), C), "mlp.0.bias": unif((4 * C,), C),
        "mlp.2.weight": unif((C, 4 * C), 4 * C), "mlp.2.bias": unif((C,), 4 * C),
        "skip_projection.weight": kaiming(C, C, 1), "skip_projection.bias": unif((C,), C),
        "output_projection.weight": torch.randn(M, C, 1, generator=g) * 0.05, "output_projection.bias": unif((M,), C),
    }
    for l in range(L):
        p = "residual_layers.%d." % l
        sd[p + "dilated_conv.weight"] = kaiming(2 * C, C, 3)
        sd[p + "dilated_conv.bias"] = unif((2 * C,), 3 * C)
        sd[p + "diffusion_projection.weight"] = unif((C, C), C)
        sd[p + "diffusion_projection.bias"] = unif((C,), C)
        sd[p + "conditioner_projection.weight"] = kaiming(2 * C, H, 1)
        sd[p + "conditioner_projection.bias"] = unif((2 * C,), H)
        sd[p + "output_projection.weight"] = kaiming(2 * C, C, 1)
        sd[p + "output_projection.bias"] = unif((2 * C,), C)
    return sd


def synth_nsf_weights(h, seed=4321, std=None):
    """Seeded synthetic, weight-norm-folded NSF-HiFiGAN generator weights with the reference's key
    names.  Scaled (fan-in) so activations stay O(1) through the stack -- the reference's own init
    (std 0.01, utils.py:22-25) would give a numerically vacuous ~0 waveform."""
    g = torch.Generator().manual_seed(seed)
    rates, ks = h["upsample_rates"], h["upsample_kernel_sizes"]
    c0 = h["upsample_initial_channel"]
    sd = {}

    def w(shape, fan_in, gain=1.0):
        return torch.randn(*shape, generator=g) * (gain / math.sqrt(fan_in))

    def b(n):
        return (torch.rand(n, generator=g) * 2 - 1) * 0.05

    sd["m_source.l_linear.weight"] = w((1, 9), 9, 2.0)
    sd["m_source.l_linear.bias"] = b(1)
    sd["conv_pre.weight"] = w((c0, h["num_mels"], 7), h["num_mels"] * 7)
    sd["conv_pre.bias"] = b(c0)
    ch = c0
    for i, (u, k) in enumerate(zip(rates, ks)):
        cin, ch = c0 // (2 ** i), c0 // (2 ** (i + 1))
        sd["ups.%d.weight" % i] = w((cin, ch, k), cin * k / u, 1.4)
        sd["ups.%d.bias" % i] = b(ch)
        if i + 1 < len(rates):
            s = int(np.prod(rates[i + 1:]))
            sd["noise_convs.%d.weight" % i] = w((ch, 1, 2 * s), 2 * s, 1.0)
        else:
            sd["noise_convs.%d.weight" % i] = w((ch, 1, 1), 1, 0.5)
        sd["noise_convs.%d.bias" % i] = b(ch)
        for j, kk in enumerate(h["resblock_kernel_sizes"]):
            p = "resblocks.%d." % (i * len(h["resblock_kernel_sizes"]) + j)
            for m in range(len(h["resblock_dilation_sizes"][j])):
                sd[p + "convs1.%d.weight" % m] = w((ch, ch, kk), ch * kk, 1.0)
                sd[p + "convs1.%d.bias" % m] = b(ch)
                sd[p + "convs2.%d.weight" % m] = w((ch, ch, kk), ch * kk, 0.5)
                sd[p + "convs2.%d.bias" % m] = b(ch)
    sd["conv_post.weight"] = w((1, ch, 7), ch * 7, 1.0)
    sd["conv_post.bias"] = b(1)
    return sd


def synth_f0(B, T, seed=11):
    """Smooth f0 contour in [80, 800] Hz with ~20 % unvoiced (0) runs (SURVEY.md section 8d)."""
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(T, dtype=torch.float32)[None, :]
    ph = torch.rand(B, 1, generator=g) * 6.28
    f0 = 220.0 * 2 ** (0.9 * torch.sin(t * 0.013 + ph) + 0.3 * torch.sin(t * 0.071 + 2 * ph))
    f0 = f0.clamp(80.0, 800.0)
    run = (torch.sin(t * 0.05 + 3 * ph) > 0.6)      # unvoiced runs, ~20 % of frames
    return torch.where(run, torch.zeros_like(f0), f0)


def synth_nsf_resblock2_weights(h, seed=4321):
    """ResBlock2 ("resblock": "2") generator weights: synth_nsf_weights of the same topology with the first two
    dilations of every list, each block's convs1.{m} renamed to convs.{m} (ResBlock2's key names, models.py:76-81)
    and convs2 dropped."""
    h1 = dict(h, resblock="1", resblock_dilation_sizes=[list(d)[:2] for d in h["resblock_dilation_sizes"]])
    return {k.replace(".convs1.", ".convs."): v for k, v in synth_nsf_weights(h1, seed).items() if ".convs2." not in k}

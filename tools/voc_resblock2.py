"""Vocoder timing of a ResBlock2 ("resblock": "2", HiFi-GAN V3-style) 44.1 kHz NSF generator, one pass, CUDA events,
best of N after warm-up, in three modes:
  default  -- every ResBlock stage on tcgen05; the 32- / 16-channel stages on the narrow kernel, here its 256-row
              window (the dilation-12 kernel-7 convs reach 36 rows)
  narrow0  -- DSVC_NSF_NARROW=0: the 32- / 16-channel stages on the FFMA GEMM
  fp32     -- DSVC_NSF_MATH=fp32: the whole generator on the FFMA GEMM
and the ResBlock1 NSF_H_44K generator (default mode) for context.  FLOPs are algorithmic, computed from the shapes.

    python tools/voc_resblock2.py [--iters N] [--out FILE]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import synthetic as S  # noqa: E402

MODES = (("default", {}), ("narrow0", {"DSVC_NSF_NARROW": "0"}), ("fp32", {"DSVC_NSF_MATH": "fp32"}))
SIZES = ((1, 862), (1, 43), (8, 689))        # a 10 s clip, a 0.5 s clip, a batch of eight 8 s clips


def generator_flops(h, T, has_source=True):
    """Multiply-adds x 2 of one item of T frames: conv_pre, the transposed convs, noise_convs, every ResBlock conv
    and conv_post."""
    rates, ks = h["upsample_rates"], h["upsample_kernel_sizes"]
    c0 = h["upsample_initial_channel"]
    rb2 = str(h.get("resblock", "1")) != "1"
    flops = 2.0 * h["num_mels"] * c0 * 7 * T
    length, ch = T, c0
    for i, (u, k) in enumerate(zip(rates, ks)):
        cout = ch // 2
        flops += 2.0 * ch * cout * k * length             # each input sample feeds k outputs per (cin, cout)
        length *= u
        if has_source:
            kn = 2 * int(np.prod(rates[i + 1:])) if i + 1 < len(rates) else 1
            flops += 2.0 * cout * kn * length
        for kk, dil in zip(h["resblock_kernel_sizes"], h["resblock_dilation_sizes"]):
            convs = 2 if rb2 else 2 * len(dil)
            flops += convs * 2.0 * cout * cout * kk * length
        ch = cout
    return flops + 2.0 * ch * 7 * length


def time_pass(voc, mel, f0, iters, warmup=3):
    for _ in range(warmup):
        w = voc.spec2wav_torch(mel, f0=f0, seed=1)
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        w = voc.spec2wav_torch(mel, f0=f0, seed=1)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best, w


def set_mode(env):
    for k in ("DSVC_NSF_NARROW", "DSVC_NSF_MATH"):
        os.environ.pop(k, None)
    os.environ.update(env)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the report here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("voc_resblock2: needs a CUDA device (sm_100)")
    import diffsvc_b200 as D
    D.hparams.update(use_nsf=True)
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                 # the report still names the device
        q = "%s (nvidia-smi: %s)" % (torch.cuda.get_device_name(0), e)
    say("# device: %s" % q)
    say("# one vocoder pass (mel + f0 -> waveform), CUDA events, best of %d after 3 warm-up passes; synthetic weights" % args.iters)
    h2, h1 = S.NSF_H_44K_V3, S.NSF_H_44K
    say("# V3-style: resblock 2, kernels %s, dilations %s; ResBlock1 NSF_H_44K: kernels %s, dilations %s" % (
        h2["resblock_kernel_sizes"], h2["resblock_dilation_sizes"], h1["resblock_kernel_sizes"], h1["resblock_dilation_sizes"]))
    sd2 = S.synth_nsf_resblock2_weights(h2)
    sd1 = S.synth_nsf_weights(h1)
    for B, T in SIZES:
        g = torch.Generator().manual_seed(B * 1000 + T)
        mel = (torch.randn(B, T, 128, generator=g) * 0.8 - 2.0).cuda()
        f0 = S.synth_f0(B, T).cuda()
        audio_s = B * T * 512 / 44100
        out = {}
        for name, h, sd, modes in (("resblock2", h2, sd2, MODES), ("resblock1", h1, sd1, MODES[:1])):
            flops = generator_flops(h, T) * B
            for mode, env in modes:
                set_mode(env)
                voc = D.NsfHifiGAN.from_state_dict(dict(h), sd, device="cuda")
                ms, w = time_pass(voc, mel, f0, args.iters)
                voc.model.release()
                out[(name, mode)] = w
                say("[voc] %s %-8s B=%d T=%d: %8.3f ms  %6.2f GFLOP  %6.1f TFLOP/s algorithmic  %6.0fx real time" % (
                    name, mode, B, T, ms, flops / 1e9, flops / ms / 1e9, audio_s / (ms / 1e3)))
        set_mode({})
        ref = out[("resblock2", "fp32")]
        say("      resblock2 max |default - fp32| = %.2e   max |narrow0 - fp32| = %.2e" % (
            (out[("resblock2", "default")] - ref).abs().max().item(), (out[("resblock2", "narrow0")] - ref).abs().max().item()))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

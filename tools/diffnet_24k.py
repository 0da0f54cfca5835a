"""The 24 kHz model of training/config.yaml (80 mel bins, C = 256, 20 layers) on the FFMA path (fp32) and the 3-pass
tensor-core path (tc3f16, mel axis padded to 128 inside the library), in one process, on the same seeded weights and
inputs, the two modes alternating over ROUNDS rounds (one handle per (mode, shape)).

CUDA events around each call; the sampler's working set (fp16 hi/lo weights ~21 MB + activations) stays L2-resident from
call to call, as it does in a user's sampler loop, so no L2 flush is made.
  cfg1       BASELINE cfg1: one 5 s clip (938 frames), 100 DDPM steps  -> us per step and ms per call
  plms1256   the notebook's 1256-frame segment, PLMS at pndm_speedup=20 over 1000 steps (51 evaluations)  -> p50 ms per call
  plms94     a 0.5 s chunk (94 frames), the same sampler  -> p50 ms per call
  plms8x     8 slices of 938 frames +- 25 % in one packed batch, the same sampler  -> p50 ms per call
  vocoder    the 24 kHz HiFi-GAN (synthetic.HIFIGAN_H_24K) with its pitch source on cfg1's 938 frames  -> p50 ms per call
and the max-abs difference between the two modes' mels over the whole output tensor (same library noise seed for DDPM), and
end-to-end cfg1 audio-sec/s (diffusion call + vocoder; the conditioning encoder is excluded).  Two caveats on the
difference: PLMS has no clamp, and with random weights its solve is expansive (mels reach hundreds), so its absolute
difference is large next to the DDPM one -- tests/test_diffnet_24k.py bounds it relative to the range; and the 8-slice batch's
tensor includes frames past each slice's length, which are not part of the result (the packed tensor-core batch leaves them
as passed in, the FFMA path's dense grid updates them), so its difference there is meaningless.

    python tools/diffnet_24k.py [--rounds N] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import synthetic as S  # noqa: E402

SR, HOP, MEL, C, H = 24000, 128, 80, 256, 256
MODES = ("fp32", "tc3f16")


def set_hparams():
    from diffsvc_b200.hparams import hparams, DEFAULTS_44K
    hparams.clear(); hparams.update(DEFAULTS_44K); hparams.update(S.HPARAMS_24K); hparams["pndm_speedup"] = 1


def model(mode, K_step):
    import diffsvc_b200 as D
    set_hparams()
    torch.manual_seed(0)
    dn = D.DiffNet(MEL, math_mode=mode)
    dn.load_state_dict(S.synth_diffnet_weights(M=MEL, C=C, H=H, L=20), strict=True)
    return D.GaussianDiffusion(None, MEL, dn, timesteps=1000, K_step=K_step, loss_type="l2", spec_min=[-5.0],
                               spec_max=[0.0]).cuda().eval()


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); out = fn(); b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b), out


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                           capture_output=True, text=True, timeout=30)
        return " | ".join(r.stdout.strip().splitlines()[:2])
    except Exception as ex:
        return "nvidia-smi unavailable (%r)" % ex


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--calls", type=int, default=5, help="timed calls per leg, mode and round")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from diffsvc_b200.vocoders.hifigan import HifiGAN
    assert torch.cuda.is_available(), "tools/diffnet_24k.py measures on the GPU"
    g = torch.Generator().manual_seed(1)

    def clip(T, B=1):
        return (torch.randn(B, H, T, generator=g) * 0.5).cuda(), torch.randn(B, 1, MEL, T, generator=g).cuda()

    c938, x938 = clip(938)
    c1256, x1256 = clip(1256)
    c94, x94 = clip(94)
    lens = (938 * (0.75 + 0.5 * torch.rand(8, generator=g))).round().long().tolist()
    c8, x8 = clip(max(lens), 8)
    legs = {
        "cfg1": (100, c938, None, lambda gd: gd.sample(x938, c938, 100, None, None, seed=3)),
        "plms1256": (1000, c1256, None, lambda gd: gd.sample(x1256, c1256, 1000, 20)),
        "plms94": (1000, c94, None, lambda gd: gd.sample(x94, c94, 1000, 20)),
        "plms8x": (1000, c8, lens, lambda gd: gd.sample(x8, c8, 1000, 20, lengths=lens)),
    }
    gds = {}
    for m in MODES:
        for k, (K, cond, ln, _) in legs.items():
            gds[(m, k)] = model(m, K)
            gds[(m, k)].denoise_fn.prepare(cond, ln)
    set_hparams()
    h = dict(S.HIFIGAN_H_24K)
    voc = HifiGAN.from_state_dict(h, S.synth_nsf_weights(h), device="cuda")
    f0 = S.synth_f0(1, 938, seed=2).cuda()
    mel938 = (torch.randn(1, 938, MEL, generator=g) * 0.8 - 2.0).cuda()

    res = {m: {k: [] for k in legs} for m in MODES}
    res_voc = []
    outs = {}
    with torch.no_grad():
        for r in range(args.rounds + 1):                       # round 0: warm-up (graph capture, module load)
            for m in MODES:
                for k, (_, _, _, fn) in legs.items():
                    for _ in range(args.calls if r > 0 else 1):
                        ms, out = event_ms(lambda: fn(gds[(m, k)]))
                        if r > 0:
                            res[m][k].append(ms)
                    outs[(m, k)] = gds[(m, k)].denorm_spec(out[:, 0].transpose(1, 2)).cpu()
            for _ in range(args.calls if r > 0 else 1):
                ms, _ = event_ms(lambda: voc.model.forward_mel(mel938, f0, 1.0, seed=5))
                if r > 0:
                    res_voc.append(ms)
    lines = ["card: %s" % card(),
             "24 kHz DiffNet (M=80, C=256, L=20, H=256), fp32 (FFMA) vs tc3f16 (3-pass tcgen05), %d rounds x %d calls per "
             "leg and mode, modes alternating; median (min .. max)" % (args.rounds, args.calls),
             "8-slice lengths: %s" % lens, ""]
    summary = {"card": card(), "lens8": lens}
    for k in legs:
        row = {}
        for m in MODES:
            v = res[m][k]
            row[m] = [x * 1000.0 / 100 for x in v] if k == "cfg1" else v
        unit = "us/step" if k == "cfg1" else "ms/call"
        mf, mt = statistics.median(row["fp32"]), statistics.median(row["tc3f16"])
        diff = (outs[("fp32", k)] - outs[("tc3f16", k)]).abs().max().item()
        summary[k] = {"unit": unit, "fp32": row["fp32"], "tc3f16": row["tc3f16"], "fp32_median": mf, "tc3f16_median": mt,
                      "speedup": mf / mt, "mel_maxabs_fp32_vs_tc3f16": diff}
        lines.append("%-9s %-8s fp32 %9.2f (%9.2f .. %9.2f)   tc3f16 %9.2f (%9.2f .. %9.2f)   x%5.2f   mel max-abs diff %.2e" % (
            k, unit, mf, min(row["fp32"]), max(row["fp32"]), mt, min(row["tc3f16"]), max(row["tc3f16"]), mf / mt, diff))
        if k == "cfg1":
            lines.append("%-9s %-8s fp32 %9.2f   tc3f16 %9.2f" % ("cfg1", "ms/call", mf * 100 / 1000.0, mt * 100 / 1000.0))
    vm = statistics.median(res_voc)
    audio = 938 * HOP / SR
    lines.append("%-9s %-8s %9.2f (%9.2f .. %9.2f)" % ("vocoder", "ms/call", vm, min(res_voc), max(res_voc)))
    e2e = {m: audio / ((summary["cfg1"][m + "_median"] * 100 / 1000.0 + vm) / 1000.0) for m in MODES}
    lines.append("cfg1 end to end (100 DDPM steps + vocoder, %.3f s of audio): fp32 %.1f audio-sec/s, tc3f16 %.1f audio-sec/s"
                 % (audio, e2e["fp32"], e2e["tc3f16"]))
    summary["vocoder_ms"] = res_voc
    summary["cfg1_audio_sec_per_s"] = e2e
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n\n" + json.dumps(summary, indent=1) + "\n")


if __name__ == "__main__":
    main()

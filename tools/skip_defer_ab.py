"""A/B of the deferred-skip layer schedule (DESIGN.md 3.1d) against the layer-by-layer one (DSVC_SKIP_DEFER=0), both
in one process, the two alternating over ROUNDS rounds (each on its own handle: the switch is read at prepare).

Per round and schedule, CUDA events:
  ddpm862  sampler alone, 1000 DDPM steps of one 862-frame clip -> us per step
  ddpm43   sampler alone, 1000 DDPM steps of one 43-frame clip  -> us per step
  plms43   the flask chunk's sampler (43 frames, PNDM interval 20: 51 evaluations)  -> ms per call
  b8x689   8 clips of 689 frames +- 25 % (packed batch, 128- / 256-wide tiles: not deferred), 200 DDPM steps -> us per step
  bench    bench.py's timed step: 1000-step DDPM of the 862-frame clip + NSF-HiFiGAN, 256 MiB L2 flush before -> audio-sec/s
and whether the two schedules' outputs are bit-identical.

    python tools/skip_defer_ab.py [--rounds N] [--out FILE]
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

SR, HOP, MEL = 44100, 512, 128


def model(defer):
    import diffsvc_b200 as D
    from diffsvc_b200.hparams import hparams, DEFAULTS_44K
    hparams.clear(); hparams.update(DEFAULTS_44K); hparams["pndm_speedup"] = 1
    torch.manual_seed(0)
    dn = D.DiffNet(MEL, math_mode="tc3f16")
    dn.load_state_dict(S.synth_diffnet_weights(), strict=True)
    return D.GaussianDiffusion(None, MEL, dn, timesteps=1000, K_step=1000, loss_type="l2", spec_min=[-5.0], spec_max=[0.0]).cuda().eval()


def prepare(gd, defer, cond, lengths=None):
    """Prepare gd's handle for `cond` with the schedule switch set accordingly."""
    if defer:
        os.environ.pop("DSVC_SKIP_DEFER", None)
    else:
        os.environ["DSVC_SKIP_DEFER"] = "0"
    gd.denoise_fn.prepare(cond, lengths)


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); out = fn(); b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b), out


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as ex:
        return "nvidia-smi unavailable (%r)" % ex


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import diffsvc_b200 as D
    g = torch.Generator().manual_seed(1)
    c862 = (torch.randn(1, 256, 862, generator=g) * 0.5).cuda(); x862 = torch.randn(1, 1, MEL, 862, generator=g).cuda()
    c43 = (torch.randn(1, 256, 43, generator=g) * 0.5).cuda(); x43 = torch.randn(1, 1, MEL, 43, generator=g).cuda()
    lens = (689 * (0.75 + 0.5 * torch.rand(8, generator=g))).round().long().tolist()
    c8 = (torch.randn(8, 256, max(lens), generator=g) * 0.5).cuda(); x8 = torch.randn(8, 1, MEL, max(lens), generator=g).cuda()
    f0 = S.synth_f0(1, 862, seed=2).cuda()
    voc = D.NsfHifiGAN.from_state_dict(dict(S.NSF_H_44K), S.synth_nsf_weights(S.NSF_H_44K), device="cuda")
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")
    # one model per (schedule, shape): each handle keeps the workspace and captured graphs of its shape
    shapes = {"ddpm862": (c862, None), "ddpm43": (c43, None), "plms43": (c43, None), "b8x689": (c8, lens)}
    gds = {(d, k): model(d) for d in (False, True) for k in shapes}
    for (d, k), gd in gds.items():
        prepare(gd, d, *shapes[k])

    def bench_step(gd, i):
        x = gd.sample(x862, c862, 1000, None, None, seed=17 + i)
        mel = gd.denorm_spec(x[:, 0].transpose(1, 2)).clamp(-6.0, 1.5)
        return voc.spec2wav_torch(mel, f0=f0, seed=i)

    legs = {
        "ddpm862": lambda gd: gd.sample(x862, c862, 1000, None, None, seed=3),
        "ddpm43": lambda gd: gd.sample(x43, c43, 1000, None, None, seed=3),
        "plms43": lambda gd: gd.sample(x43, c43, 1000, 20),
        "b8x689": lambda gd: gd.sample(x8, c8, 200, None, None, lengths=lens, seed=3),
    }
    res = {d: {k: [] for k in list(legs) + ["bench"]} for d in ("old", "new")}
    outs = {}
    with torch.no_grad():
        for r in range(args.rounds + 1):                       # round 0: warm-up (graph capture, module load)
            for d in (False, True):
                name = "new" if d else "old"
                for k, fn in legs.items():
                    ms, out = event_ms(lambda: fn(gds[(d, k)]))
                    if r > 0:
                        res[name][k].append(ms)
                    outs[(name, k)] = out.cpu()
                flush.fill_(float(r)); torch.cuda.synchronize()
                ms, wav = event_ms(lambda: bench_step(gds[(d, "ddpm862")], r))
                if r > 0:
                    res[name]["bench"].append(ms)
                outs[(name, "bench")] = wav.cpu()
    per = {"ddpm862": 1000, "ddpm43": 1000, "b8x689": 200}
    lines = ["card: %s" % card(), "rounds: %d per schedule, alternating old/new; median (min .. max)" % args.rounds, ""]
    summary = {}
    for k in list(legs) + ["bench"]:
        row = {}
        for name in ("old", "new"):
            v = res[name][k]
            if k in per:
                v = [x * 1000.0 / per[k] for x in v]            # us per DDPM step
                unit = "us/step"
            elif k == "bench":
                v = [862 * HOP / SR / (x / 1000.0) for x in v]  # audio-sec/s
                unit = "audio-sec/s"
            else:
                unit = "ms/call"
            row[name] = v
        mo, mn = statistics.median(row["old"]), statistics.median(row["new"])
        same = torch.equal(outs[("old", k)], outs[("new", k)])
        summary[k] = {"unit": unit, "old": row["old"], "new": row["new"], "old_median": mo, "new_median": mn,
                      "change_pct": (mn - mo) / mo * 100.0, "bit_identical": same}
        lines.append("%-8s %-12s old %9.2f (%9.2f .. %9.2f)   new %9.2f (%9.2f .. %9.2f)   %+6.2f %%   bit-identical: %s" % (
            k, unit, mo, min(row["old"]), max(row["old"]), mn, min(row["new"]), max(row["new"]), (mn - mo) / mo * 100.0, same))
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n\n" + json.dumps(summary, indent=1) + "\n")


if __name__ == "__main__":
    main()

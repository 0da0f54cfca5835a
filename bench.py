#!/usr/bin/env python
"""bench.py -- BASELINE.json's headline metric on synthetic inputs.

  metric  : audio-sec/s (= 1/RTF) for 1000-step DDPM @ 44.1 kHz, NSF-HiFiGAN vocoder
  workload: BASELINE.json configs[1]: one 10 s clip (862 mel frames, 128 bins) per GPU.  At N > 1 every rank runs
            its own clip (weak scaling) and the final waveforms are all-gathered with NCCL inside the timed step.
  a "step": one full pass of the hot path over the batch: 1000 DDPM denoising steps through the 20-layer WaveNet,
            denormalise + clip, NSF-HiFiGAN mel -> waveform.

  python bench.py --gpus N --steps K --warmup W            (our arm; torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  (the reference's own CPU modules from baseline/_ref,
                                                            rank 0 only, a bounded sample per step)
Prints ONE JSON line on rank 0.  Besides the contract keys the line carries (verdict r1, items 2 and 6):
  roofline        dominant kernel timed live; frac (algorithmic), frac_executed (x3 passes), the parity-mode ceiling
  layer_budget    conv / out-projection kernel us, us per DDPM step, what is left per kernel boundary
  cfg3_sliced_batch   BASELINE configs[3]: 8 ragged slices per GPU (64 at N = 8) through sharding.partition_slices
                  -> per-rank ragged batch -> sharding.gather_waveforms (NCCL); per-rank busy times, gather us
  extras (N = 1)  configs[2] (PNDM-25 latency), configs[4] (0.5 s chunk p50), stock-PyTorch-eager-on-B200 baseline
  cpu_baseline    the reference's CPU path on this box's host cores (N = 1 only)
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import synthetic as S  # noqa: E402  (neutral fixtures: seeded weights / utterances; not the checker)

SR, HOP, MEL, HID = 44100, 512, 128, 256
FLOP_EVAL_PER_FRAME = 47_677_440         # DiffNet eval, conditioner projections hoisted (SURVEY.md section 8d)
FLOP_COND_PER_FRAME = 7_864_320          # one-off conditioner projections of all 20 layers
FLOP_CONV_PER_FRAME = 2 * 3 * 384 * 768  # dilated conv of one layer (the dominant kernel)
FLOP_OUT_PER_FRAME = 2 * 384 * 768       # output projection of one layer
FLOP_VOC_PER_FRAME = 648_527_872
PASSES = 3                               # fp16 hi/lo split: xh*wh + xh*wl + xl*wh on the tensor pipe (DESIGN.md 3.1)
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--batch", type=int, default=1, help="clips per GPU")
    ap.add_argument("--frames", type=int, default=862, help="mel frames per clip (862 = 10 s @ 44.1 kHz)")
    ap.add_argument("--ddpm-steps", type=int, default=1000)
    ap.add_argument("--math", default="tc3f16", choices=["tc3f16", "fp32", "tc1f16"])
    ap.add_argument("--ref-ddpm-sample", type=int, default=20, help="reference arm: DDPM steps timed per bench step")
    ap.add_argument("--no-extras", action="store_true", help="headline only (skip cfg2/cfg3/cfg4/eager/cpu legs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the waveform the last timed step returned to DIR/wav.npy (float32; every rank's clips at N > 1)")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------ helpers
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.p = index, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200",
                                       "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 9 for i in range(4) if r[5 + i].lower().startswith("active")})
        pw = [float(r[3]) for r in self.rows if len(r) >= 9 and r[3].replace(".", "").isdigit()]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "power_w_max": max(pw) if pw else None}


def synth_inputs(B, T, seed):
    """Synthetic utterances: hubert-like units at 50 fps gathered to T mel frames, log2-f0, all frames valid."""
    g = torch.Generator().manual_seed(seed)
    Th = max(2, int(T * 50 * HOP / SR))
    hubert = torch.randn(B, Th, HID, generator=g) * 0.5
    mel2ph = (torch.arange(T, dtype=torch.float32) * (Th / T)).long().clamp(max=Th - 1)[None].repeat(B, 1) + 1
    f0_hz = S.synth_f0(B, T, seed=seed + 1)
    f0 = torch.where(f0_hz > 0, torch.log2(f0_hz.clamp(min=1.0)), torch.zeros_like(f0_hz))   # norm_interp_f0 'log'
    return hubert, mel2ph, f0, f0_hz


def build_models(math_mode, ddpm_steps):
    import diffsvc_b200 as D
    from diffsvc_b200.hparams import hparams, DEFAULTS_44K
    hparams.clear(); hparams.update(DEFAULTS_44K); hparams["pndm_speedup"] = 1
    torch.manual_seed(0)                     # the conditioning encoder's pitch embedding comes from the default generator
    sd = S.synth_diffnet_weights()
    dn = D.DiffNet(MEL, math_mode=math_mode)
    dn.load_state_dict(sd, strict=True)
    gd = D.GaussianDiffusion(None, MEL, dn, timesteps=1000, K_step=ddpm_steps, loss_type="l2", spec_min=[-5.0], spec_max=[0.0])
    gd = gd.cuda().eval()
    nsd = S.synth_nsf_weights(S.NSF_H_44K)
    voc = D.NsfHifiGAN.from_state_dict(dict(S.NSF_H_44K), nsd, device="cuda")
    return gd, voc, sd, nsd


# ------------------------------------------------------------------------------------------ CPU arm
class ReferenceCpu:
    """The reference's CPU path for this workload: its OWN `GaussianDiffusion.forward(infer=True)` (network/diff/
    diffusion.py:227-284) and `Generator.forward` (modules/nsf_hifigan/models.py:361-387) imported unmodified from
    baseline/_ref (kind "reference"); the oracle port of the same modules when that copy is absent (kind "port")."""

    def __init__(self, T, n_ddpm, device="cpu"):
        self.T, self.n, self.device = T, n_ddpm, device
        self.sd, self.nsd = S.synth_diffnet_weights(), S.synth_nsf_weights(S.NSF_H_44K)
        self.kind = "reference" if os.path.isdir(os.path.join(REF_DIR, "network", "diff")) else "port"
        if self.kind == "reference":
            import contextlib
            os.environ["DIFFSVC_REFERENCE_ROOT"] = REF_DIR
            sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
            import ref_harness as rh
            with contextlib.redirect_stdout(sys.stderr):             # the reference prints while it builds: keep stdout = ONE JSON line
                hp = rh.install()
                diffusion, net = rh.import_diffusion()
                models = rh.import_nsf_models()
                from modules.nsf_hifigan.env import AttrDict
                self.gd = diffusion.GaussianDiffusion(None, MEL, net.DiffNet(MEL), timesteps=1000, K_step=n_ddpm, loss_type="l2",
                                                      spec_min=[-5.0], spec_max=[0.0]).eval()
                self.gd.denoise_fn.load_state_dict(self.sd, strict=True)
                self.gen = models.Generator(AttrDict(S.NSF_H_44K)).eval()
                self.gen.remove_weight_norm()
                self.gen.load_state_dict(self.nsd)
            self.gd.to(device); self.gen.to(device)
            hp["pndm_speedup"] = 1
        else:
            from oracle import diffsvc_oracle as O
            self.O = O
            self.sched = O.make_schedule(O.linear_beta_schedule(1000, 0.02))
        self.inputs = synth_inputs(1, T, seed=5)

    def eval_once(self):
        g = torch.Generator().manual_seed(0)
        x = torch.randn(1, 1, MEL, self.T, generator=g).to(self.device); c = torch.randn(1, HID, self.T, generator=g).to(self.device)
        t = torch.tensor([5], device=self.device)
        with torch.no_grad():
            if self.kind == "reference":
                self.gd.denoise_fn(x, t, c)
            else:
                self.O.diffnet_forward(self.sd, x, t, c)

    def autotune_threads(self):
        """The thread count that runs one DiffNet eval fastest on this host (many-core boxes oversubscribe badly on
        these small convs); the reference gets its best configuration."""
        best, ncpu = None, os.cpu_count() or 1
        for n in sorted({min(ncpu, k) for k in (8, 16, 32, 64, ncpu)}):
            torch.set_num_threads(n)
            self.eval_once()
            dt = 1e9
            for _ in range(3):                                       # best of 3: one noisy eval must not pick the thread count
                t0 = time.perf_counter(); self.eval_once(); dt = min(dt, time.perf_counter() - t0)
            if best is None or dt < best[1]:
                best = (n, dt)
        torch.set_num_threads(best[0])
        return best[0]

    def sample(self):
        """n DDPM steps (through the public forward) + one vocoder pass of ONE clip -> (s sampler, s vocoder)."""
        hubert, mel2ph, f0, f0_hz = (t.to(self.device) for t in self.inputs)
        sync = torch.cuda.synchronize if self.device != "cpu" else (lambda: None)
        with torch.no_grad():
            sync(); t0 = time.perf_counter()
            if self.kind == "reference":
                import contextlib
                with contextlib.redirect_stderr(open(os.devnull, "w")):        # tqdm progress bars
                    ret = self.gd(hubert, mel2ph, None, None, f0.clone(), None, None, infer=True)
                mel = ret["mel_out"]
            else:
                O = self.O
                g = torch.Generator().manual_seed(1)
                cond = torch.randn(1, HID, self.T, generator=g) * 0.5
                x = torch.randn(1, 1, MEL, self.T, generator=g)
                noise = torch.randn(self.n, 1, 1, MEL, self.T, generator=g)
                mel = O.mel_from_x(O.sample(self.sd, self.sched, cond, x, self.n, noise), torch.tensor([[[-5.0]]]), torch.tensor([[[0.0]]]))
            sync(); t1 = time.perf_counter()
            mel = mel.clamp(-6.0, 1.5)                                           # after_infer clip (infer_tool.py:183)
            if self.kind == "reference":
                self.gen((2.30259 * mel).transpose(1, 2), f0_hz)                  # nsf_hifigan.py:39-43
            else:
                g = torch.Generator().manual_seed(2)
                self.O.spec2wav(self.nsd, S.NSF_H_44K, mel, f0_hz, torch.rand(1, 9, generator=g), torch.randn(1, self.T * HOP, 9, generator=g))
            sync(); t2 = time.perf_counter()
        return t1 - t0, t2 - t1


def run_reference(args, rank):
    """`--impl reference`: rank 0 only.  Each bench step times a bounded sample (n of 1000 DDPM steps + one vocoder
    pass of one clip); `value` extrapolates the DDPM part linearly to the full clip, `ms_per_step` is what was
    actually timed (so steps x ms_per_step is the wall time of the timed region)."""
    if rank != 0:
        return
    T, n = args.frames, args.ref_ddpm_sample
    ref = ReferenceCpu(T, n)
    threads = ref.autotune_threads()
    per_clip, timed = [], []
    for i in range(args.warmup + args.steps):
        td, tv = ref.sample()
        if i >= args.warmup:
            per_clip.append(td / n * args.ddpm_steps + tv); timed.append(td + tv)
    audio = T * HOP / SR
    clip_s = sum(per_clip) / len(per_clip)
    val = audio / clip_s
    line = base_line(args, val, sum(timed) / len(timed) * 1000.0)
    line.update({"impl": "reference", "dtype": "f32", "gpu_launches": 0, "extrapolated_ms_per_clip": clip_s * 1000.0,
                 "cpu_baseline": {"value": val, "unit": "audio-sec/s", "cores": threads, "kind": ref.kind,
                                  "sample": "%d of %d DDPM steps + 1 NSF-HiFiGAN pass of one %d-frame clip per bench step (ms_per_step = "
                                            "that sample), DDPM part extrapolated linearly to the clip; %s, torch CPU fp32, %d threads "
                                            "(autotuned of %d cpus)" % (n, args.ddpm_steps, T, _kind_text(ref.kind), threads, os.cpu_count() or 1)},
                 "e2e": {"value": val, "unit": "audio-sec/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    emit(line)


def _kind_text(kind):
    return ("the reference's own GaussianDiffusion.forward + Generator.forward from baseline/_ref" if kind == "reference"
            else "oracle port of the reference modules (baseline/_ref absent)")


def base_line(args, value, ms_per_step):
    return {"metric": "audio-sec/s (1/RTF), 1000-step DDPM @44.1kHz + NSF-HiFiGAN", "value": value, "unit": "audio-sec/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic",
            "config": {"workload": "BASELINE configs[1]: %d clip(s)/GPU x %d frames (%.2f s @44.1kHz, 128 mel bins), "
                                   "%d-step DDPM + NSF-HiFiGAN" % (args.batch, args.frames, args.frames * HOP / SR, args.ddpm_steps),
                       "batch_per_gpu": args.batch, "frames": args.frames, "ddpm_steps": args.ddpm_steps,
                       "parallelism": "independent clips per GPU, NCCL all-gather of waveforms" if args.gpus > 1 else "single GPU",
                       "l2": "256 MiB L2 flush between timed steps"}}


# ------------------------------------------------------------------------------------------ our arm
def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); out = fn(); b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b), out


def cfg3_sliced_batch(gd, voc, dist, rank, world, flush, n_warm=1, n_timed=2):
    """BASELINE configs[3] (SURVEY.md section 8e): 8 ragged slices (~8 s +- 25 %) per GPU -- 64 on 8 GPUs --
    partitioned longest-first onto the ranks, each rank runs its ragged sub-batch (per-item lengths) through the
    1000-step sampler + vocoder, and ONE variable-length all-gather of the waveforms reassembles the job."""
    from diffsvc_b200 import sharding
    n_slices = 8 * world
    g = torch.Generator().manual_seed(4242)
    lengths = (689 * (0.75 + 0.5 * torch.rand(n_slices, generator=g))).round().long().tolist()
    bins = sharding.partition_slices(lengths, world)
    mine = bins[rank]
    lens = [lengths[i] for i in mine]
    T = max(lens)
    hubert, mel2ph, f0, f0_hz = synth_inputs(len(mine), T, seed=900 + rank)
    for k, n in enumerate(lens):                                     # ragged: frames beyond an item's length are padding
        mel2ph[k, n:] = 0; f0[k, n:] = 0; f0_hz[k, n:] = 0
    with torch.no_grad():
        ret0 = gd.fs2(hubert.cuda(), mel2ph.cuda(), None, None, f0.cuda().clone(), None, None, skip_decoder=True, infer=True)
    cond = ret0["decoder_inp"].transpose(1, 2).contiguous()
    x0 = torch.randn(len(mine), 1, MEL, T, device="cuda")
    f0hz_d = f0_hz.cuda()
    busy, gather, total, samp = [], [], [], []
    for i in range(n_warm + n_timed):
        if dist is not None:
            dist.barrier()
        flush.fill_(float(i)); torch.cuda.synchronize()
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record()
        with torch.no_grad():
            x = gd.sample(x0, cond, 1000, None, None, lengths=lens, seed=31 + i)
            e[3].record()
            mel = gd.denorm_spec(x[:, 0].transpose(1, 2)).clamp(-6.0, 1.5)
            # the vocoder has no per-item boundary: vocode each slice alone (B = 1 semantics, as infer_tool.py:277 does)
            wavs = [voc.spec2wav_torch(mel[k:k + 1, :n], f0=f0hz_d[k:k + 1, :n], seed=8 * i + k) for k, n in enumerate(lens)]
        e[1].record()
        if dist is not None:
            full = sharding.gather_waveforms(wavs, mine, n_slices, device=torch.device("cuda", torch.cuda.current_device()))
            assert len(full) == n_slices and all(full[j].numel() == lengths[j] * HOP for j in range(n_slices))
        e[2].record(); torch.cuda.synchronize()
        if i >= n_warm:
            busy.append(e[0].elapsed_time(e[1])); gather.append(e[1].elapsed_time(e[2])); total.append(e[0].elapsed_time(e[2]))
            samp.append(e[0].elapsed_time(e[3]))
    stats = torch.tensor([sum(busy) / n_timed, sum(gather) / n_timed, sum(total) / n_timed, float(sum(lens)), sum(samp) / n_timed],
                         device="cuda", dtype=torch.float64)
    if dist is not None:
        allst = [torch.empty_like(stats) for _ in range(world)]
        dist.all_gather(allst, stats)
    else:
        allst = [stats]
    allst = torch.stack(allst).cpu()
    job_ms = float(allst[:, 2].max())
    audio = sum(lengths) * HOP / SR
    return {"workload": "BASELINE configs[3]: %d ragged slices (689 frames +- 25 %%, %.1f s audio in total), 1000-step DDPM + NSF-HiFiGAN, "
                        "sharding.partition_slices -> per-rank sub-batch, packed back to back on one frame axis (DESIGN.md 3.1e) -> "
                        "sharding.gather_waveforms" % (n_slices, audio),
            "n_slices": n_slices, "audio_sec_per_s": audio / (job_ms / 1000.0), "job_ms": job_ms,
            "per_rank_busy_ms": [round(float(v), 2) for v in allst[:, 0]], "per_rank_frames": [int(v) for v in allst[:, 3]],
            "per_rank_us_per_ddpm_step": [round(float(v), 1) for v in allst[:, 4]],          # sampler alone: ms per 1000 steps = us per step
            "sampler_algorithmic_tflops_per_rank": [round(float(f) * FLOP_EVAL_PER_FRAME * 1000 / (float(v) * 1e-3) / 1e12, 1)
                                                    for f, v in zip(allst[:, 3], allst[:, 4])],
            "gather_ms_max": float(allst[:, 1].max()), "imbalance": float(allst[:, 0].max() / allst[:, 0].mean()),
            "timed_passes": n_timed}


def latency_configs(gd, voc):
    """configs[2] (PNDM-25, 10 s clip) and configs[4] (flask: 0.5 s chunk, PNDM-50) through the public classes with
    host inputs: wall-clock per call incl. H2D / D2H, synchronised."""
    from diffsvc_b200.hparams import hparams

    def run(T, speedup, n_calls, warm):
        hparams["pndm_speedup"] = speedup
        hub, m2p, f0, f0hz = (t.pin_memory() for t in synth_inputs(1, T, seed=3))
        out = torch.empty(T * HOP).pin_memory()
        ts = []
        for i in range(warm + n_calls):
            torch.cuda.synchronize(); t0 = time.perf_counter()
            ret = gd(hub.cuda(non_blocking=True), m2p.cuda(non_blocking=True), None, None, f0.cuda(non_blocking=True), None, None, infer=True)
            wav = voc.spec2wav_torch(ret["mel_out"].clamp(-6.0, 1.5), f0=f0hz.cuda(non_blocking=True), seed=i)
            out.copy_(wav); torch.cuda.synchronize()
            if i >= warm:
                ts.append(time.perf_counter() - t0)
        return ts
    try:
        with torch.no_grad():
            a = run(862, 40, 10, 3)
            b = run(43, 20, 100, 5)
    finally:
        hparams["pndm_speedup"] = 1
    return {"cfg2_pndm25_10s": {"latency_ms_p50": statistics.median(a) * 1e3, "audio_sec_per_s": 862 * HOP / SR / statistics.median(a)},
            "cfg4_flask_0.5s_pndm50": {"latency_ms_p50": statistics.median(b) * 1e3, "latency_ms_p95": sorted(b)[int(0.95 * len(b))] * 1e3,
                                       "rtf": statistics.median(b) / (43 * HOP / SR)}}


def eager_baseline(T):
    """Second baseline (SURVEY.md section 8d): the reference's modules through STOCK PyTorch eager on this B200
    (cuDNN / cuBLAS, fp32, TF32 off), same workload, bounded sample (30 DDPM steps + 1 vocoder pass)."""
    tf = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False; torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ref = ReferenceCpu(T, 30, device="cuda")
        if ref.kind != "reference":
            raise RuntimeError("baseline/_ref absent: no reference modules to run under torch eager")
        ref.sample()
        td, tv = ref.sample()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf
    return {"kind": ref.kind, "ms_per_ddpm_step": td / 30 * 1e3, "vocoder_ms": tv * 1e3,
            "audio_sec_per_s": (T * HOP / SR) / (td / 30 * 1000 + tv), "note": "30 of 1000 DDPM steps timed, extrapolated; fp32, TF32 off"}


def profile_traffic(B, T):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this shape
    (profiles/traffic.json, written by tools/ncu_summary.py); None when no capture of this shape is committed."""
    try:
        table = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        e = table.get("conv_gate_B%d_T%d" % (B, T))
        return (e["dram_bytes_per_launch"], e["source"]) if e else (None, None)
    except Exception:
        return None, None


DUMP_LIMIT_BYTES = 64_000_000 - 4096       # 64 MB for everything written, .npy headers included


def dump_outputs(out_dir, wav):
    """DIR/wav.npy: the [clips, samples] float32 waveform of the last timed step, so that two builds run with the same
    arguments can be compared output for output.  The files stay within 64 MB in all: above that a fixed sample is
    kept, every k-th sample of the flattened array, k the least stride that fits (the stride goes to DIR/wav_stride.npy)."""
    import numpy as np
    a = wav.detach().float().cpu().numpy()
    stride = -(-a.nbytes // DUMP_LIMIT_BYTES)
    os.makedirs(out_dir, exist_ok=True)
    if stride > 1:
        a = a.reshape(-1)[::stride].copy()
        np.save(os.path.join(out_dir, "wav_stride.npy"), np.array([stride], dtype=np.float64))
    np.save(os.path.join(out_dir, "wav.npy"), a)


def emit(line):
    """The ONE JSON line, on the real stdout (fd saved in main() before everything else was pointed at stderr)."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    # stdout carries exactly one JSON line: libraries that print there (NCCL's version banner at communicator creation,
    # the reference's progress output) are sent to stderr for the whole run, at the file-descriptor level
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank)
    assert torch.cuda.is_available(), "bench.py needs a B200 (there is no CPU fallback on the product path)"
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus, "launch with torchrun --nproc-per-node %d (WORLD_SIZE=%d)" % (args.gpus, world)
    from diffsvc_b200 import _lib
    lib = _lib.load()
    B, T, NS = args.batch, args.frames, args.ddpm_steps
    gd, voc, sd, nsd = build_models(args.math, NS)
    hubert, mel2ph, f0, f0_hz = synth_inputs(B, T, seed=1000 + rank)
    pin = lambda t: t.pin_memory()
    h_hubert, h_mel2ph, h_f0, h_f0hz = pin(hubert), pin(mel2ph), pin(f0), pin(f0_hz)
    h_wav = torch.empty(B * T * HOP, dtype=torch.float32).pin_memory()
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")
    gathered = torch.empty(world * B * T * HOP, dtype=torch.float32, device="cuda") if world > 1 else None

    def vocode(mel, f0d, seed):
        mel = mel.clamp(-6.0, 1.5)                                   # after_infer clip (infer_tool.py:183)
        wav = voc.spec2wav_torch(mel, f0=f0d, seed=seed)
        if world > 1:
            dist.all_gather_into_tensor(gathered, wav)               # C0: the only cross-GPU exchange
        return wav

    # device-resident arm: conditioning + initial noise already in HBM
    with torch.no_grad():
        ret0 = gd.fs2(hubert.cuda(), mel2ph.cuda(), None, None, f0.cuda().clone(), None, None, skip_decoder=True, infer=True)
    cond_d = ret0["decoder_inp"].transpose(1, 2).contiguous()
    x0_d = torch.randn(B, 1, MEL, T, generator=torch.Generator().manual_seed(2000 + rank)).cuda()   # same x_T every run
    f0hz_d = f0_hz.cuda()

    def step_device(i):
        x = gd.sample(x0_d, cond_d, NS, None, None, seed=17 + i)
        mel = gd.denorm_spec(x[:, 0].transpose(1, 2))
        return vocode(mel, f0hz_d, seed=i)

    def step_e2e(i):
        hub = h_hubert.cuda(non_blocking=True); m2p = h_mel2ph.cuda(non_blocking=True)
        f0d = h_f0.cuda(non_blocking=True); f0hz = h_f0hz.cuda(non_blocking=True)
        ret = gd(hub, m2p, None, None, f0d, None, None, infer=True, seed=17 + i)     # the public call (diffusion.py:227)
        wav = vocode(ret["mel_out"], f0hz, seed=i)
        h_wav.copy_(wav, non_blocking=True)
        return wav

    def timed(fn, n_warm, n_steps, sampler=None):
        """ms per step (max over ranks of the per-rank sums), every rank's own ms per step, what the last step returned."""
        tot, out = 0.0, None
        for i in range(n_warm + n_steps):
            if dist is not None:
                dist.barrier()
            flush.fill_(float(i)); torch.cuda.synchronize()
            if i == n_warm and sampler is not None:
                sampler.start()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); out = fn(i); b.record()
            torch.cuda.synchronize()
            if i >= n_warm:
                tot += a.elapsed_time(b)
        per_rank = [tot / n_steps]
        if dist is not None:
            t = torch.tensor([tot / n_steps], device="cuda", dtype=torch.float64)
            every = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(every, t)
            per_rank = [float(v.item()) for v in every]
        return max(per_rank), per_rank, out

    with torch.no_grad():
        clk = ClockSampler(local)
        l0 = lib.dsvc_launch_count()
        ms_dev, ranks_dev, wav_dev = timed(step_device, args.warmup, args.steps, clk)
        clocks = clk.stop()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, (gathered if world > 1 else wav_dev).reshape(world * B, T * HOP))
        launches = (lib.dsvc_launch_count() - l0) // (args.warmup + args.steps) * args.steps
        ms_e2e, ranks_e2e, _ = timed(step_e2e, args.warmup, args.steps)
        # sampler alone, and the two kernels of a layer alone (CUDA events on the launch stream, back to back)
        ms_sampler, _ = event_ms(lambda: gd.sample(x0_d, cond_d, NS, None, None, seed=3))
        h = gd.denoise_fn.handle()
        it = 200
        stream = _lib.current_stream()

        def kernel_us(part):
            _lib.check(lib.dsvc_diffnet_run_layer(h, 5, part, 20, stream))
            ms, _ = event_ms(lambda: _lib.check(lib.dsvc_diffnet_run_layer(h, 5, part, it, stream)))
            return ms / it * 1000.0
        conv_us, out_us = kernel_us(0), kernel_us(1)

    audio = world * B * T * HOP / SR
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_burst = float(peaks.get("bf16_tflops", 1590.0))
    peak_sus = float(peaks.get("bf16_tflops_sustained", 1400.0))
    conv_tf = FLOP_CONV_PER_FRAME * B * T / conv_us / 1e6
    out_tf = FLOP_OUT_PER_FRAME * B * T / out_us / 1e6
    sampler_flop = (FLOP_EVAL_PER_FRAME * NS + FLOP_COND_PER_FRAME) * B * T
    step_us = ms_sampler * 1000.0 / NS
    L = 20
    traffic, traffic_src = profile_traffic(B, T)
    line = base_line(args, audio / (ms_dev / 1000.0), ms_dev)
    line.update({
        "dtype": "f32 (fp16 hi/lo split x3 on tcgen05, fp32 accumulate)" if args.math == "tc3f16" else args.math,
        "clocks": clocks, "gpu_launches": int(launches),
        "per_rank_ms_per_step": [round(v, 3) for v in ranks_dev],
        "e2e": {"value": audio / (ms_e2e / 1000.0), "unit": "audio-sec/s", "ms_per_step": ms_e2e,
                "per_rank_ms_per_step": [round(v, 3) for v in ranks_e2e],
                "h2d_bytes_per_step": int(sum(t.numel() * t.element_size() for t in (h_hubert, h_mel2ph, h_f0, h_f0hz))),
                "d2h_bytes_per_step": int(h_wav.numel() * 4), "api": "GaussianDiffusion.forward + NsfHifiGAN.spec2wav_torch"},
        "roofline": {"bound": "tensor", "kernel": "tc_pair_kernel<EpiGate, 64> (dilated conv k3 + conditioner + gate of one layer; cta_group::2 CTA pairs)",
                     "achieved": conv_tf, "peak": peak_burst, "unit": "TFLOP/s", "frac": conv_tf / peak_burst,
                     "frac_executed": PASSES * conv_tf / peak_burst, "frac_ceiling_parity_mode": 1.0 / PASSES,
                     "audio_sec_per_s_ceiling_parity_mode": peak_burst * 1e12 / PASSES / (FLOP_EVAL_PER_FRAME * NS * SR / HOP),
                     "traffic": traffic, "traffic_source": traffic_src, "us_per_launch": conv_us,
                     "note": "achieved = algorithmic fp32-equivalent FLOPs (2*3*C*2C per frame x frames) / CUDA-event time of the kernel "
                             "run back to back in this process; the error-compensated fp16 hi/lo split executes 3x those FLOPs on the "
                             "tensor pipe, so frac <= 0.33 and 1000-step DDPM <= ~139 audio-sec/s per B200 in parity mode; "
                             "traffic = dram bytes per launch read from profiles/traffic.json (ncu --set full of this kernel at this "
                             "shape), null when no capture of this shape is committed; peak = MEASURED_PEAKS.json bf16_tflops (burst)"
                             + ("" if peaks else " [fallback]")},
        "layer_budget": {"conv_gate_us": conv_us, "out_proj_us": out_us, "out_proj_tflops": out_tf,
                         "ddpm_step_us": step_us, "kernels_per_step": 2 * L + 3,
                         "boundary_us_per_kernel": (step_us - L * (conv_us + out_us)) / (2 * L + 3),
                         "note": "conv_gate_us / out_proj_us = launch-to-launch period of one kernel repeated back to back (so each "
                                 "includes one kernel boundary: drain, dependent release, first operand tiles); ddpm_step_us = 1000-step "
                                 "sampler alone / 1000; boundary_us_per_kernel = what a step costs beyond 20 x (conv + out-proj) periods, "
                                 "spread over its 43 kernels (head / tail kernels, the conv <-> out-proj alternation)"},
        "sampler_flops": {"achieved_tflops": sampler_flop / (ms_sampler / 1000.0) / 1e12, "peak_sustained": peak_sus,
                          "frac_of_sustained": sampler_flop / (ms_sampler / 1000.0) / 1e12 / peak_sus,
                          "note": "algorithmic DiffNet FLOPs of the whole 1000-step sampler / its CUDA-event time"},
    })
    if not args.no_extras:
        with torch.no_grad():
            line["cfg3_sliced_batch"] = cfg3_sliced_batch(gd, voc, dist, rank, world, flush)
    if rank == 0 and world == 1 and not args.no_extras:
        # single-GPU legs only: the other ranks would idle at the barrier
        line["extras"] = latency_configs(gd, voc)
        try:
            line["extras"]["torch_eager_b200"] = eager_baseline(T)
        except Exception as ex:                                      # a baseline, never a reason to lose the bench line
            line["extras"]["torch_eager_b200"] = {"unavailable": repr(ex)[:200]}
        ref = ReferenceCpu(T, args.ref_ddpm_sample)
        threads = ref.autotune_threads()
        ref.sample()
        td, tv = ref.sample()
        per_clip = td / args.ref_ddpm_sample * NS + tv
        line["cpu_baseline"] = {"value": (T * HOP / SR) / per_clip, "unit": "audio-sec/s", "cores": threads, "kind": ref.kind,
                                "sample": "%d of %d DDPM steps (%.2f s) + 1 NSF-HiFiGAN pass (%.2f s) of one %d-frame clip, DDPM part "
                                          "extrapolated linearly; %s, torch CPU fp32, %d threads"
                                          % (args.ref_ddpm_sample, NS, td, tv, T, _kind_text(ref.kind), threads)}
    if rank == 0:
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

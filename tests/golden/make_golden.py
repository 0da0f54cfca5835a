"""Generate golden input/output vectors from the UNMODIFIED reference (CPU, fp32).

Run once, with DIFFSVC_REFERENCE_ROOT pointing at a checkout of the reference:

    python tests/golden/make_golden.py                 # the small-size fixtures
    python tests/golden/make_golden.py --only-full     # full_44k.npz (tests/test_oracle_vs_reference.py)

It imports the reference's own `DiffNet`, `GaussianDiffusion` (incl. its FastSpeech2
conditioning) and NSF-HiFiGAN `Generator`, builds them at SMALL sizes with seeded
weights, records every random draw the reference makes (torch.randn / rand /
randn_like are wrapped), and writes weights + inputs + draws + outputs to
`tests/golden/*.npz`.  The reference has no tests of its own for this path
(SURVEY.md section 4), so these fixtures are what pins `oracle/diffsvc_oracle.py`.
The fixtures travel to the GPU box; the reference does not.
"""
import os
import sys
from collections import deque

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_harness as rh  # noqa: E402
sys.path.insert(0, os.path.join(HERE, "..", "..", "oracle"))
import diffsvc_oracle as O  # noqa: E402  (only gen_mel uses it: the librosa mel basis stand-in)

SMALL = dict(hidden_size=32, residual_layers=4, residual_channels=64, dilation_cycle_length=2,
             audio_num_mel_bins=16, keep_bins=16)


class DrawRecorder:
    """Wraps torch.randn / rand / randn_like so every draw of the reference is logged in order."""

    def __init__(self):
        self.log = []

    def __enter__(self):
        self._orig = (torch.randn, torch.rand, torch.randn_like)
        o_randn, o_rand, o_randn_like = self._orig

        def randn(*a, **k):
            r = o_randn(*a, **k); self.log.append(("randn", r.clone())); return r

        def rand(*a, **k):
            r = o_rand(*a, **k); self.log.append(("rand", r.clone())); return r

        def randn_like(*a, **k):
            r = o_randn_like(*a, **k); self.log.append(("randn_like", r.clone())); return r

        torch.randn, torch.rand, torch.randn_like = randn, rand, randn_like
        return self

    def __exit__(self, *exc):
        torch.randn, torch.rand, torch.randn_like = self._orig


def _np(sd, prefix="sd/"):
    return {prefix + k: v.detach().cpu().numpy() for k, v in sd.items()}


def build_small_diffusion(hp, spec_min, spec_max, K_step, seed):
    diffusion, net = rh.import_diffusion()
    torch.manual_seed(seed)
    dn = net.DiffNet(hp["audio_num_mel_bins"])
    torch.nn.init.normal_(dn.output_projection.weight, std=0.05)   # zero-init in the reference (net.py:110)
    gd = diffusion.GaussianDiffusion(None, hp["audio_num_mel_bins"], dn, timesteps=hp["timesteps"], K_step=K_step,
                                     loss_type=hp["diff_loss_type"], spec_min=spec_min, spec_max=spec_max)
    gd.eval()
    return gd, diffusion


def synth_inputs(B, T, Th, H, seed):
    g = torch.Generator().manual_seed(seed)
    hubert = torch.randn(B, Th, H, generator=g)
    mel2ph = torch.randint(1, Th + 1, (B, T), generator=g).sort(dim=1).values
    mel2ph[-1, T - 3:] = 0                       # padded tail on the last item
    f0 = torch.log2(torch.rand(B, T, generator=g) * 500 + 60)
    f0[0, 2:5] = torch.log2(torch.tensor(1300.0))  # above f0_max -> coarse bin clamp
    return hubert, mel2ph, f0


def gen_diffnet(hp):
    diffusion, net = rh.import_diffusion()
    torch.manual_seed(101)
    dn = net.DiffNet(hp["audio_num_mel_bins"]).eval()
    torch.nn.init.normal_(dn.output_projection.weight, std=0.05)
    g = torch.Generator().manual_seed(5)
    B, M, T, H = 2, hp["audio_num_mel_bins"], 24, hp["hidden_size"]
    spec = torch.randn(B, 1, M, T, generator=g)
    cond = torch.randn(B, H, T, generator=g) * 0.5
    t = torch.tensor([17, 503], dtype=torch.long)
    with torch.no_grad():
        out = dn(spec, t, cond)
    d = _np(dn.state_dict())
    d.update(spec=spec.numpy(), cond=cond.numpy(), t=t.numpy(), out=out.numpy(),
             dilation_cycle=np.int64(hp["dilation_cycle_length"]))
    np.savez_compressed(os.path.join(HERE, "diffnet_small.npz"), **d)
    print("diffnet_small: out", tuple(out.shape), float(out.abs().max()))


def gen_sampler(hp, name, K_step, speedup, spec_min, spec_max, use_gt_mel=False, add_noise_step=0, seed=7):
    gd, diffusion = build_small_diffusion(hp, spec_min, spec_max, K_step, seed)
    B, T, Th, H, M = 2, 20, 9, hp["hidden_size"], hp["audio_num_mel_bins"]
    hubert, mel2ph, f0 = synth_inputs(B, T, Th, H, seed + 1)
    ref_mels = torch.randn(B, T, M, generator=torch.Generator().manual_seed(seed + 2)) * 0.8 - 2.5
    hp["pndm_speedup"] = speedup
    kwargs = dict(use_gt_mel=True, add_noise_step=add_noise_step) if use_gt_mel else {}
    if speedup > 1:
        # the reference's PLMS path only works for B=1 (diffusion.py:186 python max on a tensor);
        # run items one at a time and stack -- per-item semantics (SURVEY.md section 8e)
        outs, draws = [], []
        for b in range(B):
            gd.noise_list = deque(maxlen=4)
            with DrawRecorder() as rec, torch.no_grad():
                ret = gd(hubert[b:b + 1], mel2ph[b:b + 1], None, ref_mels[b:b + 1], f0[b:b + 1].clone(), None, None,
                         infer=True, **kwargs)
            outs.append(ret)
            draws.append([r for _, r in rec.log])
        mel_out = torch.cat([o["mel_out"] for o in outs])
        dec = torch.cat([o["decoder_inp"] for o in outs])
        f0d = torch.cat([o["f0_denorm"] for o in outs])
        x_init = torch.cat([d[0] for d in draws])
        noises = np.zeros((0,), np.float32)
    else:
        with DrawRecorder() as rec, torch.no_grad():
            ret = gd(hubert, mel2ph, None, ref_mels, f0.clone(), None, None, infer=True, **kwargs)
        mel_out, dec, f0d = ret["mel_out"], ret["decoder_inp"], ret["f0_denorm"]
        log = [r for _, r in rec.log]
        x_init = log[0]                     # diffusion.py:268 (or the q_sample noise, :205)
        noises = torch.stack(log[1:]).numpy()
    # keep only what the inference path reads (the unused pitch_predictor / mel_out heads stay out)
    d = _np({k: v for k, v in gd.state_dict().items()
             if k.startswith("denoise_fn.") or not k.startswith("fs2.") or k == "fs2.pitch_embed.weight"})
    d.update(hubert=hubert.numpy(), mel2ph=mel2ph.numpy(), f0=f0.numpy(), ref_mels=ref_mels.numpy(),
             x_init=x_init.numpy(), noises=noises, mel_out=mel_out.numpy(), decoder_inp=dec.numpy(),
             f0_denorm=f0d.numpy(), K_step=np.int64(K_step), speedup=np.int64(speedup),
             use_gt_mel=np.int64(int(use_gt_mel)), add_noise_step=np.int64(add_noise_step),
             dilation_cycle=np.int64(hp["dilation_cycle_length"]),
             f0_bin=np.int64(hp["f0_bin"]), f0_max=np.float64(hp["f0_max"]), f0_min=np.float64(hp["f0_min"]))
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **d)
    print(name, ": mel_out", tuple(mel_out.shape), "draws", len(noises), float(mel_out.abs().max()))


def gen_nsf():
    models = rh.import_nsf_models()
    from modules.nsf_hifigan.env import AttrDict
    h = AttrDict(resblock="1", upsample_rates=[4, 2, 2], upsample_kernel_sizes=[8, 4, 4],
                 upsample_initial_channel=32, resblock_kernel_sizes=[3, 7],
                 resblock_dilation_sizes=[[1, 3, 5], [1, 3, 5]], num_mels=8, sampling_rate=16000)
    torch.manual_seed(55)
    gen = models.Generator(h).eval()
    # the reference's init (std 0.01) gives a ~0 waveform; perturb v/g so the test is not vacuous
    with torch.no_grad():
        for n, p in gen.named_parameters():
            if n.endswith("weight_v") or (n.endswith(".weight") and "noise_convs" in n):
                p.mul_(1.0 / (p.std() + 1e-8)).mul_(0.35 / np.sqrt(np.prod(p.shape[1:]) / (4 if n.startswith("ups") else 1)))
            if n.endswith("weight_g"):
                p.copy_(p * (1.0 + 0.3 * torch.randn_like(p)))
    ckpt_sd = {k: v.clone() for k, v in gen.state_dict().items()}     # weight_g / weight_v form
    g = torch.Generator().manual_seed(9)
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
    for k in ("upsample_rates", "upsample_kernel_sizes", "resblock_kernel_sizes", "resblock_dilation_sizes"):
        d["h/" + k] = np.asarray(h[k], dtype=np.int64)
    d["h/upsample_initial_channel"] = np.int64(32)
    d["h/num_mels"] = np.int64(8)
    d["h/sampling_rate"] = np.int64(16000)
    np.savez_compressed(os.path.join(HERE, "nsf_small.npz"), **d)
    print("nsf_small: wav", tuple(wav.shape), float(wav.abs().max()), float(wav.std()))


def gen_hifigan24k():
    """The 24 kHz vocoder's generator (modules/hifigan/hifigan.py:104-169), with and without the f0 source."""
    import modules.hifigan.hifigan as hg
    h = dict(resblock="1", upsample_rates=[4, 2], upsample_kernel_sizes=[8, 4], upsample_initial_channel=16,
             resblock_kernel_sizes=[3, 5], resblock_dilation_sizes=[[1, 3, 5], [1, 3, 5]], use_pitch_embed=True,
             audio_sample_rate=24000)
    torch.manual_seed(77)
    gen = hg.HifiGanGenerator(h).eval()
    with torch.no_grad():
        for n, p in gen.named_parameters():
            if n.endswith("weight_v") or (n.endswith(".weight") and "noise_convs" in n):
                p.mul_(1.0 / (p.std() + 1e-8)).mul_(0.35 / np.sqrt(np.prod(p.shape[1:]) / (4 if n.startswith("ups") else 1)))
            if n.endswith("weight_g"):
                p.copy_(p * (1.0 + 0.3 * torch.randn_like(p)))
    ckpt_sd = {k: v.clone() for k, v in gen.state_dict().items()}
    g = torch.Generator().manual_seed(19)
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
    d = _np(ckpt_sd, "ckpt/")
    d.update(mel=mel.numpy(), f0=f0.numpy(), rand_ini=rec.log[0][1].numpy(), sine_noise=rec.log[1][1].numpy(),
             wav_f0=wav_f0.numpy(), wav_plain=wav_plain.numpy())
    for k in ("upsample_rates", "upsample_kernel_sizes", "resblock_kernel_sizes", "resblock_dilation_sizes"):
        d["h/" + k] = np.asarray(h[k], dtype=np.int64)
    d["h/upsample_initial_channel"] = np.int64(16)
    d["h/audio_sample_rate"] = np.int64(24000)
    np.savez_compressed(os.path.join(HERE, "hifigan24k_small.npz"), **d)
    print("hifigan24k_small: wav", tuple(wav_f0.shape), float(wav_f0.std()), float(wav_plain.std()))


def synth_wave(n, sr, seed):
    """a few drifting partials + a little noise, peak < 1: stands in for a vocal recording"""
    g = np.random.default_rng(seed)
    t = np.arange(n) / sr
    f0 = 180.0 * 2.0 ** (0.3 * np.sin(2 * np.pi * 1.7 * t))
    phase = 2 * np.pi * np.cumsum(f0) / sr
    y = sum(a * np.sin(k * phase) for k, a in ((1, 0.4), (2, 0.2), (3, 0.1), (5, 0.05), (9, 0.02)))
    y = y * (0.6 + 0.4 * np.sin(2 * np.pi * 3.1 * t)) + 0.01 * g.standard_normal(n)
    y[: n // 10] *= 0.0005                      # a near-silent lead-in: exercises the low-energy / clip region
    return (0.9 * y / np.abs(y).max()).astype(np.float32)


def gen_mel():
    """STFT.get_mel of the reference (modules/nsf_hifigan/nvSTFT.py:72-104) on CPU.  librosa is absent here, so
    the harness serves `librosa.filters.mel` from the oracle's restatement (slaney_mel_basis): the fixture pins
    everything downstream of the basis matrix, and stores the matrix it used."""
    import modules.nsf_hifigan.nvSTFT as nv
    nv.librosa_mel_fn = lambda sr, n_fft, n_mels, fmin, fmax: O.slaney_mel_basis(sr, n_fft, n_mels, fmin, fmax)
    # nvSTFT.py:94 calls torch.stft without return_complex (torch 1.12, requirements.txt:90: a real [..., 2] view);
    # torch 2.x demands the argument, so the harness supplies the 1.12 behaviour.
    stft_now = torch.stft

    def stft_112(*a, **k):
        if "return_complex" in k:
            return stft_now(*a, **k)
        return torch.view_as_real(stft_now(*a, return_complex=True, **k))
    nv.torch.stft = stft_112
    d = {}
    for tag, (sr, n_mels, n_fft, win, hop, fmin, fmax, n) in {
            "a": (44100, 128, 2048, 2048, 512, 40, 16000, 13000),      # config_nsf.yaml
            "b": (24000, 80, 512, 512, 128, 30, 12000, 5000),          # config.yaml (24 kHz)
            "c": (22050, 80, 1024, 800, 256, 20, 11025, 6000)}.items():    # win_size < n_fft
        wav = synth_wave(n, sr, seed={"a": 1, "b": 2, "c": 3}[tag])
        stft = nv.STFT(sr, n_mels, n_fft, win, hop, fmin, fmax)
        with torch.no_grad():
            mel = stft.get_mel(torch.from_numpy(wav).unsqueeze(0))          # [1, n_mels, T] natural log
        d["%s/cfg" % tag] = np.array([sr, n_mels, n_fft, win, hop, fmin, fmax], dtype=np.int64)
        d["%s/wav" % tag] = wav
        d["%s/mel_ln" % tag] = mel.squeeze(0).numpy()
        d["%s/basis" % tag] = stft.mel_basis[str(fmax) + "_cpu"].numpy()
    torch.stft = stft_now
    np.savez_compressed(os.path.join(HERE, "mel_small.npz"), **d)
    print("mel_small", {k: v.shape for k, v in d.items()})


def gen_pe():
    """PitchExtractor of the reference (modules/fastspeech/pe.py:120-149), eval mode, seeded weights with
    non-trivial BatchNorm statistics; hidden 64 (the reference reads it from hparams)."""
    from utils.hparams import hparams
    import modules.fastspeech.pe as pe_mod
    old = {k: hparams.get(k) for k in ("hidden_size", "predictor_hidden")}
    hparams.update(hidden_size=64, predictor_hidden=-1)
    torch.manual_seed(99)
    m = pe_mod.PitchExtractor(n_mel_bins=80, conv_layers=2).eval()
    with torch.no_grad():
        for name, t in m.named_parameters():
            if name.endswith(".bias") or ".norm." in name or ".3." in name or ".2." in name:
                t.add_(0.1 * torch.randn_like(t))
        for name, b in m.named_buffers():
            if name.endswith("running_mean"):
                b.copy_(0.2 * torch.randn_like(b))
            if name.endswith("running_var"):
                b.copy_(0.5 + torch.rand_like(b))
        m.pitch_predictor.pos_embed_alpha.fill_(0.7)
        m.pitch_predictor.linear.bias.add_(torch.tensor([7.5, 0.0]))      # log2(f0) ~ 7.5 -> ~180 Hz
    B, T = 2, 50
    mel = (torch.randn(B, T, 80) * 1.2 - 3.0)
    mel[1, 37:] = 0                                                          # padding frames
    mel[0, 11, 0] = 0
    with torch.no_grad():
        ret = m(mel)
    d = {"mel": mel.numpy(), "pitch_pred": ret["pitch_pred"].numpy(), "f0_denorm_pred": ret["f0_denorm_pred"].numpy()}
    d.update(_np(m.state_dict()))
    np.savez_compressed(os.path.join(HERE, "pe_small.npz"), **d)
    hparams.update(old)
    print("pe_small", ret["pitch_pred"].shape, float(ret["f0_denorm_pred"].max()))


def full_pe_weights(shapes, seed=21):
    """Seeded PitchExtractor weights for the key -> shape table of the full-size module: fan-in scaled convs and
    projections, norm scales near 1, non-trivial BatchNorm statistics, and a predictor bias that puts log2(f0)
    near 7 (~130 Hz).  Rebuilt from the table alone, so the comparison needs no copy of the reference's module."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, shape in shapes.items():
        shape = tuple(int(s) for s in shape)
        if k.endswith("num_batches_tracked"):
            sd[k] = torch.zeros(shape, dtype=torch.long)
        elif k.endswith("running_mean"):
            sd[k] = 0.2 * torch.randn(shape, generator=g)
        elif k.endswith("running_var"):
            sd[k] = 0.5 + torch.rand(shape, generator=g)
        elif k.endswith("pos_embed_alpha") or k.endswith("_float_tensor"):
            sd[k] = torch.ones(shape)
        elif k.endswith(".weight") and len(shape) >= 2:
            sd[k] = torch.randn(shape, generator=g) / float(np.sqrt(np.prod(shape[1:])))
        elif k.endswith(".weight"):
            sd[k] = 1.0 + 0.1 * torch.randn(shape, generator=g)
        else:
            sd[k] = 0.1 * torch.randn(shape, generator=g)
    sd["pitch_predictor.linear.bias"] = sd["pitch_predictor.linear.bias"] + torch.tensor([7.0, 0.0])
    return sd


def full_inputs():
    """The inputs of tests/test_oracle_vs_reference.py, from their seeds."""
    g = torch.Generator().manual_seed(1)
    x = torch.randn(1, 1, 128, 96, generator=g)
    cond = torch.randn(1, 256, 96, generator=g) * 0.5
    noises = [torch.randn(1, 1, 128, 96, generator=g) for _ in range(3)]
    g = torch.Generator().manual_seed(2)
    T = 6
    voc_mel = torch.randn(1, 128, T, generator=g) * 2 - 5
    voc_f0 = O.synth_f0(1, T) + 100
    voc_f0[0, 2] = 0
    rand_ini = torch.rand(1, 9, generator=g)
    sine_noise = torch.randn(1, T * 512, 9, generator=g)
    g = torch.Generator().manual_seed(21)
    pe_mel = torch.randn(2, 120, 80, generator=g) - 3.0
    pe_mel[1, 100:] = 0
    g = torch.Generator().manual_seed(4)
    wav = (torch.rand(1, 30000, generator=g) * 2 - 1) * 0.3
    return dict(x=x, cond=cond, noises=noises, voc_mel=voc_mel, voc_f0=voc_f0, rand_ini=rand_ini, sine_noise=sine_noise,
                pe_mel=pe_mel, wav=wav)


FULL_T = (999, 500, 0)


def gen_full(hp):
    """The reference's modules at the FULL 44.1 kHz config (config_nsf.yaml) on seeded weights and inputs that
    tests/test_oracle_vs_reference.py rebuilds: reference outputs plus the key -> shape tables of its state dicts."""
    inp = full_inputs()
    d = {}
    diffusion, net = rh.import_diffusion()
    dn = net.DiffNet(128).eval()
    dn.load_state_dict(O.synth_diffnet_weights(), strict=True)
    gd = diffusion.GaussianDiffusion(None, 128, dn, timesteps=1000, K_step=1000, loss_type="l2",
                                     spec_min=hp["spec_min"], spec_max=hp["spec_max"]).eval()
    for k, v in dn.state_dict().items():
        d["dn_shape/" + k] = np.asarray(v.shape, dtype=np.int64)
    for k, v in gd.state_dict().items():                    # what a model checkpoint must load into (tests/test_dropin.py)
        d["gd_shape/" + k] = np.asarray(v.shape, dtype=np.int64)
    for i, tt in enumerate(FULL_T):
        t = torch.tensor([tt])
        noise = inp["noises"][i]
        orig = diffusion.noise_like
        diffusion.noise_like = lambda shape, device, repeat=False: noise
        try:
            with torch.no_grad():
                d["dn_out/%d" % tt] = dn(inp["x"], t, inp["cond"]).numpy()
                d["p_sample/%d" % tt] = gd.p_sample(inp["x"], t, inp["cond"]).numpy()
        finally:
            diffusion.noise_like = orig
        for k in O.SCHEDULE_KEYS:
            d["sched/" + k] = getattr(gd, k).numpy()

    models = rh.import_nsf_models()
    from modules.nsf_hifigan.env import AttrDict
    gen = models.Generator(AttrDict(O.NSF_H_44K)).eval()
    gen.remove_weight_norm()
    gen.load_state_dict(O.synth_nsf_weights(O.NSF_H_44K))
    for k, v in gen.state_dict().items():
        d["nsf_shape/" + k] = np.asarray(v.shape, dtype=np.int64)
    L = inp["voc_mel"].shape[-1] * 512
    draws = iter([inp["rand_ini"], inp["sine_noise"], torch.zeros(1, L, 1)])   # models.py:192, :271, :322
    o_rand, o_randn_like = torch.rand, torch.randn_like
    torch.rand = lambda *a, **k: next(draws).clone()
    torch.randn_like = lambda *a, **k: next(draws).clone()
    try:
        with torch.no_grad():
            d["nsf/wav"] = gen(inp["voc_mel"], inp["voc_f0"]).numpy()
    finally:
        torch.rand, torch.randn_like = o_rand, o_randn_like

    import modules.fastspeech.pe as pe_mod
    m = pe_mod.PitchExtractor(n_mel_bins=80, conv_layers=2).eval()
    shapes = {k: v.shape for k, v in m.state_dict().items()}
    m.load_state_dict(full_pe_weights(shapes), strict=True)
    for k, s in shapes.items():
        d["pe_shape/" + k] = np.asarray(s, dtype=np.int64)
    with torch.no_grad():
        ret = m(inp["pe_mel"])
    d["pe/pitch_pred"] = ret["pitch_pred"].numpy()
    d["pe/f0_denorm_pred"] = ret["f0_denorm_pred"].numpy()

    import modules.nsf_hifigan.nvSTFT as nv
    nv.librosa_mel_fn = lambda sr, n_fft, n_mels, fmin, fmax: O.slaney_mel_basis(sr, n_fft, n_mels, fmin, fmax)
    stft_now = torch.stft
    nv.torch.stft = lambda *a, **k: stft_now(*a, **k) if "return_complex" in k else torch.view_as_real(stft_now(*a, return_complex=True, **k))
    try:
        stft = nv.STFT(hp["audio_sample_rate"], hp["audio_num_mel_bins"], hp["fft_size"], hp["win_size"], hp["hop_size"],
                       hp["fmin"], hp["fmax"])
        with torch.no_grad():
            d["mel/out"] = stft.get_mel(inp["wav"]).numpy()
    finally:
        torch.stft = stft_now
    for k in ("audio_sample_rate", "audio_num_mel_bins", "fft_size", "win_size", "hop_size", "fmin", "fmax"):
        d["hp/" + k] = np.int64(hp[k])
    d["hp/spec_min"] = np.asarray(hp["spec_min"], dtype=np.float32)
    d["hp/spec_max"] = np.asarray(hp["spec_max"], dtype=np.float32)
    np.savez_compressed(os.path.join(HERE, "full_44k.npz"), **d)
    print("full_44k", {k: v.shape for k, v in d.items() if "shape/" not in k})


def main():
    if "--only-full" in sys.argv:
        gen_full(rh.install())
        return
    hp = rh.install(overrides=SMALL)
    if "--only-pe" in sys.argv:
        gen_pe()
        return
    if "--only-mel" in sys.argv:
        gen_mel()
        return
    gen_diffnet(hp)
    gen_sampler(hp, "ddpm_small", K_step=6, speedup=1, spec_min=[-5.0], spec_max=[0.0])
    per_bin_min = list(np.linspace(-6.0, -4.0, 16))
    per_bin_max = list(np.linspace(-0.5, 0.5, 16))
    gen_sampler(hp, "ddpm_perbin_small", K_step=5, speedup=1, spec_min=per_bin_min, spec_max=per_bin_max, seed=17)
    gen_sampler(hp, "plms_small", K_step=100, speedup=20, spec_min=[-5.0], spec_max=[0.0], seed=27)
    gen_sampler(hp, "gtmel_small", K_step=1000, speedup=1, spec_min=[-5.0], spec_max=[0.0],
                use_gt_mel=True, add_noise_step=5, seed=37)
    gen_nsf()
    gen_hifigan24k()
    gen_mel()
    gen_pe()


if __name__ == "__main__":
    main()

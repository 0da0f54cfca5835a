"""The 24 kHz DiffNet of training/config.yaml (80 mel bins, 256 residual channels) on the tensor-core path.

The tensor-core modes pad the mel axis inside the library to whole 64-wide tiles (Mp = 128 for 80 bins): zero weight
columns / rows and a zero bias past the model's M, pad columns of the operand plane cleared once, pad columns of the head
never stored.  Everything the caller sees -- outputs, injected noise, the library's Philox stream -- keeps the logical M.
Held to the gates of the 44.1 kHz model (tests/test_gpu_parity.py)."""
import pytest
import torch

import synthetic as S
from oracle import diffsvc_oracle as O

DEV = "cuda"
SPEC_MIN, SPEC_MAX = torch.tensor([[[-5.0]]]), torch.tensor([[[0.0]]])
ENV = ("DSVC_TC_BN", "DSVC_SPLITK", "DSVC_STEP", "DSVC_FUSED_LAYER", "DSVC_PACK", "DSVC_TC_PAIR", "DSVC_SKIP_DEFER")


def _hp24(**kw):
    from diffsvc_b200.hparams import hparams, DEFAULTS_44K
    hparams.clear()
    hparams.update(DEFAULTS_44K)
    hparams.update(S.HPARAMS_24K)
    hparams.update(kw)
    return hparams


def _model(math_mode=None, M=80, C=256, H=256, L=20, K_step=1000, seed=1234):
    import diffsvc_b200 as D
    _hp24(pndm_speedup=1, hidden_size=H, residual_layers=L, residual_channels=C, audio_num_mel_bins=M, keep_bins=M)
    sd = S.synth_diffnet_weights(M=M, C=C, H=H, L=L, seed=seed)
    dn = D.DiffNet(M, math_mode=math_mode)
    dn.load_state_dict(sd, strict=True)
    gd = D.GaussianDiffusion(None, M, dn, timesteps=1000, K_step=K_step, loss_type="l2", spec_min=[-5.0], spec_max=[0.0])
    return gd.to(DEV).eval(), sd


def _inputs(B, T, steps, M=80, H=256, seed=7):
    g = torch.Generator().manual_seed(seed)
    cond = torch.randn(B, H, T, generator=g) * 0.5
    x0 = torch.randn(B, 1, M, T, generator=g)
    noise = torch.randn(steps, B, 1, M, T, generator=g)
    return cond, x0, noise


def _sched():
    return O.make_schedule(O.linear_beta_schedule(1000, 0.02))


def _clear_env(monkeypatch):
    for k in ENV:
        monkeypatch.delenv(k, raising=False)


# ------------------------------------------------------------------------------- default math mode (no device needed)
def test_default_math_24k_is_tensor_core():
    import diffsvc_b200 as D
    _hp24()
    assert D.DiffNet(80).math_mode == "tc3f16"


def test_explicit_math_is_honoured():
    import diffsvc_b200 as D
    _hp24(dsvc_math="fp32")
    assert D.DiffNet(80).math_mode == "fp32"
    _hp24()
    assert D.DiffNet(80, math_mode="fp32").math_mode == "fp32"
    assert D.DiffNet(80, math_mode="tc1f16").math_mode == "tc1f16"


def test_default_math_other_widths():
    import diffsvc_b200 as D
    from diffsvc_b200.hparams import hparams, DEFAULTS_44K
    hparams.clear(); hparams.update(DEFAULTS_44K)
    assert D.DiffNet(128).math_mode == "tc3f16"           # the 44.1 kHz model: unchanged
    assert D.DiffNet(78).math_mode == "fp32"              # not a multiple of 4: the library refuses tensor cores
    hparams["residual_channels"] = 192
    assert D.DiffNet(128).math_mode == "fp32"             # residual_channels % 128 != 0


# ------------------------------------------------------------------------------- against the CPU oracle
@pytest.mark.gpu
@pytest.mark.parametrize("math_mode,tol", [("fp32", 2e-5), ("tc3f16", 1e-4)])
def test_eval_vs_oracle(math_mode, tol, monkeypatch):
    _clear_env(monkeypatch)
    gd, sd = _model(math_mode)
    cond, x0, _ = _inputs(2, 200, 1)
    for t in (999, 37, 0):
        ref = O.diffnet_forward(sd, x0, torch.tensor([t, t]), cond)
        out = gd.denoise_fn(x0.to(DEV), torch.tensor([t, t], device=DEV), cond.to(DEV)).cpu()
        assert out.shape == ref.shape
        err = (out - ref).abs().max().item()
        assert err <= tol, (math_mode, t, err)


@pytest.mark.gpu
@pytest.mark.parametrize("math_mode", ["fp32", "tc3f16"])
def test_ddpm_chain_vs_oracle(math_mode, monkeypatch):
    _clear_env(monkeypatch)
    steps, T = 60, 136
    gd, sd = _model(math_mode)
    cond, x0, noise = _inputs(1, T, steps)
    ref = O.mel_from_x(O.sample(sd, _sched(), cond, x0, steps, noise), SPEC_MIN, SPEC_MAX)
    xf = gd.sample(x0.to(DEV), cond.to(DEV), steps, None, noise.to(DEV))
    mel = gd.denorm_spec(xf[:, 0].transpose(1, 2)).cpu()
    err = (mel - ref).abs().max().item()
    assert err <= 1e-3, (math_mode, err)
    assert err <= (1e-4 if math_mode == "fp32" else 3e-4), (math_mode, err)


@pytest.mark.gpu
@pytest.mark.parametrize("math_mode", ["fp32", "tc3f16"])
def test_plms_chain_vs_oracle(math_mode, monkeypatch):
    _clear_env(monkeypatch)
    gd, sd = _model(math_mode)
    cond, x0, _ = _inputs(1, 100, 1, seed=9)
    ref = O.sample(sd, _sched(), cond, x0, 1000, None, pndm_speedup=100)
    xf = gd.sample(x0.to(DEV), cond.to(DEV), 1000, 100).cpu()
    rng = max(1.0, ref.abs().max().item())
    err = (xf - ref).abs().max().item() / rng
    assert err <= 1e-5, (math_mode, err, rng)


@pytest.mark.gpu
def test_library_noise_stream_same_in_both_modes(monkeypatch):
    """The Philox counter of the library's own noise uses the logical M, not the padded width: one seed draws the same
    noise in fp32 and tc3f16 modes, so the two chains differ by rounding only.  Another seed moves the result by O(1)."""
    _clear_env(monkeypatch)
    cond, x0, _ = _inputs(1, 200, 1, seed=17)
    mels = {}
    for mode, seed in (("fp32", 2024), ("tc3f16", 2024), ("tc3f16", 2025)):
        gd, _ = _model(mode)
        xf = gd.sample(x0.to(DEV), cond.to(DEV), 100, None, None, seed=seed)
        mels[(mode, seed)] = gd.denorm_spec(xf[:, 0].transpose(1, 2)).cpu()
    same = (mels[("fp32", 2024)] - mels[("tc3f16", 2024)]).abs().max().item()
    other = (mels[("tc3f16", 2025)] - mels[("tc3f16", 2024)]).abs().max().item()
    assert same <= 1e-3, same
    assert other > 1e-1, other


@pytest.mark.gpu
@pytest.mark.parametrize("math_mode,pack", [("fp32", "1"), ("tc3f16", "1"), ("tc3f16", "0")])
def test_ragged_batch_is_per_item(math_mode, pack, monkeypatch):
    _clear_env(monkeypatch)
    monkeypatch.setenv("DSVC_PACK", pack)
    steps, lens = 12, [150, 97, 33]
    gd, sd = _model(math_mode)
    cond, x0, noise = _inputs(len(lens), max(lens), steps, seed=21)
    xf = gd.sample(x0.to(DEV), cond.to(DEV), steps, None, noise.to(DEV), lengths=lens).cpu()
    for b, n in enumerate(lens):
        ref = O.sample(sd, _sched(), cond[b:b + 1, :, :n], x0[b:b + 1, :, :, :n], steps, noise[:, b:b + 1, :, :, :n])
        err = (xf[b:b + 1, :, :, :n] - ref).abs().max().item()
        assert err <= 2e-4, (math_mode, pack, b, err)


# ------------------------------------------------------------------------------- schedule variants at C = 256
def _kernels(fn):
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events()]


@pytest.mark.gpu
def test_skip_defer_bit_identical(monkeypatch):
    """cfg1's 938 frames: 8 frame CTAs x (8 conv + 4 residual) channel tiles fit the SMs -> the deferred skip.  The
    layer-by-layer schedule (DSVC_SKIP_DEFER=0) gives the same bits."""
    cond, x0, _ = _inputs(1, 938, 1, seed=5)
    t = torch.full((1,), 417, dtype=torch.long, device=DEV)
    outs, evals = {}, {}
    for defer in (False, True):
        _clear_env(monkeypatch)
        if not defer:
            monkeypatch.setenv("DSVC_SKIP_DEFER", "0")
        gd, _ = _model("tc3f16")
        gd.denoise_fn(x0.to(DEV), t, cond.to(DEV))                     # prepare + warm-up
        names = _kernels(lambda: evals.__setitem__(defer, gd.denoise_fn(x0.to(DEV), t, cond.to(DEV)).cpu()))
        assert any("tc_pair2_kernel" in n for n in names) == defer, defer
        outs[defer] = gd.sample(x0.to(DEV), cond.to(DEV), 30, None, None, seed=11).cpu()
    assert torch.isfinite(outs[True]).all()
    assert torch.equal(evals[False], evals[True])
    assert torch.equal(outs[False], outs[True])


@pytest.mark.gpu
def test_step_kernel_request_falls_back(monkeypatch):
    """DSVC_STEP=1 asks for the one-launch step kernel; it needs M % 64 == 0, so an 80-bin model keeps the per-layer
    kernels and the same bits."""
    cond, x0, _ = _inputs(1, 200, 1, seed=6)
    outs = {}
    for step in (False, True):
        _clear_env(monkeypatch)
        if step:
            monkeypatch.setenv("DSVC_STEP", "1")
        gd, _ = _model("tc3f16")
        outs[step] = gd.sample(x0.to(DEV), cond.to(DEV), 20, None, None, seed=3).cpu()
        t = torch.full((1,), 9, dtype=torch.long, device=DEV)
        assert not any("tc_step_kernel" in n for n in _kernels(lambda: gd.denoise_fn(x0.to(DEV), t, cond.to(DEV))))
    assert torch.equal(outs[False], outs[True])


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"DSVC_TC_PAIR": "0"}, {"DSVC_TC_BN": "128"}])
def test_tile_variants_vs_oracle(env, monkeypatch):
    _clear_env(monkeypatch)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    steps, T = 3, 300
    gd, sd = _model("tc3f16")
    cond, x0, noise = _inputs(1, T, steps, seed=31)
    ref = O.sample(sd, _sched(), cond, x0, steps, noise)
    xf = gd.sample(x0.to(DEV), cond.to(DEV), steps, None, noise.to(DEV)).cpu()
    assert (xf - ref).abs().max().item() <= 5e-5


# ------------------------------------------------------------------------------- a second odd width
@pytest.mark.gpu
@pytest.mark.parametrize("math_mode", ["fp32", "tc3f16"])
def test_36_bins_vs_oracle(math_mode, monkeypatch):
    """M = 36: one K block of the input projection and one 64-wide head tile, both mostly padding."""
    _clear_env(monkeypatch)
    kw = dict(M=36, C=128, H=64, L=4)
    gd, sd = _model(math_mode, **kw)
    assert gd.denoise_fn.math_mode == math_mode
    cond, x0, noise = _inputs(2, 150, 20, M=36, H=64, seed=8)
    for t in (999, 5):
        ref = O.diffnet_forward(sd, x0, torch.tensor([t, t]), cond)
        out = gd.denoise_fn(x0.to(DEV), torch.tensor([t, t], device=DEV), cond.to(DEV)).cpu()
        assert (out - ref).abs().max().item() <= 1e-4, (math_mode, t)
    ref = O.sample(sd, _sched(), cond, x0, 20, noise)
    xf = gd.sample(x0.to(DEV), cond.to(DEV), 20, None, noise.to(DEV)).cpu()
    assert (xf - ref).abs().max().item() <= 3e-4
    ref = O.sample(sd, _sched(), cond[:1], x0[:1], 1000, None, pndm_speedup=100)
    xf = gd.sample(x0[:1].to(DEV), cond[:1].to(DEV), 1000, 100).cpu()
    assert (xf - ref).abs().max().item() / max(1.0, ref.abs().max().item()) <= 1e-5


# ------------------------------------------------------------------------------- cfg1 end to end
@pytest.mark.gpu
def test_cfg1_end_to_end(monkeypatch):
    """BASELINE cfg1: 5 s at 24 kHz (938 frames), 100 DDPM steps through GaussianDiffusion.forward with the default math,
    then the 24 kHz HiFi-GAN with its pitch source.  Against the oracle chain on the same inputs and noise."""
    from diffsvc_b200.vocoders.hifigan import HifiGAN
    _clear_env(monkeypatch)
    T, K, Th = 938, 100, 400
    gd, sd = _model(None, K_step=K)
    assert gd.denoise_fn.math_mode == "tc3f16"
    g = torch.Generator().manual_seed(29)
    pe_w = torch.randn(300, 256, generator=g) * 256 ** -0.5
    pe_w[0] = 0
    with torch.no_grad():
        gd.fs2.pitch_embed.weight.copy_(pe_w)
    hubert = torch.randn(1, Th, 256, generator=g) * 0.5
    mel2ph = (torch.arange(T) * Th // T + 1)[None].long()
    f0 = torch.log2(S.synth_f0(1, T).clamp(min=80.0))
    x0 = torch.randn(1, 1, 80, T, generator=g)
    noise = torch.randn(K, 1, 1, 80, T, generator=g)
    ret = gd(hubert.to(DEV), mel2ph.to(DEV), None, None, f0.clone().to(DEV), None, None, infer=True,
             x_init=x0, noise=noise.to(DEV))
    mel = ret["mel_out"].cpu()

    dec, f0d = O.cond_encoder(pe_w, hubert, mel2ph, f0.clone(), 256, 1100.0, 50.0)
    ref_mel = O.mel_from_x(O.sample(sd, _sched(), dec.transpose(1, 2), x0, K, noise), SPEC_MIN, SPEC_MAX, mel2ph)
    err = (mel - ref_mel).abs().max().item()
    assert err <= 1e-3, err

    h = dict(S.HIFIGAN_H_24K)
    vsd = S.synth_nsf_weights(h, seed=4242)
    voc = HifiGAN.from_state_dict(h, vsd, device=DEV)
    rand_ini = torch.rand(1, 9, generator=g)
    sn = torch.randn(1, T * 128, 9, generator=g)
    wav = voc.spec2wav(mel[0].numpy(), f0=ret["f0_denorm"][0].cpu().numpy(), rand_ini=rand_ini, sine_noise=sn)
    ref = O.nsf_generator(vsd, h, ref_mel.transpose(1, 2), f0d, rand_ini, sn).reshape(-1)
    assert wav.shape == (T * 128,) and float(ref.std()) > 1e-2
    d = torch.from_numpy(wav) - ref
    rms = d.pow(2).mean().sqrt().item()
    assert rms <= 1e-4, (rms, d.abs().max().item())

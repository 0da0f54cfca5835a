"""ResBlock2 ("resblock": "2", the HiFi-GAN "V3" block) vocoder generators: modules/nsf_hifigan/models.py:73-94
(chosen at :337) and modules/hifigan/hifigan.py:70-91 (chosen at :119).

CPU: a restatement of the reference's ResBlock2 generator against the fixtures its own modules wrote
(tests/golden/make_golden_resblock2.py), the loader's key set against the reference's parameter names, and
the C-ABI entry point's refusal without a device.  GPU: the native generator against those fixtures and against the
restatement at the full 44.1 kHz size in all three arithmetic modes (tcgen05 with the 256-row narrow window, FFMA for
the narrow stages, FFMA everywhere)."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import synthetic as S
from oracle import diffsvc_oracle as O
from diffsvc_b200.vocoders import nsf_models as NM

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DEV = "cuda"


# ------------------------------------------------------------------------------- CPU restatement of the reference
def resblock2(sd, prefix, x, kernel_size, dilations):
    """ResBlock2.forward, models.py:86-91: two convs, dilation[0] and dilation[1]; further entries are ignored."""
    for m, d in enumerate(dilations[:2]):
        xt = F.leaky_relu(x, O.LRELU_SLOPE)
        xt = F.conv1d(xt, sd[prefix + "convs.%d.weight" % m], sd[prefix + "convs.%d.bias" % m],
                      dilation=d, padding=O.get_padding(kernel_size, d))
        x = xt + x
    return x


def generator(sd, h, mel, f0, rand_ini, noise):
    """Generator.forward (models.py:361-387) / HifiGanGenerator.forward (hifigan.py:144-169) with the block type
    chosen as at models.py:337: the oracle's nsf_generator with resblock2 in place of resblock1."""
    if str(h.get("resblock", "1")) == "1":
        return O.nsf_generator(sd, h, mel, f0, rand_ini, noise)
    rates, ksizes = list(h["upsample_rates"]), list(h["upsample_kernel_sizes"])
    rks, rds = list(h["resblock_kernel_sizes"]), list(h["resblock_dilation_sizes"])
    hop = int(np.prod(rates))
    har = None
    if f0 is not None:
        f0_up = torch.repeat_interleave(f0[:, None], hop, dim=2).transpose(1, 2)
        har = O.source_module(sd, f0_up, h["sampling_rate"], 8, rand_ini, noise).transpose(1, 2)
    x = F.conv1d(mel, sd["conv_pre.weight"], sd["conv_pre.bias"], padding=3)
    nk = len(rks)
    for i, (u, k) in enumerate(zip(rates, ksizes)):
        x = F.leaky_relu(x, O.LRELU_SLOPE)
        x = F.conv_transpose1d(x, sd["ups.%d.weight" % i], sd["ups.%d.bias" % i], stride=u, padding=(k - u) // 2)
        if har is not None:
            if i + 1 < len(rates):
                s = int(np.prod(rates[i + 1:]))
                x = x + F.conv1d(har, sd["noise_convs.%d.weight" % i], sd["noise_convs.%d.bias" % i], stride=s, padding=s // 2)
            else:
                x = x + F.conv1d(har, sd["noise_convs.%d.weight" % i], sd["noise_convs.%d.bias" % i])
        xs = None
        for j in range(nk):
            r = resblock2(sd, "resblocks.%d." % (i * nk + j), x, rks[j], rds[j])
            xs = r if xs is None else xs + r
        x = xs / nk
    x = F.leaky_relu(x)
    x = F.conv1d(x, sd["conv_post.weight"], sd["conv_post.bias"], padding=3)
    return torch.tanh(x)


def _gold(name):
    z = np.load(os.path.join(GOLD, name + ".npz"))
    h = {k[2:]: z[k].tolist() for k in z.files if k.startswith("h/")}
    if "dil/0" in z.files:          # ragged dilation lists
        h["resblock_dilation_sizes"] = [z["dil/%d" % j].tolist() for j in range(len(h["resblock_kernel_sizes"]))]
    h["resblock"] = "2"
    h.setdefault("sampling_rate", h.get("audio_sample_rate"))
    ckpt = {k[5:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("ckpt/")}
    return z, h, ckpt


# ------------------------------------------------------------------------------- CPU
def test_oracle_matches_nsf_resblock2_golden():
    z, h, ckpt = _gold("nsf_resblock2_small")
    assert len(h["resblock_dilation_sizes"][1]) == 3            # pins "the first two dilations only"
    folded_ref = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd/")}
    folded = O.fold_weight_norm(ckpt)
    assert set(folded) == set(folded_ref)
    for k in folded:
        assert (folded[k] - folded_ref[k]).abs().max().item() <= 1e-6, k
    wav = generator(folded, h, torch.from_numpy(z["mel"]), torch.from_numpy(z["f0"]),
                    torch.from_numpy(z["rand_ini"]), torch.from_numpy(z["sine_noise"]))
    ref = torch.from_numpy(z["wav"])
    assert wav.shape == ref.shape and float(ref.std()) > 1e-2
    assert (wav - ref).abs().max().item() <= 2e-6


def test_oracle_matches_hifigan24k_resblock2_golden():
    z, h, ckpt = _gold("hifigan24k_resblock2_small")
    sd = O.fold_weight_norm(ckpt)
    mel, f0 = torch.from_numpy(z["mel"]), torch.from_numpy(z["f0"])
    wav = generator(sd, h, mel, f0, torch.from_numpy(z["rand_ini"]), torch.from_numpy(z["sine_noise"]))
    assert (wav - torch.from_numpy(z["wav_f0"])).abs().max().item() <= 2e-6
    plain = generator(sd, h, mel, None, None, None)
    assert (plain - torch.from_numpy(z["wav_plain"])).abs().max().item() <= 2e-6
    sd2 = O.fold_weight_norm({k[11:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("nosrc_ckpt/")})
    nosrc = generator(sd2, h, mel, None, None, None)
    assert (nosrc - torch.from_numpy(z["wav_nosrc"])).abs().max().item() <= 2e-6


def test_loader_reads_exactly_the_reference_parameter_names():
    """The keys of a reference Generator(h) / HifiGanGenerator(h) with resblock "2" (weight-norm folded) are the keys
    the native loader consumes -- with the source and, for the 24 kHz model, without it."""
    z, h, ckpt = _gold("nsf_resblock2_small")
    assert set(NM.state_dict_keys(h, True)) == set(O.fold_weight_norm(ckpt))
    z, h, ckpt = _gold("hifigan24k_resblock2_small")
    assert set(NM.state_dict_keys(h, True)) == set(O.fold_weight_norm(ckpt))
    nosrc = {k[11:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("nosrc_ckpt/")}
    assert set(NM.state_dict_keys(h, False)) == set(O.fold_weight_norm(nosrc))
    # the synthetic full-size weights use the same names
    assert set(NM.state_dict_keys(S.NSF_H_44K_V3, True)) == set(S.synth_nsf_resblock2_weights(S.NSF_H_44K_V3))


def test_block_type_rule():
    """models.py:337: ResBlock1 only for the string '1'; an integer 1 and a missing key keep meaning ResBlock1."""
    assert NM.resblock_type({"resblock": "1"}) == 1 and NM.resblock_type({"resblock": 1}) == 1
    assert NM.resblock_type({}) == 1
    assert NM.resblock_type({"resblock": "2"}) == 2 and NM.resblock_type({"resblock": 2}) == 2
    assert NM.resblock_dilations(dict(resblock="2", resblock_dilation_sizes=[[1, 3, 5], [2, 6]])) == [[1, 3], [2, 6]]
    assert NM.resblock_dilations(dict(resblock="1", resblock_dilation_sizes=[[1, 3, 5]])) == [[1, 3, 5]]


def test_mismatched_checkpoint_names_the_missing_key():
    """A ResBlock1 checkpoint under a resblock "2" config fails like load_state_dict(strict=True), before any device
    work."""
    z = np.load(os.path.join(GOLD, "nsf_small.npz"))
    ckpt = {k[5:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("ckpt/")}
    h = {k[2:]: z[k].tolist() for k in z.files if k.startswith("h/")}
    h["resblock"] = "2"
    with pytest.raises(KeyError, match=r"resblocks\.0\.convs\.0\.weight"):
        NM.Generator(h, ckpt, device="cpu")


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only behaviour")
def test_create_ex_refuses_without_device():
    from diffsvc_b200 import _lib
    lib = _lib.load()
    h = C.c_void_p()
    cfg, w = _lib.NsfConfig(), _lib.NsfWeights()
    cfg.num_upsamples, cfg.num_kernels, cfg.num_dilations, cfg.harmonic_num = 1, 1, 2, 8
    assert lib.dsvc_nsf_create_ex(C.byref(h), C.byref(cfg), 2, C.byref(w), None) == -3
    assert b"no CPU fallback" in lib.dsvc_last_error()


# ------------------------------------------------------------------------------- GPU
def _hp(**kw):
    from diffsvc_b200.hparams import hparams, DEFAULTS_44K
    hparams.clear()
    hparams.update(DEFAULTS_44K)
    hparams.update(kw)
    return hparams


def _stats(a, b):
    d = a - b
    return d.pow(2).mean().sqrt().item(), d.abs().max().item()


@pytest.mark.gpu
def test_nsf_golden_through_weight_norm_checkpoint():
    z, h, ckpt = _gold("nsf_resblock2_small")
    gen = NM.Generator(h, ckpt, device=DEV)           # weight_g / weight_v form: folds the weight norm itself
    wav = gen(torch.from_numpy(z["mel"]).to(DEV), torch.from_numpy(z["f0"]).to(DEV),
              rand_ini=torch.from_numpy(z["rand_ini"]), sine_noise=torch.from_numpy(z["sine_noise"])).cpu()
    ref = torch.from_numpy(z["wav"])
    assert wav.shape == ref.shape
    rms, mx = _stats(wav, ref)
    print("nsf_resblock2_small: rms %.2e max %.2e" % (rms, mx))
    assert rms <= 1e-4 and mx <= 5e-4


@pytest.mark.gpu
def test_hifigan24k_golden_with_and_without_f0():
    from diffsvc_b200.vocoders.hifigan import HifiGAN
    z, h, ckpt = _gold("hifigan24k_resblock2_small")
    h = dict(h, use_pitch_embed=True)
    _hp(use_nsf=True)
    voc = HifiGAN.from_state_dict(h, ckpt, device=DEV)
    nosrc = {k[11:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("nosrc_ckpt/")}
    voc2 = HifiGAN.from_state_dict(dict(h, use_pitch_embed=False), nosrc, device=DEV)
    assert not voc2.model.has_source
    mel, f0 = z["mel"], z["f0"]
    for b in range(mel.shape[0]):
        w = voc.spec2wav(mel[b].T, f0=f0[b], rand_ini=torch.from_numpy(z["rand_ini"][b:b + 1]),
                         sine_noise=torch.from_numpy(z["sine_noise"][b:b + 1]))
        w2 = voc.spec2wav(mel[b].T)                                        # no f0: the source is skipped
        w3 = voc2.spec2wav(mel[b].T)                                       # a model without source weights
        for out, key in ((w, "wav_f0"), (w2, "wav_plain"), (w3, "wav_nosrc")):
            rms, mx = _stats(torch.from_numpy(out), torch.from_numpy(z[key][b, 0]))
            assert rms <= 1e-4 and mx <= 2e-5, (key, b, rms, mx)


def _v3_inputs(B, T, seed):
    g = torch.Generator().manual_seed(seed)
    mel = torch.randn(B, T, 128, generator=g) * 0.8 - 2.0            # log10 mel
    f0 = S.synth_f0(B, T)
    rand_ini = torch.rand(B, 9, generator=g)
    noise = torch.randn(B, T * 512, 9, generator=g)
    return mel, f0, rand_ini, noise


@pytest.mark.gpu
@pytest.mark.parametrize("B,T", [(2, 41), (1, 862)])
def test_v3_generator_all_modes_vs_oracle(B, T, monkeypatch):
    """The V3-style 44.1 kHz generator: its dilation-12 kernel-7 convs reach 36 rows, so the 32- and 16-channel stages
    run on the 256-row narrow window by default.  DSVC_NSF_NARROW=0 puts those stages on the FFMA GEMM,
    DSVC_NSF_MATH=fp32 the whole generator."""
    from diffsvc_b200.vocoders.nsf_hifigan import NsfHifiGAN
    h = S.NSF_H_44K_V3
    assert max((k // 2) * d[1] for k, d in zip(h["resblock_kernel_sizes"], h["resblock_dilation_sizes"])) > 32
    _hp()
    sd = S.synth_nsf_resblock2_weights(h, seed=91)
    mel, f0, rand_ini, noise = _v3_inputs(B, T, seed=B * 1000 + T)
    ref = generator(sd, h, 2.30259 * mel.transpose(2, 1), f0, rand_ini, noise).reshape(-1)
    assert float(ref.std()) > 1e-2
    out = {}
    for mode, env in (("default", {}), ("narrow0", {"DSVC_NSF_NARROW": "0"}), ("fp32", {"DSVC_NSF_MATH": "fp32"})):
        for k in ("DSVC_NSF_NARROW", "DSVC_NSF_MATH"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        voc = NsfHifiGAN.from_state_dict(dict(h), sd, device=DEV)
        out[mode] = voc.spec2wav_torch(mel.to(DEV), f0=f0.to(DEV), rand_ini=rand_ini, sine_noise=noise).cpu()
        voc.model.release()
        rms, mx = _stats(out[mode], ref)
        print("v3 %s B=%d T=%d: rms %.2e max %.2e" % (mode, B, T, rms, mx))
        assert rms <= 1e-4 and mx <= 5e-4, (mode, rms, mx)
    assert not torch.equal(out["default"], out["narrow0"])     # the narrow stages ran on the tensor-core kernel


@pytest.mark.gpu
def test_v3_batch_equals_items_alone():
    from diffsvc_b200.vocoders.nsf_hifigan import NsfHifiGAN
    h = S.NSF_H_44K_V3
    _hp()
    sd = S.synth_nsf_resblock2_weights(h, seed=92)
    voc = NsfHifiGAN.from_state_dict(dict(h), sd, device=DEV)
    mel, f0, rand_ini, noise = _v3_inputs(2, 37, seed=5)
    both = voc.model.forward_mel(mel.to(DEV), f0.to(DEV), 2.30259, rand_ini=rand_ini, sine_noise=noise).cpu()
    for b in range(2):
        one = voc.model.forward_mel(mel[b:b + 1].to(DEV), f0[b:b + 1].to(DEV), 2.30259, rand_ini=rand_ini[b:b + 1],
                                    sine_noise=noise[b:b + 1]).cpu()
        d = (both[b:b + 1] - one).abs().max().item()
        print("v3 batch item %d: max %.2e" % (b, d))
        assert d <= 2e-6


@pytest.mark.gpu
def test_load_model_from_files_then_spec2wav(tmp_path):
    """NsfHifiGAN() the reference's way: hparams['vocoder_ckpt'] + sibling config.json with "resblock": "2" +
    ['generator'] in weight_g / weight_v form (modules/nsf_hifigan/models.py:14-30)."""
    from diffsvc_b200.vocoders.nsf_hifigan import NsfHifiGAN
    z, h, ckpt = _gold("nsf_resblock2_small")
    h.update(n_fft=512, win_size=512, hop_size=16, fmin=40, fmax=8000)
    (tmp_path / "config.json").write_text(json.dumps(h))
    torch.save({"generator": ckpt}, tmp_path / "model")
    _hp(vocoder_ckpt=str(tmp_path / "model"), audio_sample_rate=16000, audio_num_mel_bins=8, hop_size=16, fft_size=512,
        win_size=512, fmin=40, fmax=8000)
    voc = NsfHifiGAN()
    assert voc.h.resblock == "2" and voc.model.hop == 16
    mel = torch.from_numpy(z["mel"]).transpose(1, 2) / 2.30259           # back to "log10" mel [B, T, M]
    for b in range(mel.shape[0]):
        w = voc.spec2wav(mel[b].numpy(), f0=z["f0"][b], rand_ini=torch.from_numpy(z["rand_ini"][b:b + 1]),
                         sine_noise=torch.from_numpy(z["sine_noise"][b:b + 1]))
        rms, mx = _stats(torch.from_numpy(w), torch.from_numpy(z["wav"][b, 0]))
        assert rms <= 1e-4 and mx <= 5e-4, (b, rms, mx)

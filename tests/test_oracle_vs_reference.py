"""The oracle against the reference's own modules at the FULL 44.1 kHz config (config_nsf.yaml): DiffNet, DDPM
steps, NSF-HiFiGAN generator, PitchExtractor and mel analysis.  The reference's outputs, its schedule buffers and
the key -> shape tables of its state dicts were dumped once from the unmodified reference
(`tests/golden/make_golden.py --only-full`) into tests/golden/full_44k.npz; weights and inputs are rebuilt here
from their seeds."""
import os

import numpy as np
import pytest
import torch

from make_golden import FULL_T, full_inputs, full_pe_weights
from oracle import diffsvc_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "full_44k.npz")


@pytest.fixture(scope="module")
def z():
    return np.load(GOLDEN)


@pytest.fixture(scope="module")
def hp(z):
    return {k[3:]: z[k] for k in z.files if k.startswith("hp/")}


def _shapes(z, prefix):
    return {k[len(prefix):]: tuple(int(s) for s in z[k]) for k in z.files if k.startswith(prefix)}


def test_full_diffnet_and_ddpm_steps(z):
    sd = O.synth_diffnet_weights()
    inp = full_inputs()
    x, cond = inp["x"], inp["cond"]
    sched = {k: torch.from_numpy(z["sched/" + k]) for k in O.SCHEDULE_KEYS}
    for i, tt in enumerate(FULL_T):
        t = torch.tensor([tt])
        ref = torch.from_numpy(z["dn_out/%d" % tt])
        assert float(ref.abs().max()) > 1e-3                # not vacuous
        assert (O.diffnet_forward(sd, x, t, cond) - ref).abs().max().item() <= 5e-6
        ref_x = torch.from_numpy(z["p_sample/%d" % tt])
        assert (O.p_sample(sd, sched, x, t, cond, inp["noises"][i]) - ref_x).abs().max().item() <= 5e-6


def test_synth_weight_keys_match_reference(z):
    mine = O.synth_diffnet_weights()
    ref = _shapes(z, "dn_shape/")
    assert set(mine) == set(ref)
    for k in ref:
        assert tuple(mine[k].shape) == ref[k], k


def test_full_nsf_generator(z):
    mine = O.synth_nsf_weights(O.NSF_H_44K)
    ref_shapes = _shapes(z, "nsf_shape/")
    assert set(mine) == set(ref_shapes)
    assert all(tuple(mine[k].shape) == ref_shapes[k] for k in mine)
    inp = full_inputs()
    L = inp["voc_mel"].shape[-1] * 512
    ref = torch.from_numpy(z["nsf/wav"])
    wav = O.nsf_generator(mine, O.NSF_H_44K, inp["voc_mel"], inp["voc_f0"], inp["rand_ini"], inp["sine_noise"])
    assert wav.shape == ref.shape == (1, 1, L)
    assert float(ref.std()) > 1e-3                      # not vacuous
    assert (wav - ref).abs().max().item() <= 5e-6


def test_full_pitch_extractor(z):
    """PitchExtractor at the real size (hidden 256, 80 mel bins), eval mode, perturbed BatchNorm statistics."""
    sd = full_pe_weights(_shapes(z, "pe_shape/"))
    mel = full_inputs()["pe_mel"]
    pred, f0 = O.pitch_extractor(sd, mel)
    ref_pred, ref_f0 = torch.from_numpy(z["pe/pitch_pred"]), torch.from_numpy(z["pe/f0_denorm_pred"])
    assert float(ref_f0.max()) > 50.0                   # not vacuous
    assert (pred - ref_pred).abs().max().item() <= 1e-5
    assert (f0 - ref_f0).abs().max().item() <= 1e-3
    assert (f0[1, 100:] == 0).all()


def test_full_mel_analysis(z, hp):
    """STFT.get_mel at config_nsf.yaml's analysis parameters (2048 / 512 / 128 bins, 40-16000 Hz).  librosa is
    absent: the reference ran with librosa.filters.mel served by the oracle's restatement (see make_golden.py)."""
    wav = full_inputs()["wav"]
    ref = torch.from_numpy(z["mel/out"])
    sr, n_fft, n_mels, fmin, fmax = (int(hp[k]) for k in ("audio_sample_rate", "fft_size", "audio_num_mel_bins", "fmin", "fmax"))
    basis = O.slaney_mel_basis(sr, n_fft, n_mels, fmin, fmax)
    got = O.mel_analysis(wav, n_fft, int(hp["win_size"]), int(hp["hop_size"]), basis)
    assert got.shape == ref.shape == (1, 128, 30000 // 512)
    assert (got - ref).abs().max().item() <= 1e-5

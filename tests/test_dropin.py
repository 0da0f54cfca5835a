"""Drop-in wiring: with the meta-path finder installed, the host project's own `infer_tools.infer_tool` binds OUR
classes without any edit.

The host is the reference tree when DIFFSVC_REFERENCE_ROOT names a prophesier/diff-svc checkout, and otherwise a
stand-in written here: the reference's package layout and the names its infer_tool imports
(infer_tools/infer_tool.py:13-22), with placeholder classes behind every module the finder replaces.  The state
dicts our classes must load are checked against the reference's key -> shape tables in tests/golden/full_44k.npz
(tests/golden/make_golden.py --only-full)."""
import os
import subprocess
import sys
import textwrap

import ref_harness as rh

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

HOST_STANDIN = {
    "utils/__init__.py": "",
    "utils/hparams.py": "hparams = {}\n\n\ndef set_hparams(*a, **k):\n    return hparams\n",
    "network/__init__.py": "",
    "network/diff/__init__.py": "",
    "network/diff/net.py": "class DiffNet:\n    pass\n",
    "network/diff/diffusion.py": "class GaussianDiffusion:\n    pass\n",
    "network/vocoders/__init__.py": "from network.vocoders import nsf_hifigan\n",
    # the three names the drop-in and infer_tool use: a class registry, its decorator, and a lookup that falls back
    # to resolving a dotted "package.Class" path
    "network/vocoders/base_vocoder.py": textwrap.dedent("""
        import importlib
        VOCODERS = {}


        def register_vocoder(cls):
            VOCODERS.update({key: cls for key in (cls.__name__, cls.__name__.lower())})
            return cls


        def get_vocoder_cls(hparams):
            name = hparams["vocoder"]
            found = VOCODERS.get(name)
            if found is None:
                module, _, attr = name.rpartition(".")
                found = vars(importlib.import_module(module))[attr]
            return found
    """),
    "network/vocoders/nsf_hifigan.py": textwrap.dedent("""
        from network.vocoders.base_vocoder import register_vocoder


        @register_vocoder
        class NsfHifiGAN:
            pass
    """),
    "modules/__init__.py": "",
    "modules/fastspeech/__init__.py": "",
    "modules/fastspeech/fs2.py": textwrap.dedent("""
        import torch


        class FastSpeech2(torch.nn.Module):
            def __init__(self, dictionary=None, out_dims=None):
                super().__init__()
                self.pitch_embed = torch.nn.Embedding(300, 256, 0)
    """),
    "modules/fastspeech/pe.py": "class PitchExtractor:\n    pass\n",
    "modules/nsf_hifigan/__init__.py": "",
    "modules/nsf_hifigan/models.py": "def load_model(*a, **k):\n    raise NotImplementedError\n",
    "modules/nsf_hifigan/nvSTFT.py": "class STFT:\n    pass\n",
    "infer_tools/__init__.py": "",
    "infer_tools/infer_tool.py": textwrap.dedent("""
        from modules.fastspeech.pe import PitchExtractor
        from network.diff.diffusion import GaussianDiffusion
        from network.diff.net import DiffNet
        from network.vocoders.base_vocoder import VOCODERS, get_vocoder_cls
        from utils.hparams import hparams, set_hparams


        class Svc:
            def after_infer(self, prediction, singer, in_path):
                return prediction
    """),
}


def _host(tmp_path):
    """The host tree: the reference checkout if one is named, else the stand-in written under tmp_path."""
    if rh.reference_available():
        return rh.REFERENCE_ROOT
    root = tmp_path / "host"
    for rel, src in HOST_STANDIN.items():
        (root / rel).parent.mkdir(parents=True, exist_ok=True)
        (root / rel).write_text(src)
    return str(root)


def _run(tmp_path, body, token):
    """`body` in a fresh interpreter whose working directory is a scratch project and whose hparams are the
    config_nsf.yaml values (the reference's own loader on the reference tree)."""
    (tmp_path / "infer_tools").mkdir()
    (tmp_path / "infer_tools" / "f0_temp.json").write_text('{"info": "temp_dict"}')   # infer_tool.py:52 reads it relative to cwd
    host = _host(tmp_path)
    code = textwrap.dedent("""
        import sys
        import numpy as np
        sys.path.insert(0, %r); sys.path.insert(0, %r); sys.path.insert(0, %r)
        HOST = %r
        Z = np.load(%r)
        import ref_harness as rh
        if rh.reference_available():
            rh.install()                           # stubs for librosa etc. + set_hparams(config_nsf.yaml)
        else:
            from utils.hparams import hparams
            from diffsvc_b200.hparams import DEFAULTS_44K
            hparams.update(DEFAULTS_44K)
            hparams.update(vocoder="network.vocoders.nsf_hifigan.NsfHifiGAN", spec_min=Z["hp/spec_min"].tolist(),
                           spec_max=Z["hp/spec_max"].tolist())

        def ref_shapes(prefix):
            return {k[len(prefix):]: tuple(int(s) for s in Z[k]) for k in Z.files if k.startswith(prefix)}
    """ % (ROOT, GOLDEN, host, host, os.path.join(GOLDEN, "full_44k.npz"))) + textwrap.dedent(body)
    r = subprocess.run([sys.executable, "-c", code], cwd=tmp_path, capture_output=True, text=True, timeout=300)
    assert token in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_infer_tool_binds_native_classes(tmp_path):
    _run(tmp_path, """
        import torch
        import diffsvc_b200.dropin as dropin
        dropin.install()
        import infer_tools.infer_tool as it        # the host's own, unmodified module
        import diffsvc_b200 as D
        from utils.hparams import hparams as ref_hparams
        assert it.GaussianDiffusion is D.GaussianDiffusion, it.GaussianDiffusion
        assert it.DiffNet is D.DiffNet
        assert D.hparams is ref_hparams            # one shared config dict (pndm_speedup side channel)
        from network.vocoders.base_vocoder import get_vocoder_cls, VOCODERS
        assert get_vocoder_cls(ref_hparams) is D.NsfHifiGAN, get_vocoder_cls(ref_hparams)
        assert VOCODERS["NsfHifiGAN"] is D.NsfHifiGAN
        import modules.nsf_hifigan.models as m
        assert m.load_model is D.vocoders.nsf_models.load_model
        import modules.fastspeech.fs2 as fs2
        dn = D.DiffNet(ref_hparams["audio_num_mel_bins"])
        gd = D.GaussianDiffusion(None, 128, dn, timesteps=ref_hparams["timesteps"], K_step=ref_hparams["K_step"],
                                 loss_type=ref_hparams["diff_loss_type"], spec_min=ref_hparams["spec_min"], spec_max=ref_hparams["spec_max"])
        assert isinstance(gd.fs2, fs2.FastSpeech2)  # conditioning stays the host's own module
        dropin.uninstall()
        # strict load_ckpt compatibility with the reference's GaussianDiffusion (fs2.* is the host's module on both sides)
        a = gd.state_dict()
        ref = {k: s for k, s in ref_shapes("gd_shape/").items() if not k.startswith("fs2.")}
        mine = {k: tuple(v.shape) for k, v in a.items() if not k.startswith("fs2.")}
        assert set(mine) == set(ref), set(mine) ^ set(ref)
        assert all(mine[k] == ref[k] for k in ref), [k for k in ref if mine[k] != ref[k]]
        ckpt = {k: torch.zeros(s) for k, s in ref.items()}
        ckpt.update({k: v for k, v in a.items() if k.startswith("fs2.")})
        gd.load_state_dict(ckpt, strict=True)
        print("DROPIN_OK")
    """, "DROPIN_OK")


def test_after_infer_patch_and_nvstft_alias(tmp_path):
    """install(patch_after_infer=True): the host's own Svc gets the device-side after_infer the moment
    infer_tools.infer_tool is imported; modules.nsf_hifigan.nvSTFT resolves to the mel analysis kernel's host."""
    _run(tmp_path, """
        import diffsvc_b200.dropin as dropin
        dropin.install(patch_after_infer=True)
        import infer_tools.infer_tool as it
        from diffsvc_b200 import infer_glue
        assert it.Svc.after_infer is infer_glue.after_infer, it.Svc.after_infer
        assert it.Svc._dsvc_reference_after_infer.__module__ == "infer_tools.infer_tool"
        assert it.__file__.startswith(HOST), it.__file__      # still the host's own module
        import modules.nsf_hifigan.nvSTFT as nv
        import diffsvc_b200.vocoders.nvstft as ours
        assert nv is ours and nv.STFT is ours.STFT
        # late patching of an already imported module
        dropin.uninstall()
        sys.modules.pop("infer_tools.infer_tool")
        import infer_tools.infer_tool as it2
        assert it2.Svc.after_infer is not infer_glue.after_infer
        dropin.install(patch_after_infer=True)
        assert it2.Svc.after_infer is infer_glue.after_infer
        print("PATCH_OK")
    """, "PATCH_OK")


def test_pitch_extractor_alias_and_keys(tmp_path):
    """The host's infer_tool binds our PitchExtractor, whose state_dict has the reference module's keys and shapes."""
    _run(tmp_path, """
        import diffsvc_b200.dropin as dropin
        dropin.install()
        import infer_tools.infer_tool as it
        import diffsvc_b200 as D
        assert it.PitchExtractor is D.PitchExtractor
        ours = {k: tuple(v.shape) for k, v in D.PitchExtractor().state_dict().items()}
        dropin.uninstall()
        import modules.fastspeech.pe as ref_pe
        assert ref_pe.PitchExtractor is not D.PitchExtractor
        ref = ref_shapes("pe_shape/")
        assert set(ours) == set(ref), set(ours) ^ set(ref)
        assert all(ours[k] == ref[k] for k in ref)
        print("PE_OK")
    """, "PE_OK")

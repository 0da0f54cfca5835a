"""Import harness for the UNMODIFIED reference (prophesier/diff-svc) on CPU.

Test infrastructure only.  It exists in two places of the workflow:
  * `tests/golden/make_golden.py` dumps golden tensors from the reference's own
    modules once; the tests compare against those stored vectors;
  * `tests/svc_e2e.py golden` stores what the reference's own `Svc.infer` computes
    (tests/test_svc_infer_gpu.py compares against it);
  * `tests/test_dropin.py` binds into the live tree when one is named (a stand-in
    host tree otherwise).
The reference is found through DIFFSVC_REFERENCE_ROOT (a prophesier/diff-svc
checkout).

Nothing on the product path imports this file.

What it does (SURVEY.md section 8c):
  * stubs host-only third-party libs the reference imports at module import time
    (librosa, pycwt, matplotlib, soundfile, parselmouth, ...), none of which is on
    the sampler / vocoder path;
  * restores `scipy.signal.kaiser` (removed in SciPy >= 1.13, imported by
    modules/parallel_wavegan/layers/pqmf.py:12);
  * calls `set_hparams` BEFORE importing network.diff.diffusion, so that
    `linear_beta_schedule`'s default `max_beta` is the config's 0.02
    (network/diff/diffusion.py:40 freezes it at import time).
"""
import importlib
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("DIFFSVC_REFERENCE_ROOT", "")

_STUBS = [
    "librosa", "librosa.filters", "librosa.util", "librosa.core", "pycwt", "matplotlib", "matplotlib.pylab",
    "matplotlib.pyplot", "soundfile", "parselmouth", "torchcrepe", "resampy", "webrtcvad",
    "pyloudnorm", "skimage", "skimage.transform", "h5py", "pytorch_lightning", "fairseq",
]


def reference_available():
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, "network", "diff"))


class _Anything(types.ModuleType):
    """Module stub: any attribute access returns a dummy callable/module."""

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        sub = _Anything(self.__name__ + "." + name)
        setattr(self, name, sub)
        return sub

    def __call__(self, *a, **k):
        return None


def install(config="training/config_nsf.yaml", overrides=None):
    """Make `network.*`, `modules.*`, `utils.*` of the reference importable and
    populate the reference's global `hparams`.  Returns the hparams dict."""
    if not reference_available():
        raise RuntimeError("reference tree not found (DIFFSVC_REFERENCE_ROOT=%r)" % REFERENCE_ROOT)
    for name in _STUBS:
        if name not in sys.modules:
            try:
                importlib.import_module(name)
            except Exception:
                sys.modules[name] = _Anything(name)
    import scipy.signal
    if not hasattr(scipy.signal, "kaiser"):
        import scipy.signal.windows
        scipy.signal.kaiser = scipy.signal.windows.kaiser
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    from utils.hparams import set_hparams, hparams
    cwd = os.getcwd()
    os.chdir(REFERENCE_ROOT)  # config paths in the yaml chain are relative to the repo root
    try:
        set_hparams(config=config, exp_name="", infer=True, reset=True, print_hparams=False)
    finally:
        os.chdir(cwd)
    if overrides:
        hparams.update(overrides)
    return hparams


def import_diffusion():
    """Returns (diffusion module, net module) of the reference, imported AFTER set_hparams."""
    import network.diff.net as net
    import network.diff.diffusion as diffusion
    return diffusion, net


def import_nsf_models():
    import modules.nsf_hifigan.models as models
    return models

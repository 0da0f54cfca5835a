"""The deferred-skip schedule of the WaveNet layers (csrc/diffnet.cu, skip_defer_pick): layer l's skip half of the output
projection runs in layer l+1's conv kernel (tc_pair2_kernel), the out-projection between two convs keeps the residual
half.  Same tiles, functors and skip-sum order as the layer-by-layer schedule (DSVC_SKIP_DEFER=0): every result must be
bit-identical.  Shapes that do not take it (here a batch on 128-wide tiles) must keep the old schedule."""
import pytest
import torch

from oracle import diffsvc_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _model(monkeypatch, defer):
    """A model whose handle is prepared with the schedule switch set (it is read when the handle is prepared)."""
    import diffsvc_b200 as D
    from diffsvc_b200.hparams import hparams, DEFAULTS_44K
    hparams.clear(); hparams.update(DEFAULTS_44K); hparams["pndm_speedup"] = 1
    for k in ("DSVC_TC_BN", "DSVC_SPLITK", "DSVC_STEP", "DSVC_FUSED_LAYER", "DSVC_PACK", "DSVC_TC_PAIR"):
        monkeypatch.delenv(k, raising=False)
    if defer:
        monkeypatch.delenv("DSVC_SKIP_DEFER", raising=False)
    else:
        monkeypatch.setenv("DSVC_SKIP_DEFER", "0")
    dn = D.DiffNet(128, math_mode="tc3f16")
    dn.load_state_dict(O.synth_diffnet_weights(), strict=True)
    gd = D.GaussianDiffusion(None, 128, dn, timesteps=1000, K_step=1000, loss_type="l2", spec_min=[-5.0], spec_max=[0.0])
    return gd.to(DEV).eval()


def _inputs(B, T, seed=7):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(B, 256, T, generator=g) * 0.5).to(DEV), torch.randn(B, 1, 128, T, generator=g).to(DEV)


def _both(monkeypatch, run):
    """run(gd) under the layer-by-layer schedule, then under the default one (each on its own handle)."""
    old = run(_model(monkeypatch, False)).cpu()
    new = run(_model(monkeypatch, True)).cpu()
    return old, new


def _kernels(fn):
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events()]


@pytest.mark.parametrize("T,steps", [(862, 300), (43, 300)])
def test_ddpm_bit_identical(monkeypatch, T, steps):
    cond, x0 = _inputs(1, T)
    old, new = _both(monkeypatch, lambda gd: gd.sample(x0, cond, steps, None, None, seed=11))
    assert torch.isfinite(new).all()
    assert torch.equal(old, new)


@pytest.mark.parametrize("T", [862, 43])
def test_plms_bit_identical(monkeypatch, T):
    cond, x0 = _inputs(1, T, seed=3)
    old, new = _both(monkeypatch, lambda gd: gd.sample(x0, cond, 1000, 20))
    assert torch.isfinite(new).all()
    assert torch.equal(old, new)


def test_single_eval_bit_identical_and_deferred(monkeypatch):
    """One HEAD_EVAL evaluation; the default schedule runs the two-role kernel, the layer-by-layer one does not."""
    cond, x0 = _inputs(1, 862, seed=5)
    t = torch.full((1,), 417, dtype=torch.long, device=DEV)
    outs = {}
    for defer in (False, True):
        gd = _model(monkeypatch, defer)
        gd.denoise_fn(x0, t, cond)                          # prepare + warm-up
        names = _kernels(lambda: outs.__setitem__(defer, gd.denoise_fn(x0, t, cond).cpu()))
        assert any("tc_pair2_kernel" in n for n in names) == defer, defer
    assert torch.equal(outs[False], outs[True])


def test_packed_batch_bit_identical(monkeypatch):
    """Two items packed on one frame axis: 64-wide tiles, conv + residual CTAs fit the SMs -> deferred."""
    lens = [300, 251]
    cond, x0 = _inputs(2, max(lens), seed=9)
    old, new = _both(monkeypatch, lambda gd: gd.sample(x0, cond, 50, None, None, lengths=lens, seed=4))
    for b, n in enumerate(lens):
        assert torch.equal(old[b, :, :, :n], new[b, :, :, :n]), b


def test_wide_tile_batch_falls_back(monkeypatch):
    """Four items of 600 frames take 128-wide tiles: the layer-by-layer schedule, same results."""
    cond, x0 = _inputs(4, 600, seed=13)
    old, new = _both(monkeypatch, lambda gd: gd.sample(x0, cond, 20, None, None, seed=6))
    assert torch.equal(old, new)
    gd = _model(monkeypatch, True)
    t = torch.full((4,), 300, dtype=torch.long, device=DEV)
    gd.denoise_fn(x0, t, cond)
    assert not any("tc_pair2_kernel" in n for n in _kernels(lambda: gd.denoise_fn(x0, t, cond)))

"""In-kernel stamps of one WaveNet layer's two kernels in the alternation of a real evaluation (dsvc_diffnet_run_layer part
4), under the layer-by-layer schedule (DSVC_SKIP_DEFER=0) and the default one.  Needs a -DDSVC_TIMELINE build:
tools/build_variants.py libdsvc_tl.so, then

    DSVC_LIB=diffsvc_b200/lib/libdsvc_tl.so python tools/dev_timeline_eval.py [T] [layer]

The library prints the stamps itself."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import diffsvc_b200 as D  # noqa: E402
from diffsvc_b200 import _lib  # noqa: E402
from diffsvc_b200.hparams import hparams, DEFAULTS_44K  # noqa: E402
from oracle import diffsvc_oracle as O  # noqa: E402

T = int(sys.argv[1]) if len(sys.argv) > 1 else 862
LAYER = int(sys.argv[2]) if len(sys.argv) > 2 else 5
hparams.clear(); hparams.update(DEFAULTS_44K); hparams["pndm_speedup"] = 1
lib = _lib.load()
g = torch.Generator().manual_seed(1)
cond = (torch.randn(1, 256, T, generator=g) * 0.5).cuda(); x0 = torch.randn(1, 1, 128, T, generator=g).cuda()
for defer in (False, True):
    if defer:
        os.environ.pop("DSVC_SKIP_DEFER", None)
    else:
        os.environ["DSVC_SKIP_DEFER"] = "0"
    dn = D.DiffNet(128, math_mode="tc3f16"); dn.load_state_dict(O.synth_diffnet_weights())
    gd = D.GaussianDiffusion(None, 128, dn, timesteps=1000, K_step=1000, spec_min=[-5.0], spec_max=[0.0]).cuda().eval()
    gd.sample(x0, cond, 2, None, None, seed=1); torch.cuda.synchronize()
    h = dn.handle()
    print("== lib %s  T=%d  layer %d  DSVC_SKIP_DEFER=%s" % (os.environ.get("DSVC_LIB", "product"), T, LAYER,
                                                          os.environ.get("DSVC_SKIP_DEFER", "unset")), flush=True)
    for _ in range(2):                       # the second pass is printed warm
        _lib.check(lib.dsvc_diffnet_run_layer(h, LAYER, 4, 1, _lib.current_stream())); torch.cuda.synchronize()
    dn.release()

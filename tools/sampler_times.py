"""Sampler times of the library of the tree this script sits in, one JSON line: µs per DDPM step at 862 and 43 frames and
for 8 packed clips of 689 frames +- 25 % (300 steps), µs per 43-frame PLMS-50 call; median of 5 after a warm-up call,
CUDA events.  Comparing two builds: copy it into the other checkout and run the two alternately, one process each.

    python tools/sampler_times.py LABEL
"""
import json, os, statistics, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import synthetic as S
import diffsvc_b200 as D
from diffsvc_b200.hparams import hparams, DEFAULTS_44K
MEL = 128
def model():
    hparams.clear(); hparams.update(DEFAULTS_44K); hparams["pndm_speedup"] = 1
    dn = D.DiffNet(MEL, math_mode="tc3f16"); dn.load_state_dict(S.synth_diffnet_weights(), strict=True)
    return D.GaussianDiffusion(None, MEL, dn, timesteps=1000, K_step=1000, loss_type="l2", spec_min=[-5.0], spec_max=[0.0]).cuda().eval()
g = torch.Generator().manual_seed(1)
c862 = (torch.randn(1, 256, 862, generator=g) * 0.5).cuda(); x862 = torch.randn(1, 1, MEL, 862, generator=g).cuda()
c43 = (torch.randn(1, 256, 43, generator=g) * 0.5).cuda(); x43 = torch.randn(1, 1, MEL, 43, generator=g).cuda()
lens = (689 * (0.75 + 0.5 * torch.rand(8, generator=g))).round().long().tolist()
c8 = (torch.randn(8, 256, max(lens), generator=g) * 0.5).cuda(); x8 = torch.randn(8, 1, MEL, max(lens), generator=g).cuda()
legs = {"ddpm862": (lambda gd: gd.sample(x862, c862, 1000, None, None, seed=3), 1000),
        "ddpm43": (lambda gd: gd.sample(x43, c43, 1000, None, None, seed=3), 1000),
        "plms43": (lambda gd: gd.sample(x43, c43, 1000, 20), 1),
        "b8x689": (lambda gd: gd.sample(x8, c8, 300, None, None, lengths=lens, seed=3), 300)}
out = {}
with torch.no_grad():
    for k, (fn, n) in legs.items():
        gd = model(); fn(gd); torch.cuda.synchronize()
        ts = []
        for _ in range(5):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(gd); b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1000.0 / n)
        out[k] = round(statistics.median(ts), 2)
print(json.dumps({"tree": sys.argv[1] if len(sys.argv) > 1 else "", **out}))

"""Randomised parity run: fused path and dense path against the CPU oracle over random shapes / thresholds / scenes.
usage: python tools/fuzz_parity.py [n_cases] [seed]"""
import os, sys, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import yolov4_b200 as yb
from yolov4_b200.synth import synth_head_outputs
from oracle import oracle as orc

def same(got, want):
    for g, w in zip(got, want):
        if (g is None) != (w is None):
            return False
        if w is not None:
            g = g.cpu().numpy()
            if g.shape != w.shape:
                return False
            nan = np.isnan(w)                                  # NaN payload / sign bits are not part of the contract
            if not np.array_equal(np.isnan(g), nan) or not np.array_equal(g.view(np.uint32)[~nan], w.view(np.uint32)[~nan]):
                return False
    return True

n_cases = int(sys.argv[1]) if len(sys.argv) > 1 else 40
rng = np.random.RandomState(int(sys.argv[2]) if len(sys.argv) > 2 else 0)
bad = 0
for it in range(n_cases):
    # 104, 152, 200 and 600 are multiples of 8 but not of 32: an odd grid below an even one (600: 75, 37, 18)
    img = int(rng.choice([64, 96, 160, 224, 320, 416, 104, 152, 200, 600]))
    C = int(rng.choice([1, 3, 20, 33, 80, 100]))
    B = int(rng.randint(1, 5))
    conf = float(rng.choice([1e-4, 1e-3, 0.01, 0.05, 0.2, 0.5]))
    nmst = float(rng.choice([0.1, 0.3, 0.4, 0.45, 0.5, 0.7, 0.9]))
    kw = dict(fg_prob=float(rng.choice([0.005, 0.02, 0.05, 0.15])), clustered=bool(rng.randint(0, 2)))
    cfg = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": C}
    raws = synth_head_outputs(B, img, C, seed=int(rng.randint(1 << 30)), device="cuda", **kw)
    if rng.rand() < 0.3:                                       # a few absurd logits
        r = raws[int(rng.randint(3))]
        idx = torch.randint(0, r.numel(), (20,), device="cuda")
        r.view(-1)[idx] = torch.tensor(rng.choice([np.nan, np.inf, -np.inf, 60.0, -60.0, 95.0], 20), dtype=torch.float32, device="cuda")
    want = orc.detect([r.cpu().numpy() for r in raws], C, conf, nmst, nthreads=8)
    ok1 = same(yb.detect_raw(raws, C, conf, nmst), want)
    dense = torch.cat([yb.YOLOLayer(cfg, l, device="cuda").eval()(raws[l]) for l in range(3)], 1)
    ok2 = same(yb.postprocess(dense, C, conf, nmst), want)
    rows = sum(0 if w is None else len(w) for w in want)
    if not (ok1 and ok2):
        bad += 1
        print("MISMATCH", dict(img=img, C=C, B=B, conf=conf, nms=nmst, **kw), ok1, ok2, flush=True)
    elif it % 10 == 0:
        print("case %d ok (img %d C %d B %d conf %g nms %g rows %d)" % (it, img, C, B, conf, nmst, rows), flush=True)
print("fuzz: %d cases, %d mismatches" % (n_cases, bad))
sys.exit(1 if bad else 0)

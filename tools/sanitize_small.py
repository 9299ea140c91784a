"""Small end-to-end invocation for compute-sanitizer (memcheck / racecheck / synccheck): fused path, dense path, big tier,
build_target, at sizes that finish in seconds under the tool."""
import os, sys, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import yolov4_b200 as yb
from yolov4_b200.synth import synth_head_outputs, synth_labels
from oracle import oracle as orc
CFG = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": 80}
ok = True
for kw, conf, nmst in ((dict(fg_prob=0.03, clustered=True), 0.001, 0.4), (dict(), 1e-4, 0.4)):
    raws = synth_head_outputs(2, 416, 80, seed=3, device="cuda", **kw)
    want = orc.detect([r.cpu().numpy() for r in raws], 80, conf, nmst, nthreads=4)
    got = yb.detect_raw(raws, 80, conf, nmst)
    dense = torch.cat([yb.YOLOLayer(CFG, l, device="cuda").eval()(raws[l]) for l in range(3)], 1)
    got2 = yb.postprocess(dense, 80, conf, nmst)
    for g, g2, w in zip(got, got2, want):
        ok &= np.array_equal(g.cpu().numpy().view(np.uint32), w.view(np.uint32))
        ok &= np.array_equal(g2.cpu().numpy().view(np.uint32), w.view(np.uint32))
# all-ties input: every segment goes to the big tier
z = [torch.zeros_like(r) for r in synth_head_outputs(1, 96, 4, seed=0, device="cuda")]
got = yb.detect_raw(z, 4, 0.2, 0.5)
want = orc.detect([r.cpu().numpy() for r in z], 4, 0.2, 0.5, nthreads=2)
ok &= np.array_equal(got[0].cpu().numpy().view(np.uint32), want[0].view(np.uint32))
labels = synth_labels(2, 416, n_valid=20, seed=1, device="cuda")
d = yb.YOLOLayer(CFG, 1, device="cuda").train()(raws[1])
t = yb.YOLOLoss(CFG, 0.7, device="cuda").build_target(d["output"], d["pred"], 1, labels)
w = orc.build_target(d["pred"].cpu().numpy(), labels.cpu().numpy(), 1, 80, 0.7)
for a, b in zip(t, w):
    ok &= np.array_equal(a.cpu().numpy(), b, equal_nan=True)
# fused loss, forward and backward (labels with a non-finite and a negative box: both branches of the ignore test)
labels[0, 3, 2] = float("inf"); labels[1, 2, 2] = -9.0
raws_g = [r.clone().requires_grad_(True) for r in raws]
loss = yb.fused_yolo_loss(raws_g, labels, CFG, 0.7)
loss.backward()
ok &= bool(torch.isfinite(raws_g[0].grad).any().item())
# round 2: the three scales of build_target in one launch pair, the train decode's backward from the raw tensor, the padded epilogue,
# the single-rank exchange, and (YL_FLAG=tma in the environment) the TMA flag kernel through detect_raw above
ds = [yb.YOLOLayer(CFG, l, device="cuda").train()(raws[l].clone().requires_grad_(True)) for l in range(3)]
one = yb.build_targets3([x["output"] for x in ds], [x["pred"] for x in ds], [0, 1, 2], labels, yb.ANCHORS_PX, yb.ANCHOR_MASK, 0.7, 80)
for a, b in zip(one[1], yb.YOLOLoss(CFG, 0.7, device="cuda").build_target(ds[1]["output"], ds[1]["pred"], 1, labels)):
    ok &= bool(torch.equal(a, b) or (torch.isnan(a) == torch.isnan(b)).all().item())
ds[0]["output"].sum().backward()
hp = yb.HeadPostprocessor(2, [52, 26, 13], 80, 1e-3, 0.4, cap_out=8192)
rows, meta = hp.run(raws)
out = yb.coco_rows_padded(rows, meta[:2], [[480, 640, 312, 416]] * 2, [7, 9], list(range(1, 81)))
ok &= out.shape[0] == int(meta[:2].sum())
from yolov4_b200.sharded import DetectionExchange
ex = DetectionExchange(2, 8192, torch.device("cuda", 0), slots=2)
for slot in (0, 1, 0):
    ex.push(rows, meta[:2], slot); ex.wait(slot)
    got = ex.results(slot)
    ok &= all(torch.equal(g, rows[b, :g.shape[0]]) for b, g in enumerate(got) if g is not None)
    ex.release(slot)
ok &= ex.status() == 0
ex.close()
torch.cuda.synchronize()
print("sanitize_small:", "ok" if ok else "MISMATCH")
sys.exit(0 if ok else 1)

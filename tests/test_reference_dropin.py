"""GPU: the B200 path at the drop-in boundary of the reference (zjykzj/YOLOv4), after yolov4_b200.patch_reference().

Every test runs in two forms.  The golden form always runs: the patched boundary symbols against outputs of the UNMODIFIED
reference stored under tests/golden/ by tests/golden/make_golden.py (postprocess.npz: the reference's decoded [2, 1008, 85] tensor
of seeded 128x128 head outputs and the rows of its postprocess; loss.npz: raw head tensors, labels, the reference's loss and its
autograd gradient with respect to the raw tensors).  The live form runs where the reference is installed into baseline/_ref
(tools/install_reference.sh; git-ignored): the reference model with and without the patch, on the same GPU and the same inputs.

  eval   decoded [B,M,85] within 1e-5 relative (north_star's tolerance); postprocess (utils.py:92-223) on the SAME decoded tensor:
         identical lists, bit for bit (live: yolo.model.yolov4.YOLOv4, yolov4.py:270-324, random init with non-degenerate BN)
  train  the reference's criterion (yololoss.py:373-443) on the patched layers: loss within 1e-5, gradient within 2e-5, both with
         the reference's own forward on top of the B200 YOLOLayer / build_target (its in-place mask multiplies must not break
         autograd) and with the rebound forward
"""
import os
import sys

import numpy as np
import pytest
import torch
from torch import nn

from test_cabi_cpu import _stand_in_reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "baseline", "_ref")
HAVE_REF = os.path.isdir(os.path.join(REF, "yolo"))

pytestmark = pytest.mark.gpu

IMG = 128           # grids 16 / 8 / 4: the reference's Python postprocess stays fast


@pytest.fixture(scope="module")
def ref():
    import yaml
    sys.path.insert(0, REF)
    import yolo.model.yolov4 as m4
    import yolo.model.yololayer as ml
    import yolo.model.yololoss as mlo
    import yolo.util.utils as mu
    saved = dict(layer=ml.YOLOLayer, layer4=m4.YOLOLayer, post=mu.postprocess, bt=mlo.YOLOLoss.build_target, fwd=mlo.YOLOLoss.forward)

    def restore():
        ml.YOLOLayer = saved["layer"]
        m4.YOLOLayer = saved["layer4"]
        mu.postprocess = saved["post"]
        mlo.YOLOLoss.build_target = saved["bt"]
        mlo.YOLOLoss.forward = saved["fwd"]

    cfg = yaml.safe_load(open(os.path.join(REF, "config", "yolov4_default.cfg")))
    yield dict(m4=m4, ml=ml, mlo=mlo, mu=mu, cfg=cfg, restore=restore, saved=saved)
    restore()
    sys.path.remove(REF)


def _model(m4, cfg, dev):
    torch.manual_seed(0)
    model = m4.YOLOv4(cfg["MODEL"], device=dev).to(dev)
    # the reference initialises BN weights ~ N(0, 0.01) (yolov4.py:292): every head logit is ~0 after 100 layers (SURVEY 7-2).
    # Weight 1 and statistics taken from one batch give O(1) logits on both sides of every threshold.
    for m in model.modules():
        if isinstance(m, nn.BatchNorm2d):
            nn.init.constant_(m.weight, 1.0)
            m.momentum = 1.0
    return model


def _calibrate(model, x):
    model.train()
    with torch.no_grad():
        model(x)
    return model


def _live_eval(ref):
    import yolov4_b200 as yb
    dev = torch.device("cuda")
    m4, cfg = ref["m4"], ref["cfg"]
    ref["restore"]()
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 3, IMG, IMG, generator=g).to(dev)
    model_ref = _calibrate(_model(m4, cfg, dev), x).eval()
    assert type(model_ref.head.yolo1[2]).__module__ == "yolo.model.yololayer"
    with torch.no_grad():
        out_ref = model_ref(x)
    # the reference's own postprocess, unpatched, on its own decoded tensor (it overwrites its input: clone)
    conf, nmst = 0.3, 0.45
    want = ref["saved"]["post"](out_ref.clone(), 80, conf, nmst)

    done = yb.patch_reference()
    assert "yolo.model.yolov4.YOLOLayer" in done and "yolo.util.utils.postprocess" in done
    try:
        model_b = _model(m4, cfg, dev)
        assert type(model_b.head.yolo1[2]).__module__ == "yolov4_b200.yololayer"
        model_b.load_state_dict(model_ref.state_dict(), strict=True)          # val.py:82-83: checkpoints load unchanged
        model_b.eval()
        with torch.no_grad():
            out_b = model_b(x)
        assert out_b.shape == out_ref.shape == (2, 3 * (16 * 16 + 8 * 8 + 4 * 4), 85)
        a, b = out_ref.cpu().numpy(), out_b.cpu().numpy()
        assert np.isfinite(a).all()
        rel = np.abs(a - b) / np.maximum(np.abs(a), 1e-30)
        assert rel.max() <= 1e-5, rel.max()                                   # north_star: decoded values within 1e-5 relative
        got = ref["mu"].postprocess(out_ref, 80, conf, nmst)                  # the patched symbol, same decoded input
    finally:
        ref["restore"]()
    n_rows = 0
    for gi, wi in zip(got, want):
        assert (gi is None) == (wi is None)
        if wi is not None:
            assert gi.shape == wi.shape
            assert np.array_equal(gi.cpu().numpy().view(np.uint32), wi.cpu().numpy().view(np.uint32))
            n_rows += wi.shape[0]
    assert n_rows > 50, "the test input must produce detections"


def _live_train(ref, loss_forward):
    import yolov4_b200 as yb
    from yolov4_b200.synth import synth_labels
    dev = torch.device("cuda")
    m4, mlo, cfg = ref["m4"], ref["mlo"], ref["cfg"]
    ref["restore"]()
    g = torch.Generator().manual_seed(2)
    x = torch.randn(2, 3, IMG, IMG, generator=g).to(dev)
    labels = synth_labels(2, IMG, n_valid=12, seed=3, device="cpu").double()          # as the loader collates them
    targets = {"padded_labels": labels}

    def loss_and_grads(model):
        model.train()
        model.zero_grad()
        crit = mlo.YOLOLoss(cfg["MODEL"], ignore_thresh=float(cfg["CRITERION"]["IGNORE_THRESH"]), device=dev).to(dev)
        loss = crit(model(x), targets)
        loss.backward()
        gs = [p.grad.detach().clone() for p in list(model.head.yolo1[1].parameters()) + list(model.head.yolo3[1].parameters())]
        return float(loss), gs

    model_ref = _calibrate(_model(m4, cfg, dev), x)
    loss_ref, g_ref = loss_and_grads(model_ref)
    assert np.isfinite(loss_ref) and loss_ref > 0

    done = yb.patch_reference(loss_forward=loss_forward)
    assert ("yolo.model.yololoss.YOLOLoss.forward" in done) == loss_forward
    try:
        model_b = _model(m4, cfg, dev)
        model_b.load_state_dict(model_ref.state_dict(), strict=True)
        for mr, mb in zip(model_ref.modules(), model_b.modules()):
            if isinstance(mr, nn.BatchNorm2d):
                mb.momentum = mr.momentum
        loss_b, g_b = loss_and_grads(model_b)      # the reference's forward multiplies dict['output'] in place: must back-propagate
    finally:
        ref["restore"]()
    assert abs(loss_b - loss_ref) <= 1e-5 * abs(loss_ref), (loss_b, loss_ref)
    for a, b in zip(g_ref, g_b):
        scale = float(a.abs().max())
        assert scale > 0
        assert float((a - b).abs().max()) <= 2e-5 * scale, (float((a - b).abs().max()), scale)


# ------------------------------------------------------------------------------------------------ golden form
def _patched_boundary(monkeypatch, loss_forward=True):
    """patch_reference() over stand-ins of the reference's module layout: the calls below go through the rebound symbols."""
    import yolov4_b200 as yb
    _stand_in_reference(monkeypatch)
    done = yb.patch_reference(loss_forward=loss_forward)
    assert "yolo.model.yololayer.YOLOLayer" in done and "yolo.util.utils.postprocess" in done
    return sys.modules["yolo.model.yololayer"], sys.modules["yolo.util.utils"], sys.modules["yolo.model.yololoss"]


def _golden_eval(golden_dir, monkeypatch):
    import yolov4_b200 as yb
    from yolov4_b200.synth import synth_head_outputs
    ml, mu, _ = _patched_boundary(monkeypatch)
    g = np.load(os.path.join(golden_dir, "postprocess.npz"))
    # the head outputs the reference decoded in make_golden.gen_postprocess (the same seeded generator and arguments)
    raws = [r.cuda() for r in synth_head_outputs(2, IMG, 80, seed=3, fg_prob=0.04, clustered=True)]
    cfg = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": 80}
    with torch.no_grad():
        out_b = torch.cat([ml.YOLOLayer(cfg, l, device="cuda").eval()(raws[l]) for l in range(3)], 1)
    assert out_b.shape == (2, 3 * (16 * 16 + 8 * 8 + 4 * 4), 85)
    a, b = g["pred"].astype(np.float64), out_b.cpu().numpy().astype(np.float64)
    assert np.isfinite(a).all() and np.isfinite(b).all()
    tiny = np.abs(a) < 1e-30            # sigmoid outputs below the fp32 normal range are compared absolutely (test_oracle_golden)
    assert np.abs(b[tiny]).max(initial=0.0) < 1e-30
    rel = np.abs(a - b)[~tiny] / np.abs(a[~tiny])
    assert rel.max() <= 1e-5, rel.max()                                       # north_star: decoded values within 1e-5 relative
    pred = torch.from_numpy(g["pred"]).cuda()                                 # the reference's own decoded tensor
    n_rows, i = 0, 0
    while f"s{i}_conf" in g:
        got = mu.postprocess(pred, 80, float(g[f"s{i}_conf"]), float(g[f"s{i}_nms"]))
        counts, rows = g[f"s{i}_counts"], g[f"s{i}_rows"]
        assert len(got) == len(counts)
        o = 0
        for gi, n in zip(got, counts):
            assert (gi is None) == (n == 0), (i, n)
            if n:
                assert gi.shape == (n, 7)
                assert np.array_equal(gi.cpu().numpy().view(np.uint32), rows[o:o + n].view(np.uint32)), (i, o)
            o += n
        n_rows += o
        i += 1
    assert i == 5 and n_rows > 50, "the test input must produce detections"


def _reference_forward_in_place(crit, outputs, labels):
    """The reference's YOLOLoss.forward (yololoss.py:373-443) in its own form, on top of the criterion's build_target: the mask
    products are taken in place on the layer's output (yololoss.py:402-408), then the four sums.  Written out here because the
    golden form runs without the reference's code; loss.npz holds the reference's value and gradient it must reproduce."""
    bce, l2 = nn.BCELoss(reduction="sum"), nn.MSELoss(reduction="sum")
    total = 0
    for od in outputs:
        output = od["output"]
        target, obj_mask, tgt_mask, tgt_scale = crit.build_target(output, od["pred"], int(od["layer_no"]), labels)
        sel = np.r_[0:4, 5:output.shape[-1]]
        output[..., 4] *= obj_mask
        output[..., sel] *= tgt_mask
        output[..., 2:4] *= tgt_scale
        target[..., 4] *= obj_mask
        target[..., sel] *= tgt_mask
        target[..., 2:4] *= tgt_scale
        bce_w = nn.BCELoss(weight=tgt_scale * tgt_scale, reduction="sum")
        total = total + bce_w(output[..., :2], target[..., :2]) + l2(output[..., 2:4], target[..., 2:4]) / 2 + \
            bce(output[..., 4], target[..., 4]) + bce(output[..., 5:], target[..., 5:])
    return total


def _golden_train(golden_dir, monkeypatch, loss_forward):
    import yolov4_b200 as yb
    ml, _, mlo = _patched_boundary(monkeypatch, loss_forward=loss_forward)
    assert mlo.YOLOLoss.build_target is yb.YOLOLoss.build_target
    assert (mlo.YOLOLoss.forward is yb.YOLOLoss.forward) == loss_forward
    g = np.load(os.path.join(golden_dir, "loss.npz"))
    cfg = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": int(g["C"])}
    leaves = [torch.from_numpy(g[f"raw{l}"]).cuda().requires_grad_(True) for l in range(3)]
    labels = torch.from_numpy(g["labels"]).double()                            # as the loader collates them
    # in the model the layers see a conv output, not a leaf (make_golden.gen_loss does the same)
    outs = [ml.YOLOLayer(cfg, l, device="cuda").train()(leaves[l] * 1.0) for l in range(3)]
    crit = yb.YOLOLoss(cfg, ignore_thresh=0.7, device="cuda")
    loss = crit(outs, {"padded_labels": labels}) if loss_forward else _reference_forward_in_place(crit, outs, labels)
    loss.backward()
    want = float(g["loss"])
    assert abs(loss.item() - want) <= 1e-5 * abs(want), (loss.item(), want)
    for l in range(3):
        a, b = torch.from_numpy(g[f"grad{l}"]).double(), leaves[l].grad.cpu().double()
        scale = float(a.abs().max())
        assert scale > 0
        assert float((a - b).abs().max()) <= 2e-5 * scale, (l, float((a - b).abs().max()), scale)


# ------------------------------------------------------------------------------------------------ tests
def test_eval_model_and_postprocess_patched_vs_unpatched(golden_dir, monkeypatch, request):
    _golden_eval(golden_dir, monkeypatch)
    if HAVE_REF:
        monkeypatch.undo()
        _live_eval(request.getfixturevalue("ref"))


@pytest.mark.parametrize("loss_forward", [False, True])
def test_train_loss_and_gradient_patched_vs_unpatched(golden_dir, monkeypatch, request, loss_forward):
    _golden_train(golden_dir, monkeypatch, loss_forward)
    if HAVE_REF:
        monkeypatch.undo()
        _live_train(request.getfixturevalue("ref"), loss_forward)

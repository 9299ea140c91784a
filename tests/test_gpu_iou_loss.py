"""The fused loss with an IoU box term (iou_loss='giou' | 'diou' | 'ciou') on the B200 against tests/iou_loss_spec.py.

  per run       component 0 within 1e-5 relative of the spec, component 1 exactly 0, components 2 and 3 within rtol 1e-12 of
                the iou_loss=None run; gradient channels 4.. bit for bit those of the None run; box channels 0 off the matched
                cells and within the stated bound (iou_loss_spec.GRAD_REL / GRAD_ABS) at them, NaN where the spec has NaN
  scenes        608 px, B = 4, 50 GTs per image with predictions planted near them; every valid set of loss_edge_cases;
                predictions planted exactly on their GT (the tie rule); iou_normalizer 0.07 and 0; 16-bit heads; a CUDA-graph
                replay of the three-scale chain; a few SGD steps on the box logits
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import iou_loss_spec as spec                                           # noqa: E402
import loss_edge_cases as cases                                        # noqa: E402
from oracle import oracle as orc                                      # noqa: E402  (checker only)
import yolov4_b200 as yb                                               # noqa: E402
from yolov4_b200.synth import synth_labels                             # noqa: E402
from yolov4_b200.yololoss import fused_yolo_loss, fused_yolo_loss_components   # noqa: E402

KINDS = spec.KINDS


def cfg_of(C, mask=orc.ANCHOR_MASK):
    return {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": mask, "N_CLASSES": C}


def bit_equal(a, b):
    a, b = a.detach().contiguous().cpu(), b.detach().contiguous().cpu()
    ia = a.view(torch.int16 if a.element_size() == 2 else torch.int32)
    ib = b.view(torch.int16 if b.element_size() == 2 else torch.int32)
    na, nb = torch.isnan(a.float()), torch.isnan(b.float())
    return a.shape == b.shape and torch.equal(na, nb) and torch.equal(ia[~na], ib[~nb])


def grads(heads, lab, cfg, thr, up=1.0, **kw):
    hs = [h.detach().clone().requires_grad_(True) for h in heads]
    loss = fused_yolo_loss(hs, lab, cfg, thr, **kw)
    loss.backward(torch.tensor(up, dtype=torch.float32, device="cuda"))
    return loss.detach(), [h.grad for h in hs]


def scene_608(seed=31, B=4):
    C = 80
    lab = synth_labels(B, 608, n_valid=50, seed=seed).numpy()
    raws = cases.heads(B, 608, C, seed)
    cases.plant_near_gts(raws, lab, C, orc.ANCHOR_MASK, every=2)        # the other half keeps its random predictions
    for b in range(B):                  # three 6 px GTs (layer 0, slot 0) with a 1 px prediction in the far corner of their cell
        for k, c in enumerate((2, 5, 8)):
            lab[b, 50 + k] = ((c + 0.1) * 8, (c + 0.1) * 8, 6.0, 6.0, 0.0)
            cases.plant_box(raws, C, orc.ANCHOR_MASK, b, 0, 0, ((c + 0.97) * 8, (c + 0.97) * 8, 1.0, 1.0))
    return dict(name="608", C=C, labels=np.ascontiguousarray(lab, np.float32), raws=raws, mask=orc.ANCHOR_MASK, thrs=(0.7,))


def check_run(c, kind, norm=1.0, thr=None):
    """Every check of the module docstring on one label set; returns the per-layer spec results."""
    C, mask = c["C"], c["mask"]
    thr = c["thrs"][0] if thr is None else thr
    cfg = cfg_of(C, mask)
    lab = torch.from_numpy(c["labels"]).cuda()
    heads = [torch.from_numpy(r).cuda() for r in c["raws"]]
    kw = dict(iou_loss=kind, iou_normalizer=norm)
    specs = [spec.layer_spec(c["raws"][l], c["labels"], l, C, thr, kind, norm, mask=mask) for l in range(3)]
    out = []
    for l in range(3):
        want = specs[l][0]
        got = fused_yolo_loss_components([heads[l]], lab, cfg, thr, layers=[l], **kw).cpu().numpy()
        none = fused_yolo_loss_components([heads[l]], lab, cfg, thr, layers=[l]).cpu().numpy()
        what = "%s %s n %r layer %d" % (c["name"], kind, norm, l)
        assert np.isnan(got[0]) == np.isnan(want[0]), what
        if not np.isnan(want[0]):
            assert abs(got[0] - want[0]) <= 1e-5 * abs(want[0]) + 1e-6, (what, got[0], want[0])
        assert got[1] == 0.0, what
        np.testing.assert_allclose(got[2:], none[2:], rtol=1e-12, atol=0, equal_nan=True, err_msg=what)
    _, g_iou = grads(heads, lab, cfg, thr, **kw)
    _, g_none = grads(heads, lab, cfg, thr)
    nch = 5 + C
    for l in range(3):
        cells, term, graw, p = specs[l][2]
        extreme = spec.extreme_extent(p)
        g, g0 = g_iou[l], g_none[l]
        what = "%s %s n %r layer %d" % (c["name"], kind, norm, l)
        for a in range(3):
            assert bit_equal(g[:, a * nch + 4:(a + 1) * nch], g0[:, a * nch + 4:(a + 1) * nch]), what + ": channels 4.. differ"
        box = torch.cat([g[:, a * nch:a * nch + 4] for a in range(3)], 1).cpu().numpy()
        matched = np.zeros(box.shape, bool)
        for (b, a, j, i), gr, tm, ext in zip(cells, graw, term, extreme):
            matched[b, 4 * a:4 * a + 4, j, i] = True
            got4 = box[b, 4 * a:4 * a + 4, j, i]
            if ext:                                 # extents outside [1e-30, 1e30]: the class with its own check (iou_loss_spec)
                assert not np.isnan(tm) or np.isnan(got4).all(), "%s cell %r: %r" % (what, (b, a, j, i), got4)
                continue
            assert spec.within_bound(got4, gr, norm).all(), "%s cell %r: %r vs spec %r" % (what, (b, a, j, i), got4, gr)
        assert (box[~matched] == 0).all(), what + ": box gradient off the matched cells"
        out.append((cells, graw))
    return out


@pytest.mark.parametrize("kind", KINDS)
def test_608_planted_near_gts(kind):
    c = scene_608()
    res = check_run(c, kind)
    assert sum(len(r[0]) for r in res) > 150
    # overlapping, disjoint and contained pairs all occur
    kinds = set()
    for l in range(3):
        _, p, g, _ = spec.matched_pairs(c["raws"][l], c["labels"], l, c["C"])
        lo_p, hi_p, lo_g, hi_g = p[:, :2] - p[:, 2:] / 2, p[:, :2] + p[:, 2:] / 2, g[:, :2] - g[:, 2:] / 2, g[:, :2] + g[:, 2:] / 2
        overlap = ((np.minimum(hi_p, hi_g) - np.maximum(lo_p, lo_g)) > 0).all(1)
        inside = ((lo_p >= lo_g) & (hi_p <= hi_g)).all(1) | ((lo_g >= lo_p) & (hi_g <= hi_p)).all(1)
        kinds |= {"disjoint"} if (~overlap).any() else set()
        kinds |= {"contained"} if inside.any() else set()
        kinds |= {"overlap"} if (overlap & ~inside).any() else set()
    assert kinds == {"disjoint", "contained", "overlap"}, kinds


@pytest.mark.parametrize("name", sorted(cases.VALID))
@pytest.mark.parametrize("kind", KINDS)
def test_edge_case_sets(kind, name):
    c = cases.get(name)
    for thr in c["thrs"][:2]:
        check_run(c, kind, thr=thr)


@pytest.mark.parametrize("kind", KINDS)
def test_prediction_exactly_on_its_gt(kind):
    """Labels = decoded prediction x stride (exact: the stride is a power of two), so p == g bit for bit at those cells."""
    c = scene_608(seed=41, B=2)
    lab = c["labels"].copy()
    n_exact = 0
    for l in range(3):
        _, pred = orc.decode_train(c["raws"][l], l, c["C"])
        owner = spec.last_gt_per_cell(lab, l, pred.shape[2])
        for (b, a, j, i), t in owner.items():
            lab[b, t, :4] = pred[b, a, j, i] * np.float32(orc.STRIDES[l])
    c = dict(c, labels=lab, name="exact")
    for l in range(3):
        _, p, g, _ = spec.matched_pairs(c["raws"][l], lab, l, c["C"])
        n_exact += int((p == g).all(1).sum())
    assert n_exact > 50, n_exact
    check_run(c, kind)


@pytest.mark.parametrize("kind", KINDS)
def test_normalizer_scales_box_term_only(kind):
    c = scene_608(seed=43, B=2)
    cfg = cfg_of(c["C"])
    lab = torch.from_numpy(c["labels"]).cuda()
    heads = [torch.from_numpy(r).cuda() for r in c["raws"]]
    base = fused_yolo_loss_components(heads, lab, cfg, iou_loss=kind).cpu().numpy()
    _, g1 = grads(heads, lab, cfg, 0.7, iou_loss=kind)
    for norm in (0.07, 0.0):
        check_run(c, kind, norm)
        got = fused_yolo_loss_components(heads, lab, cfg, iou_loss=kind, iou_normalizer=norm).cpu().numpy()
        np.testing.assert_allclose(got[0], base[0] * norm, rtol=1e-6, atol=1e-9)
        np.testing.assert_allclose(got[2:], base[2:], rtol=1e-12)
        _, gn = grads(heads, lab, cfg, 0.7, iou_loss=kind, iou_normalizer=norm)
        for a, b in zip(gn, g1):
            box = torch.zeros(a.shape[1], dtype=torch.bool)
            for s in range(3):
                box[s * 85:s * 85 + 4] = True
            torch.testing.assert_close(a[:, box], b[:, box] * norm, rtol=1e-6, atol=1e-12)
            assert bit_equal(a[:, ~box], b[:, ~box])


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("kind", KINDS)
def test_16bit_heads_match_widened_fp32(kind, dt):
    c = scene_608(seed=47, B=2)
    cfg = cfg_of(c["C"])
    lab = torch.from_numpy(c["labels"]).cuda()
    h16 = [torch.from_numpy(r).cuda().to(dt) for r in c["raws"]]
    wide = [h.float() for h in h16]
    kw = dict(iou_loss=kind, iou_normalizer=0.07)
    np.testing.assert_allclose(fused_yolo_loss_components(h16, lab, cfg, **kw).cpu().numpy(),
                               fused_yolo_loss_components(wide, lab, cfg, **kw).cpu().numpy(), rtol=1e-12, atol=0)
    for up in (1.0, 65536.0, 1e38):
        l16, g16 = grads(h16, lab, cfg, 0.7, up, **kw)
        l32, g32 = grads(wide, lab, cfg, 0.7, up, **kw)
        assert l16.dtype == torch.float32
        np.testing.assert_allclose(l16.item(), l32.item(), rtol=1e-6)
        for a, b in zip(g16, g32):
            assert a.dtype == dt and bit_equal(a, b.to(dt)), (kind, dt, up)
        if up == 1e38 and dt == torch.float16:           # bf16 shares fp32's exponent range: it overflows where fp32 does
            assert any(torch.isinf(a).any() for a in g16)


@pytest.mark.parametrize("kind", KINDS)
def test_cuda_graph_replay_equals_eager(kind):
    c = scene_608(seed=53, B=2)
    cfg = cfg_of(c["C"])
    lab = torch.from_numpy(c["labels"]).cuda()
    heads = [torch.from_numpy(r).cuda() for r in c["raws"]]
    eager = fused_yolo_loss_components(heads, lab, cfg, iou_loss=kind).cpu().numpy()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fused_yolo_loss_components(heads, lab, cfg, iou_loss=kind)           # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fused_yolo_loss_components(heads, lab, cfg, iou_loss=kind)
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        np.testing.assert_allclose(out.cpu().numpy(), eager, rtol=1e-12, atol=0)


@pytest.mark.parametrize("kind", KINDS)
def test_sgd_on_box_logits_lowers_the_box_term(kind):
    c = scene_608(seed=59, B=2)
    cfg = cfg_of(c["C"])
    lab = torch.from_numpy(c["labels"]).cuda()
    heads = [torch.from_numpy(r).cuda() for r in c["raws"]]
    box = torch.zeros(heads[0].shape[1], dtype=torch.bool, device="cuda")
    for s in range(3):
        box[s * 85:s * 85 + 4] = True
    vals = []
    for _ in range(6):
        vals.append(fused_yolo_loss_components(heads, lab, cfg, iou_loss=kind)[0].item())
        _, gr = grads(heads, lab, cfg, 0.7, iou_loss=kind)
        heads = [h - 0.05 * g * box[None, :, None, None] for h, g in zip(heads, gr)]
    assert all(b < a for a, b in zip(vals, vals[1:])), vals
    assert vals[-1] < 0.95 * vals[0], vals


def test_autocast_gradscaler_training_step():
    """A model under autocast with GradScaler trains with iou_loss='ciou', iou_normalizer=0.07: heads and gradients are fp16."""
    torch.manual_seed(0)
    lab = synth_labels(2, 256, n_valid=20, seed=3, device="cuda")
    convs = torch.nn.ModuleList([torch.nn.Conv2d(8, 255, 1) for _ in range(3)]).cuda()
    xs = [torch.randn(2, 8, 256 // s, 256 // s, device="cuda") for s in (8, 16, 32)]
    opt = torch.optim.SGD(convs.parameters(), lr=1e-3)
    scaler = torch.amp.GradScaler("cuda")
    cfg = cfg_of(80)
    for _ in range(3):
        opt.zero_grad()
        with torch.autocast("cuda", dtype=torch.float16):
            heads = [m(x) for m, x in zip(convs, xs)]
            for h in heads:
                h.retain_grad()
            loss = fused_yolo_loss(heads, lab, cfg, iou_loss="ciou", iou_normalizer=0.07)
        assert all(h.dtype == torch.float16 for h in heads) and loss.dtype == torch.float32
        scaler.scale(loss).backward()
        assert all(h.grad.dtype == torch.float16 for h in heads)
        scaler.step(opt)
        scaler.update()
    assert np.isfinite(loss.item())

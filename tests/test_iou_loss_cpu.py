"""CPU checks of the fused loss's IoU box term (tests/iou_loss_spec.py): the float64 spec is torchvision's three box losses, the
fp32 model of the kernel stays within the stated gradient bound of it over a million box pairs drawn like 608-pixel training
data, and the Python and C entry points validate iou_loss / iou_normalizer before any CUDA work."""
import math

import numpy as np
import pytest
import torch
from torchvision.ops import complete_box_iou_loss, distance_box_iou_loss, generalized_box_iou_loss

import iou_loss_spec as spec
from oracle import oracle as orc

TV = {"giou": generalized_box_iou_loss, "diou": distance_box_iou_loss, "ciou": complete_box_iou_loss}


def _xyxy(b):
    b = torch.as_tensor(b, dtype=torch.float64)
    return torch.stack([b[:, 0] - b[:, 2] / 2, b[:, 1] - b[:, 3] / 2, b[:, 0] + b[:, 2] / 2, b[:, 1] + b[:, 3] / 2], 1)


def _pairs():
    """(p, g) rows (cx, cy, w, h): random, disjoint, touching, contained, identical, zero-height and tied boxes."""
    rng = np.random.RandomState(0)
    rnd_p = np.concatenate([rng.uniform(0, 20, (200, 2)), rng.uniform(0.05, 6, (200, 2))], 1)
    rnd_g = np.concatenate([rnd_p[:, :2] + rng.normal(0, 2, (200, 2)), rng.uniform(0.05, 6, (200, 2))], 1)
    rows = [
        ((1.0, 1.0, 1.0, 1.0), (5.0, 5.0, 1.0, 2.0)),           # disjoint
        ((1.0, 1.0, 2.0, 2.0), (3.0, 1.0, 2.0, 2.0)),           # touching (zero-width overlap)
        ((2.0, 2.0, 1.0, 1.0), (2.25, 2.0, 4.0, 3.0)),          # contained
        ((2.0, 2.0, 4.0, 3.0), (2.25, 2.0, 1.0, 1.0)),          # containing
        ((3.5, 7.25, 1.5, 0.75), (3.5, 7.25, 1.5, 0.75)),       # identical
        ((1.0, 1.0, 2.0, 0.0), (1.5, 1.0, 2.0, 1.0)),           # zero-height prediction
        ((1.0, 1.0, 2.0, 1.0), (1.5, 1.0, 2.0, 0.0)),           # zero-height GT
        ((1.0, 1.0, 2.0, 1.0), (1.5, 1.0, 3.0, 1.0)),           # tied left edges, tied y extents
        ((1.0, 1.0, 2.0, 1.0), (0.5, 1.25, 1.0, 1.5)),          # tied left edges only
        ((0.5, 0.5, 1.0, 2.0), (0.75, 0.5, 0.5, 2.0)),          # tied right edges
    ]
    p = np.concatenate([rnd_p, np.array([r[0] for r in rows])])
    g = np.concatenate([rnd_g, np.array([r[1] for r in rows])])
    return p, g


@pytest.mark.parametrize("kind", spec.KINDS)
def test_spec_is_torchvision(kind):
    p, g = _pairs()
    pt = torch.tensor(p, dtype=torch.float64, requires_grad=True)
    want = TV[kind](_xyxy(pt), _xyxy(g), reduction="none", eps=1e-7)
    (wgrad,) = torch.autograd.grad(want.sum(), pt)
    loss, grad = spec.box_loss(kind, p, g)
    fin = ~np.isnan(want.detach().numpy())
    np.testing.assert_allclose(loss[fin], want.detach().numpy()[fin], rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(grad[fin], wgrad.numpy()[fin], rtol=1e-12, atol=1e-15)
    assert np.isnan(loss[~fin]).all() and np.isnan(grad[~fin]).all()


def test_hand_computed_values():
    # disjoint unit squares 4 apart along x: iou 0, enclosure 5 x 1
    p, g = [(0.5, 0.5, 1.0, 1.0)], [(4.5, 0.5, 1.0, 1.0)]
    assert spec.box_loss("giou", p, g)[0][0] == pytest.approx(1 + (5 - 2) / (5 + 1e-7), rel=1e-12)
    assert spec.box_loss("diou", p, g)[0][0] == pytest.approx(1 + 16 / (26 + 1e-7), rel=1e-12)
    # identical boxes: 1 - area / (area + eps), no penalty, and the gradient splits every tie evenly
    for kind in spec.KINDS:
        loss, grad = spec.box_loss(kind, [(2.0, 3.0, 2.0, 1.0)], [(2.0, 3.0, 2.0, 1.0)])
        assert loss[0] == pytest.approx(1e-7 / (2 + 1e-7), rel=1e-9)
        assert np.all(np.isfinite(grad))
    # same centre, GT twice as wide: iou 1/2, v = 4/pi^2 (atan 2 - atan 1)^2
    p, g = [(0.0, 0.0, 1.0, 1.0)], [(0.0, 0.0, 2.0, 1.0)]
    iou = 1.0 / (2.0 + 1e-7)
    v = 4 / math.pi ** 2 * (math.atan(2.0) - math.atan(1.0)) ** 2
    assert spec.box_loss("ciou", p, g)[0][0] == pytest.approx(1 - iou + v * v / (1 - iou + v + 1e-7), rel=1e-12)
    # a zero-height prediction and GT: 0 / 0 in CIoU's aspect term gives NaN in the term and all four derivatives
    loss, grad = spec.box_loss("ciou", [(0.0, 0.0, 0.0, 0.0)], [(0.0, 0.0, 0.0, 0.0)])
    assert np.isnan(loss).all() and np.isnan(grad).all()


def _draw_608(n, seed):
    """Pairs drawn like 608 training data, in grid units: GT extents anchor x exp(N(0, 0.5^2)) (5 % down to 1e-3), centres
    anywhere in the 76 / 38 / 19 grids, predictions decoded at the GT's cell; 30 % planted near their GT."""
    rng = np.random.RandomState(seed)
    f = np.float32
    layer = rng.randint(0, 3, n)
    F = np.array([76, 38, 19])[layer]
    anc = np.array([orc.masked_anchors_grid(l) for l in range(3)])
    aw = anc[layer, rng.randint(0, 3, n)]
    gwh = (aw * np.exp(rng.normal(0, 0.5, (n, 2)))).astype(f)
    small = rng.rand(n) < 0.05
    gwh[small] = np.exp(rng.uniform(np.log(1e-3), 0, (small.sum(), 2))).astype(f)
    gc = (rng.rand(n, 2) * F[:, None]).astype(f)
    ij = np.floor(gc).astype(f)
    s = (1 / (1 + np.exp(-rng.normal(0, 1.5, (n, 2))))).astype(f)
    pc = (s + ij).astype(f)
    pwh = (aw * np.exp(rng.normal(0, 0.5, (n, 2)))).astype(f)
    near = rng.rand(n) < 0.3
    pc[near] = (gc[near] + rng.normal(0, 0.05, (near.sum(), 2)) * gwh[near]).astype(f)
    pwh[near] = (gwh[near] * np.exp(rng.normal(0, 0.05, (near.sum(), 2)))).astype(f)
    pwh[small] = (gwh[small] * np.exp(rng.normal(0, 0.5, (small.sum(), 2)))).astype(f)
    s = np.clip(pc - np.floor(pc), 1e-3, 1 - 1e-3).astype(f)
    return np.concatenate([pc, pwh], 1), np.concatenate([gc, gwh], 1), s


@pytest.mark.parametrize("kind", spec.KINDS)
def test_fp32_model_within_the_bound_over_a_million_pairs(kind):
    for seed in range(4):
        p, g, s = _draw_608(250000, 100 + seed)
        L64, d64 = spec.box_loss(kind, p, g)
        L32, _ = spec.box_loss_fp32(kind, p, g)
        for norm in (1.0, 0.07):
            ok = spec.within_bound(spec.raw_grad_fp32(kind, p, g, s, norm), norm * spec.raw_chain(d64, p, s), norm)
            assert ok.all(), "%s seed %d n %r: %d entries outside the bound" % (kind, seed, norm, (~ok).sum())
        assert np.max(np.abs(L32 - L64)) < 1e-6


@pytest.mark.parametrize("kind", spec.KINDS)
def test_fp32_model_on_exact_ties_and_special_values(kind):
    f = np.float32
    p = np.array([[3.25, 7.5, 1.25, 0.5], [0.0, 0.0, 0.0, 0.0], [1.0, 1.0, np.inf, 1.0], [np.nan, 1.0, 1.0, 1.0],
                  [1.5, 1.0, 2.0, 1.0]], f)
    g = np.array([[3.25, 7.5, 1.25, 0.5], [0.5, 0.5, 1.0, 1.0], [1.0, 1.0, 1.0, 1.0], [1.0, 1.0, 1.0, 1.0],
                  [1.0, 1.0, 1.0, 1.0]], f)
    s = np.full((len(p), 2), 0.5, f)
    L64, d64 = spec.box_loss(kind, p, g)
    L32, _ = spec.box_loss_fp32(kind, p, g)
    assert np.array_equal(np.isnan(L32), np.isnan(L64))
    fin = np.isfinite(L64)
    np.testing.assert_allclose(L32[fin], L64[fin], rtol=1e-5, atol=1e-6)
    r64 = spec.raw_chain(d64, p, s)
    r32 = spec.raw_grad_fp32(kind, p, g, s)
    rows = np.isfinite(r64).all(1) | np.isnan(L64)
    assert spec.within_bound(r32[rows], r64[rows]).all()


# ------------------------------------------------------------------------------------------------ argument validation
def _cfg():
    import yolov4_b200 as yb
    return {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": 80}


@pytest.mark.parametrize("kw, exc", [
    (dict(iou_loss="CIoU"), ValueError), (dict(iou_loss="iou"), ValueError), (dict(iou_loss=1), ValueError),
    (dict(iou_loss="ciou", iou_normalizer=True), TypeError), (dict(iou_loss="ciou", iou_normalizer="0.07"), TypeError),
    (dict(iou_loss="ciou", iou_normalizer=float("nan")), ValueError),
    (dict(iou_loss="ciou", iou_normalizer=float("inf")), ValueError), (dict(iou_loss="ciou", iou_normalizer=-0.5), ValueError),
    (dict(iou_loss="ciou", iou_normalizer=1e39), ValueError), (dict(iou_normalizer=0.07), ValueError),
])
def test_python_validation_before_cuda_work(kw, exc):
    from yolov4_b200.yololoss import fused_yolo_loss, fused_yolo_loss_components
    heads = [torch.zeros(1, 255, F, F) for F in (8, 4, 2)]         # CPU heads: only the keyword check may raise first
    labels = torch.zeros(1, 60, 5, dtype=torch.float64)
    with pytest.raises(exc):
        fused_yolo_loss(heads, labels, _cfg(), **kw)
    with pytest.raises(exc):
        fused_yolo_loss_components(heads, labels, _cfg(), **kw)


P = 4096        # non-null dummy pointers, never dereferenced: only iou_loss / iou_normalizer can be refused


@pytest.mark.parametrize("iou, norm", [(4, 1.0), (-1, 1.0), (3, -1.0), (3, float("nan")), (3, float("inf")), (1, -1e-30)])
@pytest.mark.parametrize("chained", [0, 1])
def test_c_entry_rejects_bad_iou_arguments(iou, norm, chained):
    from yolov4_b200 import _cabi
    import yolov4_b200 as yb
    anch = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
    L = _cabi.lib()
    for code in (0, 1, 2):
        assert L.yl_loss_forward_ex(P, code, P, 2, 76, 60, 80, 0, anch, _cabi.ints(yb.ANCHOR_MASK[0]), 0.7, iou, norm, chained,
                                    P, P, P, P, P, P, None) == 1
    assert L.yl_loss_forward_ex(None, 0, P, 2, 76, 60, 80, 0, anch, _cabi.ints(yb.ANCHOR_MASK[0]), 0.7, 3, 0.07, chained,
                                P, P, P, P, P, P, None) == 1

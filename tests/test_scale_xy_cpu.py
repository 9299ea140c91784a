"""CPU checks of the grid-sensitivity decode (`scale_x_y=`, tests/scale_xy_spec.py): the spec reduces to the plain decode at
s = 1 and to 2 sigmoid - 0.5 + cell at s = 2, beta is darknet's float64 expression, the fp32 model of the scaled IoU gradient
stays within the stated bound, and every Python and C entry rejects a bad scale before any CUDA work."""
import numpy as np
import pytest
import torch

import iou_loss_spec
import scale_xy_spec as spec
from oracle import oracle as orc

f32 = np.float32
YOLOV4_CFG = (1.2, 1.1, 1.05)


def _raws(B=2, C=5, Fs=(8, 4, 2), seed=0):
    rng = np.random.RandomState(seed)
    return [rng.normal(0, 2.5, (B, 3 * (5 + C), F, F)).astype(f32) for F in Fs]


def test_scale_one_is_the_plain_decode_bit_for_bit():
    raws = _raws()
    for l, r in enumerate(raws):
        for s in (1.0, f32(1.0)):
            assert spec.decode_eval(r, l, 5, s).tobytes() == orc.decode_eval(r, l, 5).tobytes()
            o, p = spec.decode_train(r, l, 5, s)
            o0, p0 = orc.decode_train(r, l, 5)
            assert o.tobytes() == np.ascontiguousarray(o0).tobytes() and np.array_equal(p, p0)


def test_scale_one_loss_spec_is_the_iou_loss_spec():
    from loss_edge_cases import heads
    from yolov4_b200.synth import synth_labels
    lab = synth_labels(2, 128, n_valid=12, seed=5).numpy().astype(f32)
    raws = heads(2, 128, 80, 7)
    for l in range(3):
        comps0, grad0, (cells0, term0, graw0, p0) = iou_loss_spec.layer_spec(raws[l], lab, l, 80, 0.7, "ciou")
        comps, (cells, term, graw, p, _, _), gobj, _ = spec.layer_spec(raws[l], lab, l, 80, 0.7, "ciou", 1.0)
        assert np.array_equal(cells, cells0) and np.array_equal(p, p0)
        assert np.array_equal(term, term0, equal_nan=True) and np.array_equal(graw, graw0, equal_nan=True)
        np.testing.assert_allclose(comps, comps0, rtol=1e-6)
        F = raws[l].shape[2]
        g64 = grad0.reshape(2, 3, 85, F, F)[:, :, 4]
        np.testing.assert_allclose(gobj, g64, rtol=2e-6, atol=1e-12)


def test_scale_two_is_two_sigmoid_minus_half():
    t = np.concatenate([np.linspace(-20, 20, 4001), [0.0, -0.0, np.inf, -np.inf]]).astype(f32)
    sg = orc.sigmoidf(t)
    for cell in (0, 1, 37, 75):
        assert spec.beta(2.0) == f32(-0.5)
        got = spec.centre(t, cell, 2.0)
        want = ((f32(2) * sg).astype(f32) - f32(0.5)).astype(f32) + f32(cell)
        assert got.tobytes() == want.astype(f32).tobytes()
    assert spec.centre(f32(-np.inf), 7, 1.2) == spec.beta(1.2) + f32(7)     # sigmoid 0: the centre is beta + cell
    assert np.isnan(spec.centre(f32(np.nan), 7, 1.2))


def test_beta_is_darknets_float64_expression():
    rng = np.random.RandomState(1)
    sweep = np.concatenate([[0.5, 1.0, 1.05, 1.1, 1.2, 2.0, 1e-3, 3.0, 16.0], rng.uniform(0.01, 4, 2000)]).astype(f32)
    for s in sweep:
        want = f32(-0.5 * (np.float64(s) - 1.0))
        assert spec.beta(s).tobytes() == want.tobytes()
        if 0.5 <= s <= 2.0:                        # exact: -0.5 (s - 1) needs no more bits than s has
            assert np.float64(spec.beta(s)) == -0.5 * (np.float64(s) - 1.0)
    assert np.signbit(spec.beta(1.0))               # -0: sigmoid + beta is sigmoid for every sigmoid, +0 included


@pytest.mark.parametrize("kind", iou_loss_spec.KINDS)
@pytest.mark.parametrize("s", [1.05, 1.1, 1.2, 2.0])
def test_fp32_scaled_gradient_within_the_bound_over_a_million_pairs(kind, s):
    from test_iou_loss_cpu import _draw_608
    for seed in range(4):
        p, g, sg = _draw_608(250000, 100 + seed)
        ij = np.floor(p[:, :2]).astype(f32)
        p = p.copy()
        p[:, :2] = (((sg * f32(s)).astype(f32) + spec.beta(s)).astype(f32) + ij).astype(f32)     # the scaled centre of the cell
        _, d64 = iou_loss_spec.box_loss(kind, p, g)
        for norm in (1.0, 0.07):
            ok = iou_loss_spec.within_bound(spec.raw_grad_fp32(kind, p, g, sg, s, norm), norm * spec.raw_chain(d64, p, sg, s), norm)
            assert ok.all(), "%s s %r seed %d n %r: %d entries outside the bound" % (kind, s, seed, norm, (~ok).sum())


# ------------------------------------------------------------------------------------------------ argument validation
def _cfg():
    import yolov4_b200 as yb
    return {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": 80}


BAD = [(True, TypeError), ("1.2", TypeError), ((1.2, "1.1", 1.05), TypeError), ((1.2, True, 1.05), TypeError),
       (float("nan"), ValueError), (float("inf"), ValueError), (0.0, ValueError), (-1.2, ValueError), (1e39, ValueError),
       (1e-50, ValueError), ((1.2, 1.1), ValueError), ((1.2, 1.1, 1.05, 1.0), ValueError), ((1.2, float("nan"), 1.05), ValueError)]


@pytest.mark.parametrize("sxy, exc", BAD)
def test_python_validation_before_cuda_work(sxy, exc):
    import yolov4_b200 as yb
    from yolov4_b200.yololoss import fused_yolo_loss, fused_yolo_loss_components
    heads = [torch.zeros(1, 255, F, F) for F in (8, 4, 2)]         # CPU heads: only the keyword check may raise first
    labels = torch.zeros(1, 60, 5, dtype=torch.float64)
    with pytest.raises(exc):
        yb.detect_raw(heads, 80, 0.2, 0.5, scale_x_y=sxy)
    with pytest.raises(exc):
        yb.HeadPostprocessor(1, (8, 4, 2), 80, 0.2, 0.5, scale_x_y=sxy)
    with pytest.raises(exc):
        yb.decode_dense_cat(heads, _cfg(), scale_x_y=sxy)
    with pytest.raises(exc):
        fused_yolo_loss(heads, labels, _cfg(), iou_loss="ciou", scale_x_y=sxy)
    with pytest.raises(exc):
        fused_yolo_loss_components(heads, labels, _cfg(), iou_loss="ciou", scale_x_y=sxy)
    if not isinstance(sxy, tuple):
        with pytest.raises(exc):
            yb.YOLOLayer(_cfg(), 0, scale_x_y=sxy)


def test_yololayer_takes_one_number_and_keeps_an_empty_state_dict():
    import yolov4_b200 as yb
    with pytest.raises(TypeError):
        yb.YOLOLayer(_cfg(), 0, scale_x_y=YOLOV4_CFG)
    with pytest.raises(TypeError):
        yb.YOLOLayer(_cfg(), 0, None, 1.2)                          # keyword only: the reference's signature is unchanged
    m = yb.YOLOLayer(_cfg(), 0, scale_x_y=1.2)
    assert m.scale_x_y == float(f32(1.2)) and len(m.state_dict()) == 0 and not list(m.parameters())
    assert yb.YOLOLayer(_cfg(), 0).scale_x_y == 1.0


def test_yololayer_train_mode_with_a_scale_raises():
    import yolov4_b200 as yb
    m = yb.YOLOLayer(_cfg(), 0, scale_x_y=1.2).train()
    with pytest.raises(ValueError, match="fused_yolo_loss"):
        m(_FakeCuda())


class _FakeCuda:
    """Passes YOLOLayer's shape / device / dtype checks without a GPU; any CUDA work on it would fail."""
    shape = (1, 255, 8, 8)
    is_cuda = True
    dtype = torch.float32

    def dim(self):
        return 4


@pytest.mark.parametrize("sxy", [1.2, YOLOV4_CFG, 2.0])
def test_scale_needs_an_iou_box_term(sxy):
    from yolov4_b200.yololoss import fused_yolo_loss, fused_yolo_loss_components
    heads = [torch.zeros(1, 255, F, F) for F in (8, 4, 2)]
    labels = torch.zeros(1, 60, 5, dtype=torch.float64)
    with pytest.raises(ValueError, match="iou_loss"):
        fused_yolo_loss(heads, labels, _cfg(), scale_x_y=sxy)
    with pytest.raises(ValueError, match="iou_loss"):
        fused_yolo_loss_components(heads, labels, _cfg(), scale_x_y=sxy)


def test_all_ones_normalise_to_the_plain_decode():
    from yolov4_b200.postprocess import _check_scale_x_y
    for v in (None, 1, 1.0, (1, 1, 1), [1.0, 1.0, 1.0], np.float32(1)):
        assert _check_scale_x_y(v, 3) is None
    assert _check_scale_x_y(YOLOV4_CFG, 3) == [float(f32(v)) for v in YOLOV4_CFG]
    assert _check_scale_x_y(1.2, 2) == [float(f32(1.2))] * 2


P = 4096        # non-null dummy pointers, never dereferenced: only the scale can be refused
BAD_C = [float("nan"), float("inf"), -float("inf"), 0.0, -0.0, -1.2, -1e-30]


@pytest.mark.parametrize("s", BAD_C)
def test_c_entries_reject_bad_scales(s):
    from yolov4_b200 import _cabi
    import yolov4_b200 as yb
    L = _cabi.lib()
    anch = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
    mask = _cabi.ints([v for m in yb.ANCHOR_MASK for v in m])
    assert L.yl_decode_dense_ex(P, 1, 4, 80, anch, 8.0, s, P, 48, 0, None) == 1
    for pos in range(3):
        sc = [1.2, 1.1, 1.05]
        sc[pos] = s
        F, M = _cabi.ints([8, 4, 2]), 3 * (64 + 16 + 4)
        for dt in (0, 1, 2):
            assert L.yl_filter_raw_ex(_cabi.ptrs([P, P, P]), dt, F, 3, 1, 80, anch, mask, 0.2, _cabi.floats(sc), P, 1 << 40, M, 64,
                                      0, 1, 3, None) == 1
        assert L.yl_detect_host_ex3(None, _cabi.ptrs([P, P, P]), 0.2, 0.5, 0, 0, 0, _cabi.floats(sc), P, P) == 1
    for iou in (0, 1, 2, 3):
        for chained in (0, 1):
            assert L.yl_loss_forward_ex2(P, 0, P, 2, 76, 60, 80, 0, anch, _cabi.ints(yb.ANCHOR_MASK[0]), 0.7, iou, 1.0, s,
                                         chained, P, P, P, P, P, P, None) == 1


@pytest.mark.parametrize("s", [1.2, 2.0, 0.5, 1.0000001])
def test_c_loss_rejects_a_scale_without_an_iou_term(s):
    from yolov4_b200 import _cabi
    import yolov4_b200 as yb
    L = _cabi.lib()
    anch = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
    for dt in (0, 1, 2):
        assert L.yl_loss_forward_ex2(P, dt, P, 2, 76, 60, 80, 0, anch, _cabi.ints(yb.ANCHOR_MASK[0]), 0.7, 0, 1.0, s, 0,
                                     P, P, P, P, P, P, None) == 1

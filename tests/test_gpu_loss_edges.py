"""The fused training loss and build_target against the CPU oracle on hostile labels (tests/loss_edge_cases.py): negative and
fractional class ids (5 + cls indexes the target row with Python's negative-index wrap), more than 32 GTs on one cell,
collisions across the kernels' slices, K = 256, zero and non-positive rows among the first n, cell edges, degenerate extents,
exact ignore-test boundaries, class counts around the 32-lane stride, another anchor mask, special logits, upstream gradients
and head layouts.

  fused loss      per layer, the four components within 1e-5 relative of orc.yolo_loss_layer; the gradient of the three-scale
                  loss within 2e-5 relative with the same support; NaN where the oracle has NaN; status 0
  unfused path    YOLOLoss.forward (build_targets3 + torch) gives the oracle's value where the reference's BCE accepts its inputs
  build_target    per layer and with build_targets3, bit for bit the oracle's masks and targets, on two runs
  invalid labels  a matched class id outside [-(10+C), C) or a centre outside the grid sets status and makes
                  build_target(strict=True) raise IndexError, in exactly the layers where the reference raises
"""
import functools

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import loss_edge_cases as cases                                        # noqa: E402
from oracle import oracle as orc                                      # noqa: E402  (checker only)
import yolov4_b200 as yb                                               # noqa: E402
from yolov4_b200 import _cabi                                          # noqa: E402
from yolov4_b200.yololoss import fused_yolo_loss, fused_yolo_loss_components   # noqa: E402

VALID = sorted(cases.VALID)


def cfg_of(c):
    return {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": c["mask"], "N_CLASSES": c["C"]}


def cuda_heads(c, requires_grad=False):
    return [torch.from_numpy(r).cuda().requires_grad_(requires_grad) for r in c["raws"]]


@functools.lru_cache(maxsize=None)
def oracle_loss(name, thr):
    """Per layer: (components float64[4], gradient of their sum w.r.t. the raw head, float64)."""
    c = cases.get(name)
    return [orc.yolo_loss_layer(c["raws"][l], c["labels"], l, c["C"], thr, mask=c["mask"]) for l in range(3)]


def assert_close(got, want, rel, atol, what):
    """NaN where want is NaN, the same infinities, finite values within rel * |want| + atol."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert got.shape == want.shape, what
    assert np.array_equal(np.isnan(got), np.isnan(want)), "%s: NaN positions differ" % what
    inf = np.isinf(want)
    assert np.array_equal(np.isinf(got), inf) and np.array_equal(got[inf], want[inf]), "%s: infinities differ" % what
    fin = np.isfinite(want)
    err = np.abs(got[fin] - want[fin])
    bad = err > rel * np.abs(want[fin]) + atol
    assert not bad.any(), "%s: %d values differ, worst %r vs %r" % (what, bad.sum(), got[fin][bad][0], want[fin][bad][0])


def support(g):
    """Where a gradient is nonzero: NaN counts, magnitudes below the smallest normal fp32 do not (the oracle's float64
    gradient keeps products that fp32 arithmetic rounds to zero)."""
    return ~(np.abs(g) < np.finfo(np.float32).tiny)


def bit_equal(a, b):
    """Bitwise equality of two fp32 arrays / tensors, except that any NaN equals any NaN."""
    a = a.detach().contiguous().cpu().numpy() if isinstance(a, torch.Tensor) else np.ascontiguousarray(a, np.float32)
    b = b.detach().contiguous().cpu().numpy() if isinstance(b, torch.Tensor) else np.ascontiguousarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(a.view(np.uint32)[~na], b.view(np.uint32)[~nb])


def fused_grads(c, thr, up=1.0, heads=None):
    hs = [h.detach().clone().requires_grad_(True) for h in (heads or cuda_heads(c))]
    loss = fused_yolo_loss(hs, torch.from_numpy(c["labels"]).cuda(), cfg_of(c), thr)
    loss.backward(torch.tensor(up, dtype=torch.float32, device="cuda"))
    return loss.detach(), [h.grad for h in hs]


def forward_status(c, thr, heads=None):
    """The typed C forward of the three scales with a status buffer: (loss4, status)."""
    L = _cabi.lib()
    hs = heads or cuda_heads(c)
    code = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}[hs[0].dtype]
    lab = torch.from_numpy(c["labels"]).cuda()
    B, K, C = int(lab.shape[0]), int(lab.shape[1]), c["C"]
    loss4 = torch.zeros(4, dtype=torch.float64, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    anch = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
    keep = []
    for l, r in enumerate(hs):
        F = int(r.shape[2])
        bufs = (torch.empty((B, 3, F, F), device="cuda"), torch.empty((B, K), dtype=torch.int32, device="cuda"),
                torch.empty((B, K), dtype=torch.int32, device="cuda"), torch.empty((B, K, 4 + C), device="cuda"))
        keep.append(bufs)
        fn = L.yl_loss_forward_typed if l == 0 else L.yl_loss_forward_chained_typed
        _cabi.check(fn(r.data_ptr(), code, lab.data_ptr(), B, F, K, C, l, anch, _cabi.ints(c["mask"][l]), float(np.float32(thr)),
                       loss4.data_ptr(), bufs[0].data_ptr(), bufs[1].data_ptr(), bufs[2].data_ptr(), bufs[3].data_ptr(),
                       status.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return loss4, int(status.item())


# ------------------------------------------------------------------------------------------------ fused loss vs the oracle
@pytest.mark.parametrize("name", VALID)
def test_fused_loss_vs_oracle(name):
    c = cases.get(name)
    lab = torch.from_numpy(c["labels"]).cuda()
    heads = cuda_heads(c)
    for thr in c["thrs"]:
        want = oracle_loss(name, thr)
        for l in range(3):
            got = fused_yolo_loss_components([heads[l]], lab, cfg_of(c), thr, layers=[l]).cpu().numpy()
            assert_close(got, want[l][0], 1e-5, 1e-6, "%s thr %r layer %d components" % (name, thr, l))
        loss, grads = fused_grads(c, thr)
        total = sum(w[0].sum() for w in want)
        assert_close(loss.item(), total, 1e-5, 1e-6, "%s thr %r loss" % (name, thr))
        for l, g in enumerate(grads):
            g = g.cpu().numpy()
            assert np.array_equal(support(g), support(want[l][1])), "%s thr %r layer %d: gradient support differs" % (name, thr, l)
            assert_close(g, want[l][1], 2e-5, 1e-7, "%s thr %r layer %d gradient" % (name, thr, l))
        assert forward_status(c, thr, heads)[1] == 0, "%s: status set on labels the reference accepts" % name


def _bce_args_in_unit_interval(c, thr):
    """Whether every input and target of the reference's three BCE terms lies in [0, 1] (ATen asserts on the device
    otherwise), from the oracle's masks and targets."""
    C, nch = c["C"], 5 + c["C"]
    for l in range(3):
        out, pred = orc.decode_train(c["raws"][l], l, C, mask=c["mask"])
        target, obj_mask, tgt_mask, _ = orc.build_target(pred, c["labels"], l, C, thr, mask=c["mask"])
        sel = np.r_[0:2, 5:nch]
        m = np.concatenate([tgt_mask[..., 0:2], tgt_mask[..., 4:]], -1)
        for v in (out[..., sel] * m, target[..., sel] * m, out[..., 4] * obj_mask, target[..., 4] * obj_mask):
            if not ((v >= 0) & (v <= 1)).all():
                return False
    return True


@pytest.mark.parametrize("name", cases.UNFUSED)
def test_unfused_path_matches_the_oracle(name):
    c = cases.get(name)
    cfg = cfg_of(c)
    heads = cuda_heads(c)
    for thr in c["thrs"]:
        assert _bce_args_in_unit_interval(c, thr), "%s: the reference's BCE would reject this set" % name
        outs = [yb.YOLOLayer(cfg, l, device="cuda").train()(heads[l]) for l in range(3)]
        loss = yb.YOLOLoss(cfg, thr, device="cuda")(outs, {"padded_labels": torch.from_numpy(c["labels"]).double()})
        want = sum(w[0].sum() for w in oracle_loss(name, thr))
        assert_close(loss.item(), want, 1e-5, 1e-6, "%s thr %r unfused loss" % (name, thr))


# ------------------------------------------------------------------------------------------------ build_target vs the oracle
@pytest.mark.parametrize("name", VALID)
def test_build_target_bit_exact_on_two_runs(name):
    c = cases.get(name)
    C, mask = c["C"], c["mask"]
    lab = torch.from_numpy(c["labels"]).cuda()
    preds = [orc.decode_train(c["raws"][l], l, C, mask=mask)[1] for l in range(3)]
    preds_t = [torch.from_numpy(np.ascontiguousarray(p)).cuda() for p in preds]
    outs = [torch.empty(p.shape[:4] + (5 + C,), device="cuda") for p in preds]
    for thr in c["thrs"]:
        want = [orc.build_target(preds[l], c["labels"], l, C, thr, mask=mask) for l in range(3)]
        for run in range(2):
            for l in range(3):
                got = yb.build_target(outs[l], preds_t[l], l, lab, yb.ANCHORS_PX, mask, thr, C, strict=True)
                for what, g, w in zip(("target", "obj_mask", "tgt_mask", "tgt_scale"), got, want[l]):
                    assert bit_equal(g, w), "%s thr %r run %d layer %d: build_target %s" % (name, thr, run, l, what)
            got3 = yb.build_targets3(outs, preds_t, [0, 1, 2], lab, yb.ANCHORS_PX, mask, thr, C)
            for l in range(3):
                for what, g, w in zip(("target", "obj_mask", "tgt_mask", "tgt_scale"), got3[l], want[l]):
                    assert bit_equal(g, w), "%s thr %r run %d layer %d: build_targets3 %s" % (name, thr, run, l, what)


# ------------------------------------------------------------------------------------------------ labels the reference rejects
@pytest.mark.parametrize("name", sorted(cases.ERROR))
def test_invalid_index_sets_status_and_strict_raises(name):
    c = cases.get(name)
    C = c["C"]
    assert forward_status(c, 0.7)[1] == 1, "%s: the fused loss must set status" % name
    lab = torch.from_numpy(c["labels"]).cuda()
    raised = []
    for l in range(3):
        pred = orc.decode_train(c["raws"][l], l, C)[1]
        try:
            want = orc.build_target(pred, c["labels"], l, C, 0.7)
        except IndexError:
            want = None
        raised.append(want is None)
        pred_t = torch.from_numpy(np.ascontiguousarray(pred)).cuda()
        out = torch.empty(pred.shape[:4] + (5 + C,), device="cuda")
        if want is None:
            with pytest.raises(IndexError):
                yb.build_target(out, pred_t, l, lab, yb.ANCHORS_PX, c["mask"], 0.7, C, strict=True)
        else:
            got = yb.build_target(out, pred_t, l, lab, yb.ANCHORS_PX, c["mask"], 0.7, C, strict=True)
            assert all(bit_equal(g, w) for g, w in zip(got, want)), (name, l)
    assert any(raised)


def test_k257_raises_before_any_kernel():
    """K = 257 label slots (TG_MAXK + 1): both paths refuse the call before they launch anything; the C entry points leave
    their output buffers untouched."""
    C = 4
    c = cases.get("bad_class_4")
    heads = cuda_heads(c)
    lab = torch.zeros(1, 257, 5, device="cuda")
    lab[0, :3] = torch.from_numpy(c["labels"][0, :3]).cuda()
    lab[0, 0, 4] = 1.0
    cfg = cfg_of(c)
    with pytest.raises(_cabi.YoloHeadError):
        fused_yolo_loss([h.clone().requires_grad_(True) for h in heads], lab, cfg, 0.7)
    with pytest.raises(_cabi.YoloHeadError):
        fused_yolo_loss_components(heads, lab, cfg, 0.7)
    outs = [yb.YOLOLayer(cfg, l, device="cuda").train()(heads[l]) for l in range(3)]
    with pytest.raises(_cabi.YoloHeadError):
        yb.build_target(outs[0]["output"], outs[0]["pred"], 0, lab, yb.ANCHORS_PX, yb.ANCHOR_MASK, 0.7, C)
    with pytest.raises(_cabi.YoloHeadError):
        yb.YOLOLoss(cfg, 0.7, device="cuda")(outs, {"padded_labels": lab})
    # the C entry points, with sentinels in every output
    L = _cabi.lib()
    torch.cuda.synchronize()
    F = int(heads[0].shape[2])
    loss4 = torch.full((4,), 7.0, dtype=torch.float64, device="cuda")
    gobj = torch.full((1, 3, F, F), 7.0, device="cuda")
    ints = [torch.full((1, 257), 7, dtype=torch.int32, device="cuda") for _ in range(2)]
    mgrad = torch.full((1, 257, 4 + C), 7.0, device="cuda")
    status = torch.full((1,), 5, dtype=torch.int32, device="cuda")
    anch = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
    rc = L.yl_loss_forward_typed(heads[0].data_ptr(), 0, lab.data_ptr(), 1, F, 257, C, 0, anch, _cabi.ints(yb.ANCHOR_MASK[0]), 0.7,
                                 loss4.data_ptr(), gobj.data_ptr(), ints[0].data_ptr(), ints[1].data_ptr(), mgrad.data_ptr(),
                                 status.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert rc != 0
    pred = outs[0]["pred"]
    tgt = [torch.full(s, 7.0, device="cuda") for s in ((1, 3, F, F, 5 + C), (1, 3, F, F), (1, 3, F, F, 4 + C), (1, 3, F, F, 2))]
    rc = L.yl_build_target(pred.data_ptr(), _cabi.longs(pred.stride()), lab.data_ptr(), 1, F, 257, C, 0, anch,
                           _cabi.ints(yb.ANCHOR_MASK[0]), 0.7, tgt[0].data_ptr(), tgt[1].data_ptr(), tgt[2].data_ptr(),
                           tgt[3].data_ptr(), status.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert rc != 0
    torch.cuda.synchronize()
    assert (loss4 == 7.0).all() and (gobj == 7.0).all() and (mgrad == 7.0).all() and int(status.item()) == 5
    assert all((t == 7).all() for t in ints) and all((t == 7.0).all() for t in tgt)


# ------------------------------------------------------------------------------------------------ ignore-test boundary
@pytest.mark.parametrize("contained", [False, True])
def test_ignore_boundary_shows_in_the_objectness_gradient(contained):
    """At thr = v (the fp32 IoU of the planted prediction and the GT) the cell is kept, at the float below v it is ignored;
    the objectness gradient of the cell (logit 6) is nonzero exactly when the cell is kept."""
    name = "ignore_boundary_%s" % ("contained" if contained else "overlap")
    c = cases.get(name)
    b, a, j, i = c["cell"]
    ch = a * (5 + c["C"]) + 4
    v = c["v"]
    for thr, kept in ((float(v), True), (float(np.nextafter(v, np.float32(-np.inf))), False)):
        assert (oracle_loss(name, thr)[0][1][b, ch, j, i] != 0) == kept
        _, grads = fused_grads(c, thr)
        assert (float(grads[0][b, ch, j, i]) != 0) == kept, (name, thr)


# ------------------------------------------------------------------------------------------------ upstream gradients
@pytest.mark.parametrize("up", [0.0, -3.5, 1e30])
def test_upstream_gradient(up):
    """grad = fp32(g * up): with up = 1e30 it overflows to +-inf exactly where |g * up| exceeds fp32 (a matched cell with
    tw = 1e9 on every layer); with up = 0 only NaN survives."""
    c = cases.big_wh_logit(cases.get("special_logits"))
    _, grads = fused_grads(c, 0.7, up)
    with np.errstate(over="ignore", invalid="ignore"):
        want = [(w[1] * up).astype(np.float32) for w in
                [orc.yolo_loss_layer(c["raws"][l], c["labels"], l, c["C"], 0.7) for l in range(3)]]
    for l, (g, w) in enumerate(zip(grads, want)):
        assert_close(g.cpu().numpy(), w, 2e-5, 1e-7 * abs(up), "up %r layer %d" % (up, l))
    if up == 1e30:
        assert all(np.isinf(w).any() for w in want)


# ------------------------------------------------------------------------------------------------ head layouts
def test_channels_last_and_sliced_heads_equal_contiguous():
    c = cases.get("class_ids")
    lab = torch.from_numpy(c["labels"]).cuda()
    cfg = cfg_of(c)
    heads = cuda_heads(c)
    base_loss, base_g = fused_grads(c, 0.7, heads=heads)
    base_c = fused_yolo_loss_components(heads, lab, cfg, 0.7).cpu().numpy()
    cl = [h.contiguous(memory_format=torch.channels_last) for h in heads]
    big = [torch.randn(h.shape[0], h.shape[1] + 9, h.shape[2], h.shape[3], device="cuda") for h in heads]
    for h, g in zip(heads, big):
        g[:, 4:4 + h.shape[1]] = h
    sliced = [g[:, 4:4 + h.shape[1]] for h, g in zip(heads, big)]
    for form, hs in (("channels_last", cl), ("sliced", sliced)):
        assert not any(h.is_contiguous() for h in hs)
        loss, gr = fused_grads(c, 0.7, heads=hs)
        np.testing.assert_allclose(loss.item(), base_loss.item(), rtol=1e-6)
        assert all(bit_equal(a, b) for a, b in zip(gr, base_g)), form
        np.testing.assert_allclose(fused_yolo_loss_components(hs, lab, cfg, 0.7).cpu().numpy(), base_c, rtol=1e-12, atol=0)
    two = fused_yolo_loss_components([heads[2], heads[0]], lab, cfg, 0.7, layers=[2, 0]).cpu().numpy()
    per = sum(fused_yolo_loss_components([heads[l]], lab, cfg, 0.7, layers=[l]).cpu().numpy() for l in (2, 0))
    np.testing.assert_allclose(two, per, rtol=1e-12, atol=0)


# ------------------------------------------------------------------------------------------------ 16-bit heads
def test_fp16_heads_with_negative_class_ids_match_widened_fp32():
    from test_gpu_half_loss import check_against_widened
    c = cases.get("class_ids")
    heads = [h.half() for h in cuda_heads(c)]
    check_against_widened(heads, torch.from_numpy(c["labels"]).cuda(), cfg_of(c), ups=(1.0, 65536.0))
    assert forward_status(c, 0.7, heads)[1] == 0

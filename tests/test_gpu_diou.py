"""DIoU-NMS on the GPU: every result equals the literal algorithm of diou_spec bit for bit, per class and agnostic, on every
entry point that takes the option."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import yolov4_b200 as yb                                              # noqa: E402
from yolov4_b200 import _cabi                                         # noqa: E402
from yolov4_b200.synth import synth_head_outputs                      # noqa: E402

import agnostic_spec                                                  # noqa: E402
import diou_spec as spec                                              # noqa: E402
from cap_spec import cap_detections                                   # noqa: E402
from oracle import oracle as orc                                      # noqa: E402  (checker only)
from test_gpu_half_inputs import assert_lists_bit_equal               # noqa: E402

CFG80 = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": 80}
SMALL_R, SMEM_R = 256, 1024                                           # k_segment_nms_bins / shared-memory big tier limits


def _fused(raws, C, conf, thr, **kw):
    return yb.detect_raw(raws, C, conf, thr, diou=True, **kw)


def _decoded(raws, C):
    return orc.decode_eval_cat([r.detach().float().cpu().numpy() for r in raws], C)


def iou_but_not_diou_pairs(pred, C, conf, thr):
    """Same-class candidate pairs with IoU >= thr > DIoU: the pairs on which the two rules can disagree."""
    cand = agnostic_spec.candidates(pred, C, conf)
    ar = agnostic_spec.areas(cand["box"])
    n = 0
    for c in np.unique(cand["cls"]):
        idx = np.nonzero(cand["cls"] == c)[0]
        bx, a = cand["box"][idx], ar[idx]
        for i in range(1, len(idx)):
            iou = agnostic_spec.iou_ge(bx[i], a[i], bx[:i], a[:i], thr)
            n += int((iou & ~spec.diou_ge(bx[i], a[i], bx[:i], a[:i], thr)).sum())
    return n


def check_oracle_free(rows_list, pred_list, C, conf, thr):
    """Two checks that do not use the spec's greedy pass (per class): no two kept rows of a class reach DIoU >= thr, and every
    candidate that was not kept reaches DIoU >= thr with an earlier kept candidate of its class."""
    for rows, pred in zip(rows_list, pred_list):
        cand = agnostic_spec.candidates(pred, C, conf)
        if rows is None:
            assert len(cand["s"]) == 0
            continue
        rows = np.asarray(rows.cpu().numpy() if hasattr(rows, "cpu") else rows, np.float32)
        n = len(cand["s"])
        allr = agnostic_spec.rows_of(cand, np.arange(n))
        cls_sorted = np.lexsort((-cand["row"], -cand["s"], cand["cls"]))
        key = {allr[j].tobytes(): j for j in range(n)}
        kept_idx = np.array([cls_sorted[key[r.tobytes()]] for r in rows], np.int64)
        kept = np.zeros(n, bool)
        kept[kept_idx] = True
        order = agnostic_spec.image_order(cand)
        pos = np.empty(n, np.int64)
        pos[order] = np.arange(n)
        ar = agnostic_spec.areas(cand["box"])
        for i in range(n):
            earlier = (cand["cls"] == cand["cls"][i]) & kept & (pos < pos[i])
            hit = spec.diou_ge(cand["box"][i], ar[i], cand["box"][earlier], ar[earlier], thr).any()
            assert hit != kept[i], "a kept row reaches DIoU >= thr with an earlier kept row" if kept[i] else \
                "a dropped candidate has no suppressor"


# i.i.d. boxes at conf 0.2 do not overlap within a class enough for the two rules to disagree: there, DIoU equals IoU
@pytest.mark.parametrize("clustered,conf,nmst,differs", [(False, 1e-4, 0.4, True), (True, 1e-4, 0.4, True),
                                                          (False, 0.2, 0.5, False), (True, 0.2, 0.5, True)])
def test_fused_608(clustered, conf, nmst, differs):
    raws = synth_head_outputs(2, 608, 80, seed=0, device="cuda", clustered=clustered)
    got = _fused(raws, 80, conf, nmst)
    assert_lists_bit_equal(got, spec.detect(raws, 80, conf, nmst), what=f"608 clustered={clustered} conf {conf}")
    dense = _decoded(raws, 80)
    assert (iou_but_not_diou_pairs(dense[0], 80, conf, nmst) > 0) == differs
    iou = yb.detect_raw(raws, 80, conf, nmst)
    same = all((g is None and w is None) or (g is not None and w is not None and torch.equal(g, w)) for g, w in zip(got, iou))
    assert same != differs
    if differs:
        assert sum(len(g) for g in got) > sum(len(w) for w in iou), "DIoU-NMS keeps more rows than IoU-NMS"
    check_oracle_free(got[:1], dense[:1], 80, conf, nmst)


@pytest.mark.parametrize("img,C,B", [(416, 80, 2), (96, 4, 3), (64, 128, 2)])
def test_fused_other_shapes(img, C, B):
    raws = synth_head_outputs(B, img, C, seed=img + C, device="cuda", fg_prob=0.05, clustered=True)
    for conf, nmst in ((1e-3, 0.45), (0.2, 0.5)):
        assert_lists_bit_equal(_fused(raws, C, conf, nmst), spec.detect(raws, C, conf, nmst), what=f"{img} C {C} conf {conf}")
    assert_lists_bit_equal(_fused(raws, C, 0.2, 0.5, agnostic=True), spec.detect(raws, C, 0.2, 0.5, agnostic=True),
                           what=f"{img} C {C} agnostic")


def _dense(raws):
    return torch.cat([yb.YOLOLayer(CFG80, l, device="cuda").eval()(r) for l, r in enumerate(raws)], 1)


@pytest.mark.parametrize("conf,nmst", [(1e-4, 0.4), (0.2, 0.5)])
def test_dense_postprocess_608(conf, nmst):
    raws = synth_head_outputs(2, 608, 80, seed=5, device="cuda", clustered=True, fg_prob=0.02)
    dense = _dense(raws)
    got = yb.postprocess(dense, 80, conf, nmst, diou=True)
    assert_lists_bit_equal(got, spec.postprocess(dense.cpu().numpy(), 80, conf, nmst), what=f"dense conf {conf}")


def _pathological():
    """The inputs of the parity suite's pathological-values test (NaN / inf / negative / duplicates)."""
    rng = np.random.RandomState(5)
    B, M, C = 2, 600, 6
    pred = np.zeros((B, M, 5 + C), np.float32)
    pred[..., 0:2] = rng.rand(B, M, 2) * 100
    pred[..., 2:4] = rng.rand(B, M, 2) * 40
    pred[..., 4] = rng.rand(B, M)
    pred[..., 5:] = rng.rand(B, M, C) ** 3
    pred[0, 0:20, 2:4] = 0.0
    pred[0, 5:10, 0:2] = pred[0, 0:5, 0:2]
    pred[0, 30, 0] = np.nan
    pred[0, 31, 2] = np.inf
    pred[0, 32, 7] = np.nan
    pred[1, 40, 4] = np.nan
    pred[1, 41, 4] = -0.5
    pred[1, 50:60, :] = pred[1, 60:70, :]
    pred[1, 70:75, 4] = -2.0                                   # negative obj x negative cls: a positive score
    pred[1, 70:75, 5:] = -0.75
    return pred


@pytest.mark.parametrize("agnostic", [False, True])
def test_dense_postprocess_pathological_values(agnostic):
    pred = _pathological()
    gpu = torch.from_numpy(pred).cuda()
    for nmst in (0.45, 1e-4, 0.0, -0.5, 1.0, 1.5):
        got = yb.postprocess(gpu, 6, 0.05, nmst, agnostic=agnostic, diou=True)
        assert_lists_bit_equal(got, spec.postprocess(pred, 6, 0.05, nmst, agnostic), what=f"pathological nms {nmst} agnostic {agnostic}")


def test_big_tier_shared_memory():
    """416, 4 classes at conf 0.05: every segment holds 256 < n <= 1024 candidates, so all go to k_segment_nms_big's
    shared-memory form (thr > 0: positive-threshold decision; thr <= 0: literal decision)."""
    raws = synth_head_outputs(1, 416, 4, seed=7, device="cuda", fg_prob=0.05, clustered=True)
    cand = agnostic_spec.candidates(_decoded(raws, 4)[0], 4, 0.05)
    counts = np.bincount(cand["cls"], minlength=4)
    assert counts.min() > SMALL_R and counts.max() <= SMEM_R
    for nmst in (0.45, 0.0):
        assert_lists_bit_equal(_fused(raws, 4, 0.05, nmst), spec.detect(raws, 4, 0.05, nmst), what=f"big tier thr {nmst}")


def test_big_tier_global_memory():
    """All-zero logits on 20 / 10 / 5 grids, 2 classes: 1575 candidates per class, all tied at 0.25, so every segment takes the
    in-place global-memory form."""
    raws = [torch.zeros(2, 21, f, f, device="cuda") for f in (20, 10, 5)]
    raws[0][1, 4] = -20.0                                      # image 1: anchor 0 of the stride-8 grid drops out
    cand = agnostic_spec.candidates(_decoded(raws, 2)[0], 2, 0.2)
    assert np.bincount(cand["cls"]).min() > SMEM_R
    for nmst in (0.5, 0.0):
        assert_lists_bit_equal(_fused(raws, 2, 0.2, nmst), spec.detect(raws, 2, 0.2, nmst), what=f"global form thr {nmst}")


def test_agnostic_608_and_survivors_beyond_shared_memory():
    raws = synth_head_outputs(2, 608, 80, seed=3, device="cuda", clustered=True)
    assert_lists_bit_equal(_fused(raws, 80, 1e-4, 0.4, agnostic=True), spec.detect(raws, 80, 1e-4, 0.4, agnostic=True),
                           what="agnostic 608")
    # 416 with 4 classes at conf 0: 10,647 distinct boxes, more than k_segment_nms_agnostic stages in shared memory
    raws = synth_head_outputs(1, 416, 4, seed=41, device="cuda")
    assert_lists_bit_equal(_fused(raws, 4, 0.0, 0.45, agnostic=True), spec.detect(raws, 4, 0.0, 0.45, agnostic=True),
                           what="agnostic global path")


@pytest.mark.parametrize("agnostic", [False, True])
def test_with_max_det(agnostic):
    raws = synth_head_outputs(3, 608, 80, seed=61, device="cuda", clustered=True, fg_prob=0.02)
    unc = _fused(raws, 80, 1e-4, 0.4, agnostic=agnostic)
    assert min(len(u) for u in unc) > 300
    for k in (1, 100, 300, 100000):
        assert_lists_bit_equal(_fused(raws, 80, 1e-4, 0.4, agnostic=agnostic, max_det=k), cap_detections(unc, k),
                               what=f"max_det {k}")


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_half_heads_equal_the_widened_fp32_result(dt):
    raws = [r.to(dt) for r in synth_head_outputs(2, 608, 80, seed=13, device="cuda", clustered=True)]
    wide = [r.float() for r in raws]
    for agn in (False, True):
        assert_lists_bit_equal(_fused(raws, 80, 1e-4, 0.4, agnostic=agn), _fused(wide, 80, 1e-4, 0.4, agnostic=agn),
                               what=f"{dt} agnostic {agn}")


@pytest.mark.parametrize("n_groups,dt", [(1, torch.float32), (2, torch.float32), (1, torch.float16), (2, torch.bfloat16)])
def test_head_postprocessor_run_and_replay(n_groups, dt):
    B = 4
    raws = [r.to(dt) for r in synth_head_outputs(B, 608, 80, seed=11, device="cuda", clustered=True)]
    want = _fused(raws, 80, 1e-4, 0.4)
    assert_lists_bit_equal(want, spec.detect([r.float() for r in raws], 80, 1e-4, 0.4), what="detect_raw")
    # clustered images at conf 1e-4 keep ~22.6k DIoU rows each, above the default cap_out of 16384
    hp = yb.HeadPostprocessor(B, [76, 38, 19], 80, 1e-4, 0.4, n_groups=n_groups, diou=True, cap_out=32768)
    hp.run(raws)
    torch.cuda.synchronize()
    assert_lists_bit_equal(hp.results(), want, what="run")
    hp.capture(raws)
    hp.meta.zero_()
    hp.replay()
    torch.cuda.synchronize()
    assert_lists_bit_equal(hp.results(), want, what="replay")
    fresh = [r.to(dt) for r in synth_head_outputs(B, 608, 80, seed=12, device="cuda", clustered=True)]
    for dst, src in zip(hp._captured_inputs, fresh):
        dst.copy_(src)
    hp.replay()
    torch.cuda.synchronize()
    assert_lists_bit_equal(hp.results(), _fused(fresh, 80, 1e-4, 0.4), what="replay, new inputs")
    ha = yb.HeadPostprocessor(B, [76, 38, 19], 80, 1e-4, 0.4, n_groups=n_groups, diou=True, agnostic=True, max_det=300)
    ha.run(fresh)
    torch.cuda.synchronize()
    assert_lists_bit_equal(ha.results(), _fused(fresh, 80, 1e-4, 0.4, agnostic=True, max_det=300), what="agnostic capped run")


def test_detect_host_ex2():
    L = _cabi.lib()
    B, C = 4, 80
    raws = synth_head_outputs(B, 416, C, seed=21, fg_prob=0.02, clustered=True)
    host = [r.numpy() for r in raws]
    gpu = [r.cuda() for r in raws]
    Fs = [r.shape[2] for r in raws]
    ctx = ctypes.c_void_p()
    cap_out = 32768
    anch = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
    mask = _cabi.ints([v for m in yb.ANCHOR_MASK for v in m])
    _cabi.check(L.yl_context_create(ctypes.byref(ctx), 0, B, _cabi.ints(Fs), 3, C, anch, mask, 1024, cap_out))
    try:
        rows = np.zeros((B, cap_out, 7), np.float32)
        counts = np.zeros((B,), np.int32)
        ptrs = _cabi.ptrs([h.ctypes.data for h in host])
        for bad in (-1, 2):
            assert L.yl_detect_host_ex2(ctx, ptrs, 0.001, 0.4, 0, 0, bad, rows.ctypes.data, counts.ctypes.data) == 1
        for conf, nmst, k, agn in ((0.001, 0.4, 0, 0), (0.2, 0.5, 0, 0), (0.001, 0.4, 100, 0), (0.001, 0.4, 0, 1)):
            for d in (1, 0):
                _cabi.check(L.yl_detect_host_ex2(ctx, ptrs, float(np.float32(conf)), float(np.float32(nmst)), k, agn, d,
                                                 rows.ctypes.data, counts.ctypes.data))
                want = yb.detect_raw(gpu, C, conf, nmst, max_det=k or None, agnostic=bool(agn), diou=bool(d))
                got = [rows[b, :counts[b]] if counts[b] else None for b in range(B)]
                assert_lists_bit_equal(got, want, what=f"host path conf {conf} max_det {k} agnostic {agn} diou {d}")
    finally:
        _cabi.check(L.yl_context_destroy(ctx))

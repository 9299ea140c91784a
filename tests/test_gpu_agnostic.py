"""Class-agnostic NMS on the GPU: every result equals the literal algorithm of agnostic_spec (greedy over all candidates, no
first-copy reduction) bit for bit, on every entry point that takes the option."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import yolov4_b200 as yb                                              # noqa: E402
from yolov4_b200 import _cabi                                         # noqa: E402
from yolov4_b200.synth import synth_head_outputs                      # noqa: E402

import agnostic_spec as spec                                          # noqa: E402
from cap_spec import cap_detections                                   # noqa: E402
from oracle import oracle as orc                                      # noqa: E402  (checker only)
from test_gpu_half_inputs import assert_lists_bit_equal               # noqa: E402

CFG80 = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": 80}
AGN_CAP = 4096                                                        # survivors k_segment_nms_agnostic stages in shared memory


def _iou_ge_matrix(a, b, thr):
    """Literal IoU(a_i, b_j) >= thr for all pairs (fp32, NaN-propagating)."""
    aa, ab = spec.areas(a), spec.areas(b)
    return np.stack([spec.iou_ge(a[i], aa[i], b, ab, thr) for i in range(len(a))]) if len(a) else np.zeros((0, len(b)), bool)


def check_oracle_free(rows_list, pred_list, C, conf, thr):
    """Two checks that do not use the spec's greedy pass: kept rows with valid boxes never overlap at IoU >= thr, and every
    candidate that was not kept overlaps an earlier kept candidate at IoU >= thr."""
    for rows, pred in zip(rows_list, pred_list):
        cand = spec.candidates(pred, C, conf)
        if rows is None:
            assert len(cand["s"]) == 0
            continue
        rows = np.asarray(rows.cpu().numpy() if hasattr(rows, "cpu") else rows, np.float32)
        box = rows[:, :4]
        valid = (box[:, 0] < box[:, 2]) & (box[:, 1] < box[:, 3])
        m = _iou_ge_matrix(box[valid], box[valid], thr)
        np.fill_diagonal(m, False)
        assert not m.any(), "two kept rows overlap at IoU >= thr"
        # the kept candidates, identified by their row bytes (rows_of lists candidate cls_sorted[j] as row j)
        n = len(cand["s"])
        allr = spec.rows_of(cand, np.arange(n))
        cls_sorted = np.lexsort((-cand["row"], -cand["s"], cand["cls"]))
        key = {allr[j].tobytes(): j for j in range(n)}
        order = spec.image_order(cand)
        pos_in_order = np.empty(len(order), np.int64)
        pos_in_order[order] = np.arange(len(order))
        kept_idx = np.array([cls_sorted[key[r.tobytes()]] for r in rows], np.int64)
        kept = np.zeros(len(order), bool)
        kept[kept_idx] = True
        kb, kp = cand["box"][kept_idx], pos_in_order[kept_idx]
        ka = spec.areas(kb)
        ca = spec.areas(cand["box"])
        for i in np.nonzero(~kept)[0]:
            earlier = kp < pos_in_order[i]
            assert spec.iou_ge(cand["box"][i], ca[i], kb[earlier], ka[earlier], thr).any(), "a dropped candidate has no suppressor"


def _fused(raws, C, conf, thr, **kw):
    return yb.detect_raw(raws, C, conf, thr, agnostic=True, **kw)


@pytest.mark.parametrize("clustered,conf,nmst", [(False, 1e-4, 0.4), (True, 1e-4, 0.4), (False, 0.2, 0.5), (True, 0.2, 0.5)])
def test_fused_608(clustered, conf, nmst):
    raws = synth_head_outputs(2, 608, 80, seed=0, device="cuda", clustered=clustered)
    got = _fused(raws, 80, conf, nmst)
    want = spec.detect(raws, 80, conf, nmst)
    assert_lists_bit_equal(got, want, what=f"608 clustered={clustered} conf {conf}")
    dense = orc.decode_eval_cat([r.cpu().numpy() for r in raws], 80)
    check_oracle_free(got, dense, 80, conf, nmst)
    per_class = yb.detect_raw(raws, 80, conf, nmst)
    assert sum(len(g) for g in got) < sum(len(p) for p in per_class), "agnostic NMS keeps fewer rows than per-class NMS"


@pytest.mark.parametrize("img,C,B", [(416, 80, 2), (96, 4, 3), (64, 128, 2)])
def test_fused_other_shapes(img, C, B):
    raws = synth_head_outputs(B, img, C, seed=img + C, device="cuda", fg_prob=0.05, clustered=True)
    for conf, nmst in ((1e-3, 0.45), (0.2, 0.5)):
        assert_lists_bit_equal(_fused(raws, C, conf, nmst), spec.detect(raws, C, conf, nmst), what=f"{img} C {C} conf {conf}")


def _dense(raws):
    return torch.cat([yb.YOLOLayer(CFG80, l, device="cuda").eval()(r) for l, r in enumerate(raws)], 1)


@pytest.mark.parametrize("conf,nmst", [(1e-4, 0.4), (0.2, 0.5)])
def test_dense_postprocess_608(conf, nmst):
    raws = synth_head_outputs(2, 608, 80, seed=5, device="cuda", clustered=True, fg_prob=0.02)
    dense = _dense(raws)
    got = yb.postprocess(dense, 80, conf, nmst, agnostic=True)
    assert_lists_bit_equal(got, spec.postprocess(dense.cpu().numpy(), 80, conf, nmst), what=f"dense conf {conf}")


def test_dense_postprocess_pathological_values():
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
    gpu = torch.from_numpy(pred).cuda()
    for conf, nmst in ((0.05, 0.45), (0.3, 0.0001), (0.0, 0.5), (0.05, 0.0), (0.05, -0.5), (0.05, 1.0), (0.05, 1.5)):
        got = yb.postprocess(gpu, C, conf, nmst, agnostic=True)
        assert_lists_bit_equal(got, spec.postprocess(pred, C, conf, nmst), what=f"pathological conf {conf} nms {nmst}")


@pytest.mark.parametrize("nmst", [0.0, -0.25])
def test_threshold_le_zero(nmst):
    raws = synth_head_outputs(2, 96, 20, seed=31, device="cuda", fg_prob=0.05, clustered=True)
    got = _fused(raws, 20, 0.05, nmst)
    assert_lists_bit_equal(got, spec.detect(raws, 20, 0.05, nmst), what=f"thr {nmst}")


def test_all_ties_across_and_inside_classes():
    """All-zero logits: every score is exactly 0.25 and boxes repeat on every cell, so ties decide everything."""
    raws = [torch.zeros(2, 255, f, f, device="cuda") for f in (8, 4, 2)]
    raws[0][1, 4] = -20.0                                      # image 1: the stride-8 boxes drop out
    for nmst in (0.5, 0.0):
        got = _fused(raws, 80, 0.2, nmst)
        assert_lists_bit_equal(got, spec.detect(raws, 80, 0.2, nmst), what=f"all ties thr {nmst}")
        assert all(len(np.unique(g[:, :4].cpu().numpy(), axis=0)) == len(g) for g in got), "one label per box"


def test_survivors_beyond_shared_memory():
    """416 with 4 classes at conf 0: every one of the 10,647 boxes passes in every class, so the image has more distinct
    survivors than k_segment_nms_agnostic stages in shared memory and takes the global-memory path."""
    raws = synth_head_outputs(1, 416, 4, seed=41, device="cuda")
    cand = spec.candidates(orc.decode_eval_cat([r.cpu().numpy() for r in raws], 4)[0], 4, 0.0)
    assert len(cand["s"]) == 4 * 10647 and len(np.unique(cand["row"])) > AGN_CAP
    for nmst in (0.45, 0.0):
        got = _fused(raws, 4, 0.0, nmst)
        assert_lists_bit_equal(got, spec.detect(raws, 4, 0.0, nmst), what=f"global path thr {nmst}")


def test_one_class_equals_per_class():
    raws = synth_head_outputs(3, 416, 1, seed=51, device="cuda", fg_prob=0.05, clustered=True)
    for conf, nmst in ((1e-3, 0.45), (0.2, 0.5)):
        assert_lists_bit_equal(_fused(raws, 1, conf, nmst), yb.detect_raw(raws, 1, conf, nmst), what=f"C=1 conf {conf}")


def test_with_max_det():
    raws = synth_head_outputs(3, 608, 80, seed=61, device="cuda", clustered=True, fg_prob=0.02)
    unc = _fused(raws, 80, 1e-4, 0.4)
    assert min(len(u) for u in unc) > 300
    for k in (1, 100, 300, 100000):
        assert_lists_bit_equal(_fused(raws, 80, 1e-4, 0.4, max_det=k), cap_detections(unc, k), what=f"max_det {k}")


@pytest.mark.parametrize("n_groups,dt", [(1, torch.float32), (2, torch.float32), (1, torch.float16), (3, torch.bfloat16)])
def test_head_postprocessor_run_and_replay(n_groups, dt):
    B = 6
    raws = [r.to(dt) for r in synth_head_outputs(B, 608, 80, seed=11, device="cuda")]
    want = _fused(raws, 80, 1e-4, 0.4)
    assert_lists_bit_equal(want, spec.detect([r.float() for r in raws], 80, 1e-4, 0.4), what="detect_raw")
    hp = yb.HeadPostprocessor(B, [76, 38, 19], 80, 1e-4, 0.4, n_groups=n_groups, agnostic=True)
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
    # with a cap, uncapped counts the agnostic rows
    hk = yb.HeadPostprocessor(B, [76, 38, 19], 80, 1e-4, 0.4, n_groups=n_groups, agnostic=True, max_det=300)
    hk.run(fresh)
    torch.cuda.synchronize()
    assert_lists_bit_equal(hk.results(), _fused(fresh, 80, 1e-4, 0.4, max_det=300), what="capped run")
    assert torch.equal(hk.uncapped, hp.meta[:B])


@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
def test_detect_host_ex(dt):
    L = _cabi.lib()
    B, C = 5, 80
    raws = [r.to(dt) for r in synth_head_outputs(B, 416, C, seed=21, fg_prob=0.02, clustered=True)]
    if dt == torch.float32:
        host, code = [r.numpy() for r in raws], 0
    else:
        host, code = [r.view(torch.int16).numpy().view(np.uint16) for r in raws], 2
    gpu = [r.cuda() for r in raws]
    Fs = [r.shape[2] for r in raws]
    ctx = ctypes.c_void_p()
    cap_out = 32768                                               # per-class rows at conf 1e-3 exceed 24k
    anch = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
    mask = _cabi.ints([v for m in yb.ANCHOR_MASK for v in m])
    _cabi.check(L.yl_context_create_typed(ctypes.byref(ctx), 0, B, _cabi.ints(Fs), 3, C, code, anch, mask, 1024, cap_out))
    try:
        rows = np.zeros((B, cap_out, 7), np.float32)
        counts = np.zeros((B,), np.int32)
        ptrs = _cabi.ptrs([h.ctypes.data for h in host])
        for bad in (-1, 2):
            assert L.yl_detect_host_ex(ctx, ptrs, 0.001, 0.4, 0, bad, rows.ctypes.data, counts.ctypes.data) == 1
        for conf, nmst, k in ((0.001, 0.4, 0), (0.2, 0.5, 0), (0.001, 0.4, 100)):
            for agn in (1, 0, 1):                                  # the scratch is added on the first agnostic call
                _cabi.check(L.yl_detect_host_ex(ctx, ptrs, float(np.float32(conf)), float(np.float32(nmst)), k, agn,
                                                rows.ctypes.data, counts.ctypes.data))
                want = yb.detect_raw(gpu, C, conf, nmst, max_det=k or None, agnostic=bool(agn))
                got = [rows[b, :counts[b]] if counts[b] else None for b in range(B)]
                assert_lists_bit_equal(got, want, what=f"host path conf {conf} agnostic {agn} max_det {k}")
    finally:
        _cabi.check(L.yl_context_destroy(ctx))


def test_exchange_sized_by_the_output_single_rank():
    from yolov4_b200.sharded import DetectionExchange
    B = 4
    dev = torch.device("cuda", 0)
    hp = yb.HeadPostprocessor(B, [52, 26, 13], 80, 1e-3, 0.4, device=dev, agnostic=True)
    raws = synth_head_outputs(B, 416, 80, seed=71, device=dev, fg_prob=0.02, clustered=True)
    rows, meta = hp.run(raws)
    torch.cuda.synchronize()
    want = hp.results()
    cap = ((max(len(w) for w in want) + 3) // 4) * 4
    small = yb.HeadPostprocessor(B, [52, 26, 13], 80, 1e-3, 0.4, device=dev, agnostic=True, cap_out=cap)
    rows, meta = small.run(raws)
    ex = DetectionExchange(B, small.cap_out, dev, slots=2)
    try:
        ex.push(rows, meta[:B], 0)
        ex.wait(0)
        got = ex.results(0)
        torch.cuda.synchronize()
        assert_lists_bit_equal(got, want, what="exchange")
        ex.release(0)
        torch.cuda.synchronize()
        assert ex.status() == 0
    finally:
        ex.close()

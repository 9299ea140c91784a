"""YOLOv4's grid-sensitivity decode (`scale_x_y=`) on the B200 against tests/scale_xy_spec.py, with yolov4.cfg's scales
(1.2, 1.1, 1.05) and with s = 2:

  decode        YOLOLayer(..., scale_x_y=s) eval and decode_dense_cat bit for bit the spec at 76/38/19, odd grids, batch tails
  detection     detect_raw bit for bit the literal algorithm on the spec-decoded tensor: per class (orc.postprocess), agnostic,
                DIoU, max_det; dense (k_flag_tma) and sparse (k_flag_raw) thresholds; aligned and unaligned heads; 16-bit heads;
                clustered inputs on which the scale changes which pairs NMS suppresses.  HeadPostprocessor run / replay and
                yl_detect_host_ex3 equal detect_raw
  identity      None, 1.0 and (1, 1, 1) give the same bytes and launch the same kernels
  loss          giou / diou / ciou, fp32 and fp16: components, the objectness gradient plane bit for bit, the box gradient within
                iou_loss_spec's bound, graph replay, SGD on the box logits
  special       +-inf, NaN, +-0 on tx / ty give the spec's centres (beta + cell for sigmoid 0)
"""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import yolov4_b200 as yb                                              # noqa: E402
from yolov4_b200 import _cabi                                         # noqa: E402
from yolov4_b200.synth import synth_head_outputs                      # noqa: E402
from yolov4_b200.yololoss import fused_yolo_loss, fused_yolo_loss_components   # noqa: E402

import agnostic_spec                                                  # noqa: E402
import diou_spec                                                      # noqa: E402
import iou_loss_spec                                                  # noqa: E402
import scale_xy_spec as spec                                          # noqa: E402
from cap_spec import cap_detections                                   # noqa: E402
from oracle import oracle as orc                                      # noqa: E402  (checker only)
from test_gpu_half_inputs import assert_lists_bit_equal               # noqa: E402
from test_gpu_iou_loss import bit_equal, cfg_of, scene_608            # noqa: E402

CFG80 = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": 80}
YOLOV4 = (1.2, 1.1, 1.05)
SCALES = [YOLOV4, (2.0, 2.0, 2.0)]


def _np(raws):
    return [r.detach().float().cpu().numpy() for r in raws]


def _unaligned(r):
    buf = torch.empty(r.numel() + 1, dtype=r.dtype, device=r.device)
    u = buf[1:].view(r.shape)
    u.copy_(r)
    assert u.is_contiguous() and u.data_ptr() % 16 != 0
    return u


# ------------------------------------------------------------------------------------------------ decode
@pytest.mark.parametrize("sc", SCALES)
@pytest.mark.parametrize("B, Fs, C", [(2, (76, 38, 19), 80), (3, (13, 7, 5), 80), (5, (9, 5, 3), 20)])
def test_yololayer_and_decode_dense_cat_equal_the_spec(sc, B, Fs, C):
    rng = np.random.RandomState(B)
    raws = [torch.from_numpy(rng.normal(0, 3, (B, 3 * (5 + C), F, F)).astype(np.float32)).cuda() for F in Fs]
    cfg = dict(CFG80, N_CLASSES=C)
    want = spec.decode_eval_cat(_np(raws), C, sc)
    got = yb.decode_dense_cat(raws, cfg, scale_x_y=sc).cpu()
    assert bit_equal(got, torch.from_numpy(want))
    off = 0
    for l, r in enumerate(raws):
        layer = yb.YOLOLayer(cfg, l, scale_x_y=sc[l]).eval()
        n = 3 * Fs[l] ** 2
        assert bit_equal(layer(r).cpu(), torch.from_numpy(want[:, off:off + n]))
        off += n
    plain = orc.decode_eval_cat(_np(raws), C)
    assert not np.array_equal(plain[..., :2], want[..., :2]) and np.array_equal(plain[..., 2:], want[..., 2:])


# ------------------------------------------------------------------------------------------------ detection
def _literal(raws, C, conf, nmst, sc, agnostic=False, diou=False, max_det=None):
    pred = spec.decode_eval_cat(_np(raws), C, sc)
    if diou:
        rows = diou_spec.postprocess(pred, C, conf, nmst, agnostic=agnostic)
    elif agnostic:
        rows = agnostic_spec.postprocess(pred, C, conf, nmst)
    else:
        rows = orc.postprocess(pred, C, conf, nmst, nthreads=8)
    return cap_detections(rows, max_det) if max_det is not None else rows


@pytest.mark.parametrize("conf, nmst", [(1e-4, 0.4), (0.2, 0.5)])
@pytest.mark.parametrize("sc", SCALES)
def test_detect_raw_equals_the_literal_algorithm(sc, conf, nmst):
    raws = synth_head_outputs(2, 608, 80, seed=3, device="cuda")
    for kw in (dict(), dict(agnostic=True), dict(diou=True), dict(max_det=100)):
        got = yb.detect_raw(raws, 80, conf, nmst, scale_x_y=sc, **kw)
        assert_lists_bit_equal(got, _literal(raws, 80, conf, nmst, sc, **kw), what=f"{sc} {conf} {kw}")
        una = yb.detect_raw([_unaligned(r) for r in raws], 80, conf, nmst, scale_x_y=sc, **kw)
        assert_lists_bit_equal(una, got, what=f"unaligned {sc} {conf} {kw}")


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("conf, nmst", [(1e-4, 0.4), (0.2, 0.5)])
def test_16bit_heads_equal_the_widened_fp32_path(conf, nmst, dt):
    h16 = [r.to(dt) for r in synth_head_outputs(2, 608, 80, seed=5, device="cuda")]
    got = yb.detect_raw(h16, 80, conf, nmst, scale_x_y=YOLOV4)
    assert_lists_bit_equal(got, yb.detect_raw([h.float() for h in h16], 80, conf, nmst, scale_x_y=YOLOV4))


def _decisions(rows_list):
    """The kept (class, cls_conf, obj_conf) triples of every image: what NMS decided, whatever the boxes are."""
    return [None if r is None else sorted(map(tuple, np.asarray(r.cpu() if hasattr(r, "cpu") else r)[:, 4:7].tolist()))
            for r in rows_list]


@pytest.mark.parametrize("conf, nmst", [(1e-4, 0.4), (0.2, 0.5)])
def test_clustered_inputs_where_the_scale_changes_suppression(conf, nmst):
    raws = synth_head_outputs(2, 608, 80, seed=0, device="cuda", clustered=True)
    for kw in (dict(), dict(agnostic=True), dict(diou=True)):
        got = yb.detect_raw(raws, 80, conf, nmst, scale_x_y=YOLOV4, **kw)
        assert_lists_bit_equal(got, _literal(raws, 80, conf, nmst, YOLOV4, **kw), what=f"clustered {kw}")
        plain = yb.detect_raw(raws, 80, conf, nmst, **kw)
        assert _decisions(got) != _decisions(plain), "the scale changes no NMS decision here: %r" % (kw,)


def test_head_postprocessor_and_host_entry_equal_detect_raw():
    raws = synth_head_outputs(4, 608, 80, seed=7, device="cuda")
    want = yb.detect_raw(raws, 80, 1e-4, 0.4, scale_x_y=YOLOV4)
    hp = yb.HeadPostprocessor(4, [76, 38, 19], 80, 1e-4, 0.4, scale_x_y=YOLOV4)
    hp.run(raws)
    assert_lists_bit_equal(hp.results(), want, what="run")
    hp.capture(raws)
    hp.rows.zero_()
    hp.replay()
    torch.cuda.synchronize()
    assert_lists_bit_equal(hp.results(), want, what="replay")

    L = _cabi.lib()
    ctx = ctypes.c_void_p()
    cap_out = 16384
    _cabi.check(L.yl_context_create(ctypes.byref(ctx), torch.cuda.current_device(), 4, _cabi.ints([76, 38, 19]), 3, 80,
                                    _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh]),
                                    _cabi.ints([v for m in yb.ANCHOR_MASK for v in m]), 1024, cap_out))
    try:
        host = [r.cpu().contiguous() for r in raws]
        rows = np.zeros((4, cap_out, 7), np.float32)
        counts = np.zeros(4, np.int32)
        hp_ptrs = _cabi.ptrs([h.data_ptr() for h in host])
        _cabi.check(L.yl_detect_host_ex3(ctx, hp_ptrs, 1e-4, 0.4, 0, 0, 0, _cabi.floats(YOLOV4), rows.ctypes.data,
                                         counts.ctypes.data))
        assert_lists_bit_equal([rows[b, :counts[b]] if counts[b] else None for b in range(4)], want, what="yl_detect_host_ex3")
        for bad in (0.0, float("nan"), float("inf"), -1.0):
            assert L.yl_detect_host_ex3(ctx, hp_ptrs, 1e-4, 0.4, 0, 0, 0, _cabi.floats([1.2, bad, 1.05]), rows.ctypes.data,
                                        counts.ctypes.data) == 1
    finally:
        L.yl_context_destroy(ctx)


# ------------------------------------------------------------------------------------------------ identity at s = 1
def _kernel_names(fn):
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "emcpy" not in e.name
            and "emset" not in e.name]


def test_unit_scales_are_the_plain_path():
    raws = synth_head_outputs(2, 608, 80, seed=9, device="cuda")
    lab = torch.from_numpy(scene_608(seed=61, B=2)["labels"]).cuda()
    runs = {}
    for sxy in (None, 1.0, (1, 1, 1)):
        det = yb.detect_raw(raws, 80, 1e-4, 0.4, scale_x_y=sxy)
        dense = yb.decode_dense_cat(raws, CFG80, scale_x_y=sxy)
        comps = fused_yolo_loss_components(raws, lab, CFG80, iou_loss="ciou", scale_x_y=sxy)
        names = (_kernel_names(lambda: yb.detect_raw(raws, 80, 1e-4, 0.4, scale_x_y=sxy)),
                 _kernel_names(lambda: yb.decode_dense_cat(raws, CFG80, scale_x_y=sxy)),
                 _kernel_names(lambda: fused_yolo_loss_components(raws, lab, CFG80, iou_loss="ciou", scale_x_y=sxy)))
        runs[sxy] = (det, dense, comps, names)
    base = runs[None]
    assert any("k_emit_flagged" in n for n in base[3][0]) and any("k_loss_obj" in n for n in base[3][2])
    for sxy in (1.0, (1, 1, 1)):
        det, dense, comps, names = runs[sxy]
        assert_lists_bit_equal(det, base[0])
        assert bit_equal(dense, base[1]) and torch.equal(comps, base[2])
        assert names == base[3], sxy
    scaled = _kernel_names(lambda: yb.detect_raw(raws, 80, 1e-4, 0.4, scale_x_y=YOLOV4))
    assert len(scaled) == len(base[3][0]) and scaled != base[3][0]      # the same launches, the scaled emit kernel


# ------------------------------------------------------------------------------------------------ fused loss
def check_loss(c, kind, sc, dt=torch.float32):
    """Components, objectness plane (bit for bit) and box gradient (bound) of one scene against the spec; returns how many
    cells the scaled ignore test treats differently from the unscaled one."""
    C, thr = c["C"], c["thrs"][0]
    cfg = cfg_of(C)
    lab = torch.from_numpy(c["labels"]).cuda()
    heads = [torch.from_numpy(r).cuda().to(dt) for r in c["raws"]]
    wide = [h.float().cpu().numpy() for h in heads]
    kw = dict(iou_loss=kind, scale_x_y=sc)
    hs = [h.detach().clone().requires_grad_(True) for h in heads]
    fused_yolo_loss(hs, lab, cfg, thr, **kw).backward()
    nch = 5 + C
    n_ignore_diff = 0
    for l in range(3):
        comps, (cells, term, graw, p, _, _), gobj, obj_mask = spec.layer_spec(wide[l], c["labels"], l, C, thr, kind, sc[l])
        _, pred0 = orc.decode_train(wide[l], l, C)
        n_ignore_diff += int((orc.build_target(pred0, c["labels"], l, C, thr)[1] != obj_mask).sum())
        got = fused_yolo_loss_components([heads[l]], lab, cfg, thr, layers=[l], iou_loss=kind, scale_x_y=sc[l]).cpu().numpy()
        what = "%s s %r layer %d %s" % (kind, sc[l], l, dt)
        assert abs(got[0] - comps[0]) <= 1e-5 * abs(comps[0]) + 1e-6, (what, got[0], comps[0])
        assert got[1] == 0.0
        np.testing.assert_allclose(got[2], comps[2], rtol=1e-5, err_msg=what)
        np.testing.assert_allclose(got[3], comps[3], rtol=1e-5, err_msg=what)
        g = hs[l].grad
        obj = torch.stack([g[:, a * nch + 4] for a in range(3)], 1)
        assert bit_equal(obj, torch.from_numpy(gobj).to(dt)), what + ": objectness gradient plane"
        box = torch.cat([g[:, a * nch:a * nch + 4] for a in range(3)], 1).float().cpu().numpy()
        extreme = iou_loss_spec.extreme_extent(p)
        for (b, a, j, i), gr, ext in zip(cells, graw, extreme):
            if ext:
                continue
            got4 = box[b, 4 * a:4 * a + 4, j, i]
            if dt == torch.float32:
                assert iou_loss_spec.within_bound(got4, gr).all(), "%s cell %r: %r vs %r" % (what, (b, a, j, i), got4, gr)
            else:                                   # the fp32 value rounded once to fp16: one more half-ulp
                assert np.all(np.abs(got4 - gr) <= 1e-3 * np.abs(gr) + 1e-6 + 1e-4 * iou_loss_spec.GRAD_ABS), (what, got4, gr)
    return n_ignore_diff


@pytest.mark.parametrize("dt", [torch.float32, torch.float16])
@pytest.mark.parametrize("kind", iou_loss_spec.KINDS)
def test_fused_loss_equals_the_spec(kind, dt):
    c = scene_608(seed=31, B=2)
    assert check_loss(c, kind, YOLOV4, dt) > 0, "the scale changes no ignore decision in this scene"
    check_loss(c, kind, (2.0, 2.0, 2.0), dt)


def test_fused_loss_graph_replay_equals_eager_and_sgd_lowers_the_box_term():
    c = scene_608(seed=53, B=2)
    cfg = cfg_of(c["C"])
    lab = torch.from_numpy(c["labels"]).cuda()
    heads = [torch.from_numpy(r).cuda() for r in c["raws"]]
    kw = dict(iou_loss="ciou", scale_x_y=YOLOV4)
    eager = fused_yolo_loss_components(heads, lab, cfg, **kw).cpu().numpy()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fused_yolo_loss_components(heads, lab, cfg, **kw)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fused_yolo_loss_components(heads, lab, cfg, **kw)
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        np.testing.assert_allclose(out.cpu().numpy(), eager, rtol=1e-12, atol=0)
    box = torch.zeros(heads[0].shape[1], dtype=torch.bool, device="cuda")
    for a in range(3):
        box[a * 85:a * 85 + 4] = True
    vals = []
    for _ in range(6):
        vals.append(fused_yolo_loss_components(heads, lab, cfg, **kw)[0].item())
        hs = [h.detach().clone().requires_grad_(True) for h in heads]
        fused_yolo_loss(hs, lab, cfg, **kw).backward()
        heads = [h - 0.05 * h2.grad * box[None, :, None, None] for h, h2 in zip(heads, hs)]
    assert all(b < a for a, b in zip(vals, vals[1:])) and vals[-1] < 0.95 * vals[0], vals


# ------------------------------------------------------------------------------------------------ special logits
def test_special_logits_on_tx_ty():
    C, F = 4, 4
    specials = np.array([np.inf, -np.inf, np.nan, 0.0, -0.0, 88.0, -88.0, 1e-30], np.float32)
    raws = []
    for l, f in enumerate((F, 2, 1)):
        r = np.full((1, 3 * (5 + C), f, f), 3.0, np.float32)           # objectness / classes pass, w / h finite
        for a in range(3):
            k = (np.arange(f * f) + 3 * a + l).reshape(f, f)
            r[0, a * (5 + C)] = specials[k % len(specials)]
            r[0, a * (5 + C) + 1] = specials[(k + 2) % len(specials)]
        raws.append(torch.from_numpy(r).cuda())
    for sc in SCALES:
        want = spec.decode_eval_cat(_np(raws), C, sc)
        cfg = dict(CFG80, N_CLASSES=C)
        assert bit_equal(yb.decode_dense_cat(raws, cfg, scale_x_y=sc).cpu(), torch.from_numpy(want))
        # sigmoid(-inf) = 0: the centre is (beta + cell) * stride
        cx = want[0, :F * F, 0].reshape(F, F)
        tx = _np(raws)[0][0, 0]
        jj, ii = np.nonzero(tx == -np.inf)
        assert len(ii) and np.array_equal(cx[jj, ii], ((spec.beta(sc[0]) + ii.astype(np.float32)) * np.float32(8)).astype(np.float32))
        got = yb.detect_raw(raws, C, 0.2, 0.5, scale_x_y=sc)
        assert_lists_bit_equal(got, orc.postprocess(want, C, 0.2, 0.5), what=f"special {sc}")

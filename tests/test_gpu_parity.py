"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle and the reference-generated goldens.

Bars (BASELINE.json north_star): decoded values within 1e-5 relative of the reference; kept indices, counts,
rows and loss masks bit-exact.  Because the product and the oracle share the spec math, product-vs-oracle
comparisons below are bit-exact everywhere, including decoded values.
"""
import ctypes
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as orc                                     # noqa: E402  (checker only)
import yolov4_b200 as yb                                              # noqa: E402
from yolov4_b200 import _cabi                                         # noqa: E402
from yolov4_b200.synth import synth_head_outputs, synth_labels        # noqa: E402

CFG80 = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": 80}
REL = 1e-5


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def _split(counts, rows):
    out, o = [], 0
    for n in counts:
        out.append(rows[o:o + n] if n else None)
        o += n
    return out


def bit_equal(a, b):
    """Bitwise equality of fp32 arrays, except that any NaN equals any NaN (x86 and the GPU propagate different payloads)."""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a.view(np.uint32)[~na], b.view(np.uint32)[~nb]))


def assert_lists_bit_equal(got, ref, what=""):
    assert len(got) == len(ref), what
    for b, (g, r) in enumerate(zip(got, ref)):
        assert (g is None) == (r is None), f"{what} image {b}: None mismatch"
        if r is None:
            continue
        g = g.detach().cpu().numpy() if isinstance(g, torch.Tensor) else g
        assert g.shape == r.shape, f"{what} image {b}: {g.shape} vs {r.shape}"
        if not bit_equal(g, r):
            gb, rb = np.ascontiguousarray(g).view(np.uint32), np.ascontiguousarray(r).view(np.uint32)
            bad = np.argwhere((gb != rb) & ~(np.isnan(g) & np.isnan(r)))
            raise AssertionError(f"{what} image {b}: {len(bad)} words differ, first at {bad[0]}: {g[bad[0][0]]} vs {r[bad[0][0]]}")


def assert_rel(a, b, rel=REL, what=""):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    fin = np.isfinite(b)
    assert np.array_equal(np.isfinite(a), fin), what
    err = np.abs(a[fin] - b[fin])
    assert (err <= rel * np.abs(b[fin]) + 1e-30).all(), f"{what}: max rel {np.max(err / (np.abs(b[fin]) + 1e-30))}"


# ------------------------------------------------------------------------------------------------ decode
@pytest.mark.parametrize("tag", ["c80", "c4"])
def test_decode_eval_vs_reference_golden_and_oracle(golden_dir, tag):
    g = _load(golden_dir, "decode.npz")
    C = int(g[f"{tag}_C"])
    cfg = dict(CFG80, N_CLASSES=C)
    outs = []
    for l in range(3):
        layer = yb.YOLOLayer(cfg, l, device="cuda").eval()
        outs.append(layer(torch.from_numpy(g[f"{tag}_raw{l}"]).cuda()))
    got = torch.cat(outs, 1).cpu().numpy()
    ref = g[f"{tag}_eval"]
    tiny = np.abs(ref) < 1e-30
    assert_rel(np.where(tiny, 0, got), np.where(tiny, 0, ref), what="vs reference")
    want = orc.decode_eval_cat([g[f"{tag}_raw{l}"] for l in range(3)], C)
    assert bit_equal(got, want), "vs oracle (bit-exact)"


def test_bounded_reciprocal_is_ieee_for_every_float_of_its_range():
    """sigmoid = RN(1 / (1 + exp(-x))) (DESIGN.md 4): for |x| <= 86 the reciprocal is MUFU.RCP + one FMA Newton step
    without __frcp_rn's range check; it must equal the IEEE quotient on all 1.05e9 floats of [1, 2^125]."""
    bad = torch.ones(1, dtype=torch.int64, device="cuda")
    _cabi.check(_cabi.lib().yl_selftest_rcp(bad.data_ptr(), torch.cuda.current_stream().cuda_stream))
    assert int(bad.item()) == 0


def test_decode_eval_608_bit_exact_vs_oracle():
    raws = synth_head_outputs(2, 608, 80, seed=4, device="cuda")
    raws[2][0, :, :3, :3] = float("nan")
    raws[1][1, :, 5, 5] = 95.0        # exp overflow -> inf, sigmoid -> 1
    raws[1][1, :, 6, 6] = -120.0
    want = orc.decode_eval_cat([r.cpu().numpy() for r in raws], 80)
    outs = [yb.YOLOLayer(CFG80, l, device="cuda").eval()(raws[l].clone()) for l in range(3)]
    got = torch.cat(outs, 1).cpu().numpy()
    assert got.shape == (2, 22743, 85)
    assert np.isnan(got).sum() == 3 * 85 * 9 and np.isinf(got).sum() == 2 * 3
    assert bit_equal(got, want)
    # one-buffer form (no torch.cat) gives the same tensor
    assert torch.equal(torch.nan_to_num(yb.decode_dense_cat(raws, CFG80)), torch.nan_to_num(torch.cat(outs, 1)))
    # the reference overwrites its input in place; we must not touch it
    assert torch.equal(raws[0], synth_head_outputs(2, 608, 80, seed=4, device="cuda")[0])


@pytest.mark.parametrize("tag", ["c80", "c4"])
def test_decode_train_outputs_and_strides(golden_dir, tag):
    g = _load(golden_dir, "decode.npz")
    C = int(g[f"{tag}_C"])
    cfg = dict(CFG80, N_CLASSES=C)
    for l in range(3):
        raw = torch.from_numpy(g[f"{tag}_raw{l}"]).cuda()
        layer = yb.YOLOLayer(cfg, l, device="cuda").train()
        d = layer(raw)
        assert d["layer_no"] == l
        F = raw.shape[2]
        n_ch = 5 + C
        assert d["output"].shape == (2, 3, F, F, n_ch) and d["pred"].shape == (2, 3, F, F, 4)
        # same strides as the reference's permuted views (SURVEY.md 7-10)
        assert d["output"].stride() == (3 * n_ch * F * F, n_ch * F * F, F, 1, F * F)
        ro, rp = g[f"{tag}_train_output{l}"], g[f"{tag}_train_pred{l}"]
        o, p = d["output"].detach().cpu().numpy(), d["pred"].cpu().numpy()
        tiny = np.abs(ro) < 1e-30
        assert_rel(np.where(tiny, 0, o), np.where(tiny, 0, ro), what="train output vs reference")
        assert_rel(p, rp, what="train pred vs reference")
        oo, op = orc.decode_train(g[f"{tag}_raw{l}"], l, C)
        assert np.array_equal(o, oo) and np.array_equal(p, op), "vs oracle (bit-exact)"


def test_decode_train_backward_matches_autograd():
    raw = synth_head_outputs(2, 96, 80, seed=9, device="cuda")[0].requires_grad_(True)
    layer = yb.YOLOLayer(CFG80, 0, device="cuda").train()
    d = layer(raw)
    w = torch.randn_like(d["output"])
    (d["output"] * w).sum().backward()
    x = raw.detach().clone().requires_grad_(True)
    o = x.reshape(2, 3, 85, 12, 12).permute(0, 1, 3, 4, 2)
    idx = np.r_[:2, 4:85]
    ref = o.clone()
    ref[..., idx] = torch.sigmoid(o[..., idx])
    (ref * w).sum().backward()
    torch.testing.assert_close(raw.grad, x.grad, rtol=1e-5, atol=1e-7)


# ------------------------------------------------------------------------------------------------ postprocess
def test_postprocess_bit_exact_vs_reference_goldens(golden_dir):
    g = _load(golden_dir, "postprocess.npz")
    pred = torch.from_numpy(g["pred"]).cuda()
    i = 0
    while f"s{i}_conf" in g:
        conf, nmst = float(g[f"s{i}_conf"]), float(g[f"s{i}_nms"])
        before = pred.clone()
        out = yb.postprocess(pred, 80, conf, nmst)
        assert torch.equal(pred, before)
        assert all(o is None or (o.is_cuda and o.dtype == torch.float32) for o in out)
        assert_lists_bit_equal(out, _split(g[f"s{i}_counts"], g[f"s{i}_rows"]), what=f"setting {i}")
        i += 1
    assert i == 5
    assert yb.postprocess(pred, 80, float(g["empty_conf"]), 0.4) == [None, None]
    out = yb.postprocess(torch.from_numpy(g["ties_pred"]).cuda(), 3, 0.2, 0.5)
    assert_lists_bit_equal(out, _split(g["ties_counts"], g["ties_rows"]), what="all-ties")


def test_postprocess_cpu_tensor_roundtrip(golden_dir):
    """detect.py:115-118 hands postprocess a CPU tensor; results come back on the CPU."""
    g = _load(golden_dir, "postprocess.npz")
    out = yb.postprocess(torch.from_numpy(g["pred"]), 80, 0.2, 0.5)
    assert all(o.device.type == "cpu" for o in out if o is not None)
    assert_lists_bit_equal(out, _split(g["s1_counts"], g["s1_rows"]))


@pytest.mark.parametrize("seed,clustered,conf,nmst", [(0, False, 1e-4, 0.4), (1, True, 1e-4, 0.4), (2, True, 0.2, 0.5),
                                                      (3, True, 0.005, 0.4), (4, False, 0.001, 0.4)])
def test_postprocess_dense_vs_oracle_608(seed, clustered, conf, nmst):
    raws = synth_head_outputs(2, 608, 80, seed=seed, device="cuda", clustered=clustered, fg_prob=0.02 if clustered else 0.005)
    dense = torch.cat([yb.YOLOLayer(CFG80, l, device="cuda").eval()(raws[l]) for l in range(3)], 1)
    want = orc.postprocess(dense.cpu().numpy(), 80, conf, nmst, nthreads=8)
    got = yb.postprocess(dense, 80, conf, nmst)
    assert_lists_bit_equal(got, want, what="dense path")
    fused = yb.detect_raw(raws, 80, conf, nmst)
    assert_lists_bit_equal(fused, want, what="fused path")
    if clustered:
        n_cand = int(((dense[:, :, 5:] * dense[:, :, 4:5]) >= float(np.float32(conf))).sum())
        assert sum(0 if w is None else len(w) for w in want) < n_cand, "NMS must suppress something in the clustered case"


def test_fused_vs_oracle_detect_416_and_odd_shapes():
    for img, C, B in ((416, 80, 3), (96, 4, 5), (64, 20, 1), (96, 20, 4)):
        raws = synth_head_outputs(B, img, C, seed=img, device="cuda", fg_prob=0.05, clustered=True)
        want = orc.detect([r.cpu().numpy() for r in raws], C, 0.01, 0.45, nthreads=8)
        got = yb.detect_raw(raws, C, 0.01, 0.45)
        assert_lists_bit_equal(got, want, what=f"img {img} C {C}")


def test_postprocess_pathological_values():
    """NaN / inf / zero-area / negative values in an already decoded tensor (utils.py NaN semantics, SURVEY.md 7-5)."""
    rng = np.random.RandomState(5)
    B, M, C = 2, 600, 6
    pred = np.zeros((B, M, 5 + C), np.float32)
    pred[..., 0:2] = rng.rand(B, M, 2) * 100
    pred[..., 2:4] = rng.rand(B, M, 2) * 40
    pred[..., 4] = rng.rand(B, M)
    pred[..., 5:] = rng.rand(B, M, C) ** 3
    pred[0, 0:20, 2:4] = 0.0                       # zero-area boxes: 0/0 IoU -> kept
    pred[0, 5:10, 0:2] = pred[0, 0:5, 0:2]
    pred[0, 30, 0] = np.nan                         # NaN coordinate
    pred[0, 31, 2] = np.inf
    pred[0, 32, 7] = np.nan                         # NaN class -> row dropped by the max() pre-filter
    pred[1, 40, 4] = np.nan                         # NaN objectness
    pred[1, 41, 4] = -0.5                           # negative objectness
    pred[1, 50:60, :] = pred[1, 60:70, :]           # exact duplicates -> score ties + IoU 1
    for conf, nmst in ((0.05, 0.45), (0.3, 0.0001), (0.0, 0.5)):
        want = orc.postprocess(pred, C, conf, nmst)
        got = yb.postprocess(torch.from_numpy(pred).cuda(), C, conf, nmst)
        assert_lists_bit_equal(got, want, what=f"conf {conf} nms {nmst}")


def test_nms_small_tier_code_paths():
    """Segments built to hit every branch of k_segment_nms_bins: a dense cluster whose candidate pairs overflow the pair
    queues (passed on to the big tier), segments of exactly 256 / 257 records (tier boundary), scores that tie in their
    upper 27 bits (64-bit re-rank), exact ties, chains (a suppresses b, b would suppress c), boxes with NaN / zero /
    negative extents inside an otherwise ordinary segment, and thresholds near 0 and 1."""
    rng = np.random.RandomState(11)
    C = 6
    rows = []

    def add(cls, xy, wh, score):
        r = np.zeros((len(xy), 5 + C), np.float32)
        r[:, 0:2], r[:, 2:4], r[:, 4] = xy, wh, 1.0
        r[:, 5 + cls] = score
        rows.append(r)

    n = 250                                                     # class 0: one dense cluster, all pairs overlap -> queue overflow
    add(0, 300 + rng.randn(n, 2) * 6, 80 + rng.rand(n, 2) * 30, 0.2 + 0.7 * rng.rand(n))
    add(1, rng.rand(256, 2) * 580 + 10, 10 + rng.rand(256, 2) * 60, 0.2 + 0.7 * rng.rand(256))      # exactly 256 records
    add(2, rng.rand(257, 2) * 580 + 10, 10 + rng.rand(257, 2) * 60, 0.2 + 0.7 * rng.rand(257))      # 257: big tier
    base = np.float32(0.5)                                      # class 3: scores that differ only in their low mantissa bits
    sc = (base.view(np.uint32) + rng.randint(0, 32, 90).astype(np.uint32)).view(np.float32)
    add(3, 200 + rng.randn(90, 2) * 40, 40 + rng.rand(90, 2) * 40, sc)
    add(3, 200 + rng.randn(10, 2) * 40, 40 + rng.rand(10, 2) * 40, np.full(10, 0.5, np.float32))    # and exact ties
    k = 60                                                      # class 4: chains of shifted boxes (greedy order matters)
    add(4, np.stack([100 + 12.0 * np.arange(k), np.full(k, 400.0)], 1), np.full((k, 2), 40.0), np.linspace(0.9, 0.3, k))
    add(5, rng.rand(100, 2) * 500 + 50, 20 + rng.rand(100, 2) * 80, 0.2 + 0.7 * rng.rand(100))      # class 5: odd boxes inside
    odd = rows[-1]
    odd[3, 0] = np.nan; odd[7, 2] = 0.0; odd[9, 3] = -5.0; odd[11, 2] = np.inf; odd[13, 1] = -np.inf
    pred = np.concatenate(rows, 0)[rng.permutation(sum(len(r) for r in rows))][None]
    for conf, nmst in ((0.1, 0.4), (0.1, 0.45), (0.1, 0.999), (0.1, 1e-6), (0.1, 0.7)):
        want = orc.postprocess(pred, C, conf, nmst)
        got = yb.postprocess(torch.from_numpy(pred).cuda(), C, conf, nmst)
        assert_lists_bit_equal(got, want, what=f"conf {conf} nms {nmst}")


def test_oversized_segments_take_the_global_path_and_capacity_grows():
    """All-zero logits = the random-init degenerate case (SURVEY.md 7-2): every score is exactly 0.25, every pair
    survives, segments (1575 candidates) exceed both the default cap_seg and the shared-memory limit."""
    raws = [torch.zeros(2, 255, f, f, device="cuda") for f in (20, 10, 5)]
    raws[0][1, 4] = -20.0                           # image 1: first layer silenced
    want = orc.detect([r.cpu().numpy() for r in raws], 80, 0.2, 0.5, nthreads=8)
    got = yb.detect_raw(raws, 80, 0.2, 0.5)
    assert_lists_bit_equal(got, want)
    assert len(want[0]) > 20000


def test_head_postprocessor_graph_replay_matches_eager():
    raws = synth_head_outputs(8, 608, 80, seed=11, device="cuda")
    want = yb.detect_raw(raws, 80, 1e-4, 0.4)
    hp = yb.HeadPostprocessor(8, [76, 38, 19], 80, 1e-4, 0.4, n_groups=4).capture(raws)
    for _ in range(3):
        hp.replay()
    torch.cuda.synchronize()
    got = hp.results()
    assert_lists_bit_equal(got, [w.cpu().numpy() for w in want])
    # new data in the captured buffers is picked up by the next replay
    fresh = synth_head_outputs(8, 608, 80, seed=12, device="cuda")
    for dst, src in zip(hp._captured_inputs, fresh):
        dst.copy_(src)
    hp.replay()
    torch.cuda.synchronize()
    assert_lists_bit_equal(hp.results(), [w.cpu().numpy() for w in yb.detect_raw(fresh, 80, 1e-4, 0.4)])


def test_full_size_properties_b64():
    """BASELINE config 2 shape (B=64 @608, conf 1e-4, nms 0.4): size-independent properties."""
    raws = synth_head_outputs(64, 608, 80, seed=0, device="cuda")
    out = yb.detect_raw(raws, 80, 1e-4, 0.4)
    assert len(out) == 64
    total = 0
    for o in out:
        assert o is not None and o.shape[1] == 7
        cls = o[:, 6]
        assert torch.all(cls[1:] >= cls[:-1]), "classes ascending"
        score = o[:, 4] * o[:, 5]
        same = cls[1:] == cls[:-1]
        assert torch.all(score[1:][same] <= score[:-1][same]), "score descending inside a class"
        assert torch.all(score >= float(np.float32(1e-4)))
        total += o.shape[0]
    assert 64 * 8000 < total < 64 * 16000
    # idempotence: NMS output fed back as the only candidates is kept entirely -> batch sharding is exact:
    sub = yb.detect_raw([r[10:14] for r in raws], 80, 1e-4, 0.4)
    for a, b in zip(sub, out[10:14]):
        assert torch.equal(a, b), "image results do not depend on batch composition"
    # spot-check four images against the oracle
    want = orc.detect([r[:4].cpu().numpy() for r in raws], 80, 1e-4, 0.4, nthreads=8)
    assert_lists_bit_equal(out[:4], want)


# ------------------------------------------------------------------------------------------------ host-buffer C ABI
def test_detect_host_c_abi_matches_oracle():
    L = _cabi.lib()
    B, C = 6, 80
    raws = [r.numpy() for r in synth_head_outputs(B, 416, C, seed=21, fg_prob=0.02, clustered=True)]
    Fs = [r.shape[2] for r in raws]
    ctx = ctypes.c_void_p()
    cap_out = 32768
    anch = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
    mask = _cabi.ints([v for m in yb.ANCHOR_MASK for v in m])
    _cabi.check(L.yl_context_create(ctypes.byref(ctx), 0, B, _cabi.ints(Fs), 3, C, anch, mask, 1024, cap_out))
    rows = np.zeros((B, cap_out, 7), np.float32)
    counts = np.zeros((B,), np.int32)
    ptrs = _cabi.ptrs([r.ctypes.data for r in raws])
    for conf, nmst in ((0.001, 0.4), (0.2, 0.5)):
        _cabi.check(L.yl_detect_host(ctx, ptrs, float(np.float32(conf)), float(np.float32(nmst)), rows.ctypes.data, counts.ctypes.data))
        want = orc.detect(raws, C, conf, nmst, nthreads=8)
        got = [rows[b, :counts[b]] if counts[b] else None for b in range(B)]
        assert_lists_bit_equal(got, want, what=f"host path conf {conf}")
    _cabi.check(L.yl_context_destroy(ctx))


def test_c_abi_argument_errors():
    L = _cabi.lib()
    assert L.yl_decode_dense(None, 1, 4, 80, None, 8.0, None, 48, 0, None) == 1
    assert L.yl_post_workspace_bytes(0, 10, 80, 16) == 0
    assert L.yl_nms(None, 0, 1, 10, 80, 16, 0.5, None, 1, None, 0, 1, None) == 1
    assert b"invalid argument" in L.yl_error_string(1)
    x = torch.zeros(1, 3 * 205, 4, 4, device="cuda")
    with pytest.raises(_cabi.YoloHeadError):
        yb.detect_raw([x], 200, 0.5, 0.5)           # more classes than YL_MAX_CLASSES
    with pytest.raises(TypeError):
        yb.YOLOLayer(CFG80, 0).eval()(torch.zeros(1, 255, 4, 4))     # CPU tensor: no fallback


# ------------------------------------------------------------------------------------------------ build_target
@pytest.mark.parametrize("layer", [0, 1, 2])
def test_build_target_vs_reference_golden(golden_dir, layer):
    g = _load(golden_dir, "build_target.npz")
    C = int(g["C"])
    pred = torch.from_numpy(g[f"pred{layer}"]).cuda()
    F = pred.shape[2]
    crit = yb.YOLOLoss(dict(CFG80, N_CLASSES=C), ignore_thresh=0.7, device="cuda")
    output = torch.empty(pred.shape[0], 3, F, F, 5 + C, device="cuda")
    labels = torch.from_numpy(g["labels"]).double()          # the loader hands float64 (SURVEY.md A8)
    target, obj_mask, tgt_mask, tgt_scale = [t.cpu().numpy() for t in crit.build_target(output, pred, layer, labels)]
    assert np.array_equal(obj_mask, g[f"obj_mask{layer}"])
    assert np.array_equal(tgt_mask, g[f"tgt_mask{layer}"])
    assert np.array_equal(tgt_scale, g[f"tgt_scale{layer}"], equal_nan=True)
    rt = g[f"target{layer}"]
    sel = np.ones(rt.shape[-1], bool)
    sel[2:4] = False
    assert np.array_equal(target[..., sel], rt[..., sel])
    np.testing.assert_allclose(target[..., 2:4], rt[..., 2:4], rtol=1e-5, atol=1e-6)


def test_build_target_608_b8_bit_exact_vs_oracle_with_strided_pred():
    B = 8
    raws = synth_head_outputs(B, 608, 80, seed=31, device="cuda")
    labels = synth_labels(B, 608, n_valid=50, seed=32, device="cuda")
    labels[3] = 0.0                                           # an image without objects
    labels[5, 7] = labels[5, 6]                               # duplicate GT (collision)
    labels[5, 8, :4] = labels[5, 6, :4]
    labels[5, 8, 4] = (labels[5, 6, 4] + 3) % 80              # same cell, other class
    crit = yb.YOLOLoss(CFG80, ignore_thresh=0.7, device="cuda")
    for l in range(3):
        d = yb.YOLOLayer(CFG80, l, device="cuda").train()(raws[l])
        pred = d["pred"].clone() if l == 1 else d["pred"]    # contiguous copy and strided view both work
        # make the ignore mask non-trivial: plant a few GT boxes as predictions
        s = float(8 << l)
        for b in (0, 1, 2):
            for t in range(0, 50, 5):
                i, j = int(labels[b, t, 0] / s), int(labels[b, t, 1] / s)
                pred[b, t % 3, j, i, :] = labels[b, t, :4] / s * 1.03
        got = crit.build_target(d["output"], pred, l, labels)
        want = orc.build_target(pred.cpu().numpy(), labels.cpu().numpy(), l, 80, 0.7)
        for name, gt, wt in zip(("target", "obj_mask", "tgt_mask", "tgt_scale"), got, want):
            assert np.array_equal(gt.cpu().numpy(), wt, equal_nan=True), f"layer {l} {name}"
        assert (want[1] == 0).sum() > 0 and want[2].sum() > 0


def test_build_targets3_one_launch_equals_three_calls():
    """yl_build_target3 (one launch pair for the three scales, what YOLOLoss.forward uses) against three yl_build_target calls."""
    B = 4
    raws = synth_head_outputs(B, 608, 80, seed=33, device="cuda")
    labels = synth_labels(B, 608, n_valid=50, seed=34, device="cuda")
    labels[2] = 0.0
    crit = yb.YOLOLoss(CFG80, ignore_thresh=0.7, device="cuda")
    ds = [yb.YOLOLayer(CFG80, l, device="cuda").train()(raws[l]) for l in range(3)]
    for l in range(3):                                         # plant a few GT boxes as predictions: non-trivial ignore masks
        s = float(8 << l)
        for t in range(0, 50, 7):
            i, j = int(labels[0, t, 0] / s), int(labels[0, t, 1] / s)
            ds[l]["pred"][0, t % 3, j, i, :] = labels[0, t, :4] / s * 1.02
    one = yb.build_targets3([d["output"] for d in ds], [d["pred"] for d in ds], [0, 1, 2], labels, yb.ANCHORS_PX, yb.ANCHOR_MASK, 0.7, 80)
    for l in (2, 0, 1):                                        # any order, and a subset
        three = crit.build_target(ds[l]["output"], ds[l]["pred"], l, labels)
        for a, b in zip(one[l], three):
            assert torch.equal(a, b)
    sub = yb.build_targets3([ds[2]["output"], ds[0]["output"]], [ds[2]["pred"], ds[0]["pred"]], [2, 0], labels, yb.ANCHORS_PX,
                            yb.ANCHOR_MASK, 0.7, 80)
    for a, b in zip(sub[0], one[2]):
        assert torch.equal(a, b)
    for a, b in zip(sub[1], one[0]):
        assert torch.equal(a, b)
    assert sum(int((o[1] == 0).sum()) for o in one) > 0


@pytest.mark.parametrize("ign", [0.7, 0.3, 0.0, -0.5, 1.0])
def test_build_target_ignore_mask_pathological_boxes(ign):
    """The ignore test walks the well-formed GTs in area order and skips those whose area rules the threshold out; GTs
    and predictions with non-finite / huge / non-positive extents take the literal NaN-propagating formula
    (yololoss.py:64-91, 276-294).  Every combination must give the oracle's masks bit for bit."""
    B, img, C = 4, 160, 4
    cfg = dict(CFG80, N_CLASSES=C)
    raws = synth_head_outputs(B, img, C, seed=77, device="cuda", fg_prob=0.05)
    rng = np.random.RandomState(5)
    K = 16
    labels = np.zeros((B, K, 5), np.float32)
    for b in range(B):
        n = 12
        labels[b, :n, 0:2] = rng.uniform(4, img - 4, (n, 2))
        labels[b, :n, 2:4] = np.exp(rng.uniform(np.log(4.0), np.log(img * 0.8), (n, 2)))
        labels[b, :n, 4] = rng.randint(0, C, n)
    labels[0, 2, 2:4] = labels[0, 1, 2:4]                     # equal areas (ties in the area order)
    labels[0, 3, 2:4] = labels[0, 1, 3:1:-1]                  # same area, transposed box
    labels[1, 1, 2] = np.inf                                  # not "simple": literal formula
    labels[1, 4, 3] = 1e30
    labels[1, 5, 2] = 0.0                                     # zero area
    labels[2, 0, 2] = -20.0                                   # negative width (area < 0)
    labels[2, 3, 2:4] = (-20.0, -30.0)                        # negative width and height (area > 0)
    labels[3, 2, 3] = np.nan
    lab = torch.from_numpy(labels).cuda()
    crit = yb.YOLOLoss(cfg, ignore_thresh=ign, device="cuda")
    for l in range(3):
        d = yb.YOLOLayer(cfg, l, device="cuda").train()(raws[l])
        pred = d["pred"].clone()
        s = float(8 << l)
        F = pred.shape[2]
        for b in range(B):                                    # predictions planted on / near ground truths
            for t in range(0, 12, 2):
                i, j = min(int(labels[b, t, 0] / s), F - 1), min(int(labels[b, t, 1] / s), F - 1)
                v = torch.from_numpy(labels[b, t, :4] / s).cuda()
                pred[b, t % 3, j, i, :] = torch.nan_to_num(v, nan=1.0, posinf=3.0, neginf=1.0).abs() * (1.0 + 0.02 * (t % 5))
        pred[0, 0, 0, 0, 2] = float("nan")
        pred[0, 1, 0, 1, 3] = float("inf")
        pred[1, 2, 1, 0, 2] = 0.0
        pred[2, 0, 1, 1, 2] = -1.5
        pred[3, 1, 0, 0, 0] = 1e25
        got = crit.build_target(d["output"], pred, l, lab)
        want = orc.build_target(pred.cpu().numpy(), labels, l, C, ign)
        for name, gt, wt in zip(("target", "obj_mask", "tgt_mask", "tgt_scale"), got, want):
            assert np.array_equal(gt.cpu().numpy(), wt, equal_nan=True), f"ign {ign} layer {l} {name}"


def test_yololoss_forward_runs_and_backprops():
    raws = [r.requires_grad_(True) for r in synth_head_outputs(2, 96, 80, seed=41, device="cuda")]
    labels = synth_labels(2, 96, n_valid=6, seed=42, device="cuda")
    labels[..., 2:4].clamp_(max=60.0)
    outs = [yb.YOLOLayer(CFG80, l, device="cuda").train()(raws[l]) for l in range(3)]
    loss = yb.YOLOLoss(CFG80, 0.7, device="cuda")(outs, {"padded_labels": labels.double()})
    assert torch.isfinite(loss)
    loss.backward()
    assert all(r.grad is not None and torch.isfinite(r.grad).all() for r in raws)


# ------------------------------------------------------------------------------------------------ N2 fused loss
def test_fused_loss_vs_reference_golden(golden_dir):
    """Loss value and gradient w.r.t. the raw head tensors against the reference's YOLOLoss.forward + autograd
    (tests/golden/loss.npz): 1e-5 relative on the loss, 2e-5 relative on the gradient, identical gradient support."""
    g = _load(golden_dir, "loss.npz")
    C = int(g["C"])
    cfg = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": C}
    raws = [torch.from_numpy(g[f"raw{l}"]).cuda().requires_grad_(True) for l in range(3)]
    labels = torch.from_numpy(g["labels"]).cuda()
    loss = yb.fused_yolo_loss(raws, labels, cfg, 0.7)
    assert abs(loss.item() - float(g["loss"])) <= 1e-5 * abs(float(g["loss"]))
    loss.backward()
    for l in range(3):
        got, ref = raws[l].grad.cpu().numpy().astype(np.float64), g[f"grad{l}"].astype(np.float64)
        assert np.array_equal(got != 0, ref != 0), "layer %d: gradient support differs" % l
        assert np.allclose(got, ref, rtol=2e-5, atol=1e-7), (l, np.abs(got - ref).max())
    # per layer, through the oracle's four components
    for l in range(3):
        one = yb.fused_yolo_loss_components([raws[l].detach()], labels, cfg, 0.7, layers=[l])
        want, _ = orc.yolo_loss_layer(g[f"raw{l}"], g["labels"], l, C, 0.7)
        assert np.allclose(one.cpu().numpy(), want, rtol=1e-5, atol=1e-6), (l, one, want)


def test_fused_loss_608_vs_oracle_and_unfused_path():
    """B=4 @608, 50 GT/image: fused loss against the oracle (value, gradient) and against the unfused CUDA path
    (YOLOLayer.train -> YOLOLoss.forward in torch on top of yl_build_target)."""
    B, C = 4, 80
    raws_np = [r.numpy() for r in synth_head_outputs(B, 608, C, seed=77)]
    labels = synth_labels(B, 608, n_valid=50, seed=78)
    raws = [torch.from_numpy(r).cuda().requires_grad_(True) for r in raws_np]
    loss = yb.fused_yolo_loss(raws, labels.cuda(), CFG80, 0.7)
    loss.backward()
    want = 0.0
    for l in range(3):
        ls, gr = orc.yolo_loss_layer(raws_np[l], labels.numpy(), l, C, 0.7)
        want += ls.sum()
        got = raws[l].grad.cpu().numpy().astype(np.float64)
        assert np.array_equal(got != 0, gr != 0)
        assert np.allclose(got, gr, rtol=2e-5, atol=1e-7), (l, np.abs(got - gr).max())
    assert abs(loss.item() - want) <= 1e-5 * abs(want), (loss.item(), want)
    raws2 = [torch.from_numpy(r).cuda().requires_grad_(True) for r in raws_np]
    outs = [yb.YOLOLayer(CFG80, l, device="cuda").train()(raws2[l]) for l in range(3)]
    loss2 = yb.YOLOLoss(CFG80, 0.7, device="cuda")(outs, {"padded_labels": labels.double().cuda()})
    loss2.backward()
    assert abs(loss2.item() - loss.item()) <= 2e-5 * abs(loss.item())
    for l in range(3):
        assert torch.allclose(raws2[l].grad, raws[l].grad, rtol=1e-4, atol=1e-6)


def test_fused_loss_graph_replay_matches_eager_and_oracle():
    """The six forward kernels of the three scales overlap on the device (programmatic dependent launch, yl_loss_forward):
    a replayed CUDA graph -- where the overlap is tightest and the caching allocator would love to reuse a freed per-scale
    buffer -- must give the eager value and the oracle's."""
    from yolov4_b200.yololoss import fused_yolo_loss_components
    B = 16
    raws = synth_head_outputs(B, 608, 80, seed=41, device="cuda")
    labels = synth_labels(B, 608, n_valid=50, seed=42, device="cuda")
    eager = fused_yolo_loss_components(raws, labels, CFG80, 0.7).clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fused_yolo_loss_components(raws, labels, CFG80, 0.7)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fused_yolo_loss_components(raws, labels, CFG80, 0.7)
    for _ in range(5):
        g.replay()
        torch.cuda.synchronize()
        assert torch.allclose(out, eager, rtol=1e-12, atol=0), (out.tolist(), eager.tolist())
    want = sum(orc.yolo_loss_layer(raws[l].cpu().numpy(), labels.cpu().numpy(), l, 80, 0.7)[0] for l in range(3))
    np.testing.assert_allclose(out.cpu().numpy(), want, rtol=1e-5)



# ------------------------------------------------------------------------------------------------ N1 epilogue
def test_coco_and_detect_epilogue_bit_exact_vs_reference(golden_dir):
    g = _load(golden_dir, "epilogue.npz")
    outs, o = [], 0
    for k in g["counts"]:
        outs.append(torch.from_numpy(g["rows"][o:o + k]).cuda() if k else None)
        o += k
    coco = yb.coco_rows(outs, g["img_info"].tolist(), g["image_ids"].tolist(), g["class_ids"].tolist()).cpu().numpy()
    assert coco.dtype == np.float64 and np.array_equal(coco.view(np.uint64), g["coco"].view(np.uint64))
    det = yb.detect_rows(outs, g["img_info"].tolist(), g["class_ids"].tolist()).cpu().numpy()
    assert np.array_equal(det.view(np.uint64), g["detect"].view(np.uint64))
    d = yb.coco_dicts(outs, g["img_info"].tolist(), g["image_ids"].tolist(), g["class_ids"].tolist())
    assert len(d) == int(g["counts"].sum()) and d[0]["image_id"] == 139 and d[0]["bbox"] == g["coco"][0, 2:6].tolist()
    assert yb.coco_rows([None, None], g["img_info"].tolist()[:2], [1, 2], g["class_ids"].tolist()).shape == (0, 7)
    # the padded form of the device path (rows [B, cap_out, 7] + counts), one launch for the batch: the same bits
    cap = 64
    rows = torch.full((len(outs), cap, 7), float("nan"), device="cuda")
    for b, o_ in enumerate(outs):
        if o_ is not None:
            rows[b, :o_.shape[0]] = o_
    counts = torch.from_numpy(g["counts"].astype(np.int32)).cuda()
    for mode, want in ((0, g["coco"]), (1, g["detect"])):
        ids = g["image_ids"].tolist() if mode == 0 else list(range(len(outs)))
        got = yb.coco_rows_padded(rows, counts, g["img_info"].tolist(), ids, g["class_ids"].tolist(), mode=mode).cpu().numpy()
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64))


# ------------------------------------------------------------------------------------------------ BASELINE-size reference pins
def _fullsize(golden_dir):
    import sys
    if golden_dir not in sys.path:
        sys.path.insert(0, golden_dir)
    import fullsize_inputs as fi
    return fi, _load(golden_dir, "fullsize.npz")


def test_fullsize_608_postprocess_and_fused_vs_reference_golden(golden_dir):
    """BASELINE configs 2 / 3 at 608x608 against the REFERENCE's postprocess (fullsize.npz): dense decode -> postprocess, and the
    fused raw path, bit for bit; then raw -> detections against the reference's own decode + postprocess (counted flips)."""
    import hashlib
    from test_oracle_golden import _check_refdec
    fi, g = _fullsize(golden_dir)
    raws_c = fi.raws_cpu()
    raws = [r.cuda() for r in raws_c]
    dense = torch.cat([yb.YOLOLayer(CFG80, l, device="cuda").eval()(raws[l]) for l in range(3)], 1)
    pred = dense.cpu().numpy()
    # the golden was generated from the oracle's decoded tensor: the CUDA decode must be that tensor
    assert bit_equal(pred, orc.decode_eval_cat([r.numpy() for r in raws_c], fi.C))
    for tag, conf, nmst in fi.SETTINGS:
        counts = g[f"{tag}_counts"]
        if tag == "det":
            want = _split(counts, g["det_rows"])
        else:
            want = fi.rows_from_kept(pred, counts, g["val_kept_idx"], g["val_kept_cls"])
            assert hashlib.sha256(np.ascontiguousarray(np.concatenate(want, 0)).tobytes()).hexdigest() == str(g["val_sha256"])
        assert_lists_bit_equal(yb.postprocess(dense, fi.C, conf, nmst), want, what=f"dense {tag}")
        fused = yb.detect_raw(raws, fi.C, conf, nmst)
        assert_lists_bit_equal(fused, want, what=f"fused {tag}")
    fused = yb.detect_raw(raws, fi.C, fi.SETTINGS[0][1], fi.SETTINGS[0][2])
    _check_refdec(fi, g, pred, [f.cpu().numpy() for f in fused])


@pytest.mark.parametrize("layer", [0, 1, 2])
def test_fullsize_608_build_target_vs_reference_golden(golden_dir, layer):
    """BASELINE config 4 shape (608x608, 50 GT / image) against the reference's build_target (fullsize.npz, stored sparse)."""
    from test_oracle_golden import _check_fullsize_bt
    fi, g = _fullsize(golden_dir)
    raws = fi.raws_cpu()
    labels = fi.labels_cpu()
    d = yb.YOLOLayer(CFG80, layer, device="cuda").train()(raws[layer].cuda())
    _, p_or = orc.decode_train(raws[layer].numpy(), layer, fi.C)
    assert bit_equal(d["pred"].cpu().numpy(), p_or)            # the golden's pred is the oracle's: the CUDA train decode equals it
    p = fi.plant_pred(d["pred"].cpu().numpy().copy(), labels.numpy(), layer)
    crit = yb.YOLOLoss(CFG80, ignore_thresh=0.7, device="cuda")
    got = crit.build_target(d["output"], torch.from_numpy(p).cuda(), layer, labels.double())
    _check_fullsize_bt(fi, g, layer, [t.cpu().numpy() for t in got])


# ------------------------------------------------------------------------------------------------ non-default forms (read at load)
@pytest.mark.parametrize("env", [{"YL_FLAG": "ldg"}, {"YL_PDL": "0"}])
def test_alternative_kernel_forms_bit_exact_in_a_fresh_process(env):
    """The forms selected by environment switches when the library loads (k_flag_raw as the streaming flag kernel at every
    threshold, no programmatic dependent launch) produce the oracle's bits too.  A fresh process per form."""
    import subprocess
    import sys
    code = r'''
import sys, numpy as np, torch
sys.path.insert(0, %r)
import yolov4_b200 as yb
from yolov4_b200.synth import synth_head_outputs
from oracle import oracle as orc
cfg = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": 80}
for img, B, conf, kw in ((608, 3, 1e-4, {}), (416, 2, 1e-3, dict(fg_prob=0.03, clustered=True)), (608, 2, 0.2, {})):
    raws = synth_head_outputs(B, img, 80, seed=img + B, device="cuda", **kw)
    want = orc.detect([r.cpu().numpy() for r in raws], 80, conf, 0.4, nthreads=8)
    got = yb.detect_raw(raws, 80, conf, 0.4)
    dense = yb.decode_dense_cat(raws, cfg)
    got2 = yb.postprocess(dense, 80, conf, 0.4)
    for g, g2, w in zip(got, got2, want):
        assert (g is None) == (w is None) and (g2 is None) == (w is None)
        if w is not None:
            assert np.array_equal(g.cpu().numpy().view(np.uint32), w.view(np.uint32))
            assert np.array_equal(g2.cpu().numpy().view(np.uint32), w.view(np.uint32))
print("forms-ok")
''' % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))),)
    e = dict(os.environ)
    e.update(env)
    p = subprocess.run([sys.executable, "-c", code], env=e, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and "forms-ok" in p.stdout, p.stderr[-2000:]

"""The dense front end (yl_filter_dense, the filter behind postprocess) on both of its kernels: k_filter_dense_rows<NJ> for a
16-byte aligned base and k_filter_dense_unaligned otherwise.  Every case runs through the C ABI (yl_post_reset,
yl_filter_dense, yl_nms) with the input copied to each base residue mod 16, and checks two things: every image's candidate
total (meta[2B+b]) and largest class segment (meta[B+b]) equal the counts of the literal filter (agnostic_spec.candidates),
since NMS can hide an extra candidate, and the rows equal the C oracle's bit for bit."""
import importlib

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import yolov4_b200 as yb                                              # noqa: E402
from yolov4_b200 import _cabi                                         # noqa: E402
from yolov4_b200.synth import synth_head_outputs                      # noqa: E402

import agnostic_spec as spec                                          # noqa: E402
import dense_edge_cases as dec                                        # noqa: E402
from oracle import oracle as orc                                      # noqa: E402  (checker only)
from test_gpu_parity import assert_lists_bit_equal                    # noqa: E402

CFG80 = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": 80}
NMS = 0.45
RESIDUES = (0, 1, 2, 3)           # base offset in floats: data_ptr() % 16 = 0 (k_filter_dense_rows), 4, 8, 12 (unaligned)


def _f32(x):
    return float(np.float32(x))


def _pow2(n):
    p = 1
    while p < n:
        p <<= 1
    return p


def at_residue(pred, off):
    """pred ([B, M, 5+C] NumPy array or CUDA tensor) copied into a CUDA buffer `off` floats past a 16-byte boundary."""
    t = torch.as_tensor(pred).cuda()
    buf = torch.empty(t.numel() + 4, dtype=torch.float32, device="cuda")
    v = buf[off:off + t.numel()].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 == 4 * off
    return v


def expected_counts(pred, num_classes, conf):
    """Per image: candidates of the literal filter, and the size of its largest (image, class) segment."""
    tot, seg = [], []
    for p in pred:
        cls = spec.candidates(p, num_classes, conf)["cls"]
        tot.append(len(cls))
        seg.append(int(np.bincount(cls).max()) if len(cls) else 0)
    return np.array(tot), np.array(seg)


def run_cabi(x, num_classes, conf, cap_seg, cap_out, groups=None):
    """yl_post_reset, yl_filter_dense over each (img_first, img_count) of groups (default: the whole batch) into one
    workspace, one yl_nms over all images.  Returns (rows [B, cap_out, 7], meta [3B]) as NumPy arrays."""
    B, M, nch = x.shape
    C = nch - 5
    L = _cabi.lib()
    nb = L.yl_post_workspace_bytes(B, M, C, cap_seg)
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    rows = torch.full((B, cap_out, 7), 7.0, device="cuda")
    meta = torch.full((3 * B,), -1, dtype=torch.int32, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    _cabi.check(L.yl_post_reset(ws.data_ptr(), nb, B, M, C, cap_seg, st))
    for i0, n in groups or [(0, B)]:
        _cabi.check(L.yl_filter_dense(x.data_ptr(), B, M, C, num_classes, _f32(conf), ws.data_ptr(), nb, cap_seg, i0, n, st))
    _cabi.check(L.yl_nms(ws.data_ptr(), nb, B, M, C, cap_seg, _f32(NMS), rows.data_ptr(), cap_out, meta.data_ptr(), 0, B, st))
    torch.cuda.synchronize()
    return rows.cpu().numpy(), meta.cpu().numpy()


def check_dense(pred, num_classes, conf, residues=RESIDUES, extra=(), groups=None, what=""):
    """Runs pred at every base residue (and on the tensors of extra, (label, CUDA tensor) pairs holding the same values) and
    asserts the counts, the rows and that every run wrote the same bytes.  Failures are collected per run first, so that a
    failing case names every base that fails."""
    pred = np.ascontiguousarray(pred, np.float32)
    B = pred.shape[0]
    tot, seg = expected_counts(pred, num_classes, conf)
    want = orc.postprocess(pred, num_classes, conf, NMS, nthreads=8)
    cap_seg, cap_out = _pow2(max(16, seg.max())), _pow2(max(16, tot.max()))
    runs = [("base %% 16 = %d" % (4 * off), at_residue(pred, off)) for off in residues] + list(extra)
    fails, first = {}, None
    for label, x in runs:
        rows, meta = run_cabi(x, num_classes, conf, cap_seg, cap_out, groups)
        got = [rows[b, :meta[b]] if meta[b] > 0 else None for b in range(B)]
        try:
            assert np.array_equal(meta[2 * B:], tot), "candidates per image %s, literal filter %s" % (meta[2 * B:], tot)
            assert np.array_equal(meta[B:2 * B], seg), "largest segment per image %s, literal filter %s" % (meta[B:2 * B], seg)
            assert_lists_bit_equal(got, want, what="rows vs oracle")
            if first is None:
                first = got
            assert all(g is None and f is None or np.array_equal(g.view(np.uint32), f.view(np.uint32))
                       for g, f in zip(got, first)), "rows differ from the first run's bytes"
        except AssertionError as e:
            fails[label] = str(e).split("\n")[0]
    assert not fails, "%s conf %r num_classes %d: %d of %d runs fail: %s" % (what, float(conf), num_classes, len(fails), len(runs), fails)
    return want


def random_dense(B, M, C, seed, num_classes=None):
    """Overlapping boxes, about half of the rows passing the row filter at conf 0.2 (one in fifteen at C = 1), and rows aimed
    at the row filter: a NaN class inside and one outside the first num_classes, the best classes past num_classes, negative
    and NaN objectness."""
    nc = C if num_classes is None else num_classes
    rng = np.random.RandomState(seed)
    p = np.zeros((B, M, 5 + C), np.float32)
    p[..., 0:2] = rng.rand(B, M, 2) * 200
    p[..., 2:4] = 10 + rng.rand(B, M, 2) * 60
    p[..., 4] = 0.6 * rng.rand(B, M)
    p[..., 5:] = rng.rand(B, M, C) ** 6
    for b in range(B):
        r = rng.permutation(M)
        p[b, r[0], 5 + rng.randint(nc)] = np.nan
        if nc < C:
            p[b, r[1], 5 + nc + rng.randint(C - nc)] = np.nan
            p[b, r[2], 5 + nc:] = 0.99                        # passes per class, but the row filter only sees the first nc
            p[b, r[2], 4] = 0.9
        if M > 4:
            p[b, r[3], 4] = -0.5
            p[b, r[4], 4] = np.nan
    return p


# ------------------------------------------------------------------------------------------------ base residues
@pytest.mark.parametrize("conf", [1e-4, 0.2])
def test_every_base_residue_608(conf):
    """One decoded 608 image at every base residue, and as the slice dense[1:2] of a batch, which starts 7 732 620 B (12 mod
    16) into it.  B=1 at 608 also makes the aligned kernel load the last batch's three trailing floats one by one."""
    raws = synth_head_outputs(2, 608, 80, seed=21, device="cuda")
    dense = torch.cat([yb.YOLOLayer(CFG80, l, device="cuda").eval()(raws[l]) for l in range(3)], 1)
    img = dense[1:2]
    assert img.shape == (1, 22743, 85) and img.data_ptr() % 16 == 12 and (22743 * 85) % 4 == 3
    want = check_dense(img.cpu().numpy(), 80, conf, extra=[("dense[1:2]", img)], what="608")
    assert want[0] is not None and len(want[0]) > (50 if conf == 0.2 else 1000)


@pytest.mark.parametrize("conf", dec.TABLE_CONF, ids=[repr(float(c)) for c in dec.TABLE_CONF])
def test_special_value_truth_table(conf):
    """Objectness in {-inf, -1, -0, +0, 1.4e-45, 1e-30, 0.5, 1, FLT_MAX, +inf, NaN} against a class max in {-inf, -1, -0, +0,
    0.5, 1, +inf, NaN}: the row filter is obj * max >= conf literally, so 0 * inf and inf * 0 (NaN) drop a row whatever
    its other classes pass.  Image 1 holds the rows of image 0 in reverse order."""
    t = dec.truth_table()
    check_dense(np.stack([t, t[::-1]]), dec.TABLE_NUM_CLASSES, conf, what="truth table")


def _cls_for_product(obj, target):
    """A float32 cls with fl32(obj * cls) == target, or None."""
    c = np.float32(np.float64(target) / np.float64(obj))
    cands = [c]
    for d in (-np.inf, np.inf):
        x = c
        for _ in range(4):
            x = np.nextafter(x, np.float32(d))
            cands.append(x)
    for x in cands:
        if np.float32(obj * x) == target:
            return x
    return None


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_one_ulp_threshold_edges(seed):
    """conf = fl32(obj * cls) of a sampled pair (positive or negative objectness); rows whose product is conf, one ulp below
    and one ulp above it, each with its edge class at a random column and the row's other classes below it (so the edge
    class decides the row filter too)."""
    rng = np.random.RandomState(100 + seed)
    C = 5
    sign = 1 if seed % 2 == 0 else -1
    conf = np.float32(sign * rng.uniform(0.05, 1)) * np.float32(rng.uniform(1e-4, 1))
    targets = (np.nextafter(conf, np.float32(-np.inf)), conf, np.nextafter(conf, np.float32(np.inf)))
    rows = []
    for obj in (sign * rng.uniform(0.05, 1, 80)).astype(np.float32):
        for t in targets:
            cls = _cls_for_product(obj, t)
            if cls is None:
                continue
            i = len(rows)
            r = np.zeros(5 + C, np.float32)
            r[:5] = (10 + 20 * (i % 16), 10 + 20 * (i // 16), 8, 8, obj)
            r[5:] = cls * np.float32(0.5) * rng.rand(C).astype(np.float32)
            r[5 + rng.randint(C)] = cls
            rows.append(r)
    pred = np.array(rows, np.float32)
    prod = (pred[:, 4:5] * pred[:, 5:]).astype(np.float32)
    edge = prod.max(1) if sign > 0 else prod.min(1)
    for t in targets:
        assert (edge == t).sum() >= 40, "too few rows at one ulp from conf"
    check_dense(np.stack([pred, pred[::-1]]), C, conf, what="ulp edges")


# ------------------------------------------------------------------------------------------------ class counts and shapes
CLASS_COUNTS = (1, 27, 28, 59, 60, 91, 92, 123, 124, 128)


def test_class_counts_reach_every_instantiation():
    """The class counts below put 5+C on both sides of every multiple of 32: every NJ of k_filter_dense_rows, and 8, 7 and 6
    warps per CTA (two 32-row buffers per warp in 226 KB, yl_filter_dense)."""
    nj = {(5 + C + 31) // 32 for C in CLASS_COUNTS}
    warps = {min(8, (226 * 1024 - 256) // (2 * 32 * (5 + C) * 4)) for C in CLASS_COUNTS}
    assert nj == {1, 2, 3, 4, 5} and warps == {6, 7, 8}


@pytest.mark.parametrize("C,num_classes", [(C, C) for C in CLASS_COUNTS] + [(C, max(1, C // 3)) for C in CLASS_COUNTS if C > 1])
def test_every_class_count_form(C, num_classes):
    check_dense(random_dense(3, 45, C, seed=C, num_classes=num_classes), num_classes, 0.2, what="C %d" % C)


@pytest.mark.parametrize("B,M", [(11, 3), (7, 5), (3, 31), (3, 33)])
def test_batches_that_span_images(B, M):
    """M < 32 puts several images into one 32-row batch; B*M and 5+C = 25 are odd, so the tensor ends in trailing floats."""
    check_dense(random_dense(B, M, 20, seed=B * M), 20, 0.2, what="B %d M %d" % (B, M))


@pytest.mark.parametrize("k", [1, 2, 3, 4])
def test_image_groups_into_one_workspace(k):
    """yl_filter_dense on images [0, k) and [k, B) into one workspace (k*M = 13 k: a group boundary inside a 32-row batch),
    then one yl_nms over all B: the single-call result and the oracle's."""
    pred = random_dense(5, 13, 20, seed=50 + k)
    check_dense(pred, 20, 0.2, what="one call")
    check_dense(pred, 20, 0.2, groups=[(0, k), (k, 5 - k)], what="groups [0,%d) [%d,5)" % (k, k))


# ------------------------------------------------------------------------------------------------ capacity, num_classes
def test_overflowing_segments_keep_exact_counts_and_postprocess_grows():
    """All ties: every row passes in every class, 1500 candidates per (image, class) segment, far past cap_seg = 64 and past
    postprocess's first cap_seg of 1024."""
    B, M, C = 2, 1500, 3
    i = np.arange(M)
    pred = np.zeros((B, M, 5 + C), np.float32)
    pred[..., 0], pred[..., 1], pred[..., 2:4], pred[..., 4:] = 4 * (i % 50), 4 * (i // 50), 12, 0.5   # IoU 0.5 side by side
    want = orc.postprocess(pred, C, 0.2, NMS, nthreads=8)
    for off in RESIDUES:
        x = at_residue(pred, off)
        _, meta = run_cabi(x, C, 0.2, 64, 1024)
        assert meta[B:2 * B].tolist() == [M] * B and meta[2 * B:].tolist() == [C * M] * B, f"base % 16 = {4 * off}"
        assert_lists_bit_equal(yb.postprocess(x, C, 0.2, NMS), want, what=f"postprocess, base % 16 = {4 * off}")
        assert importlib.import_module("yolov4_b200.postprocess")._cap_hint[(B, M, C)][0] >= M   # the cap_seg it settled on


def test_num_classes_above_C_means_C():
    """The reference slices image_pred[:, 5:5 + num_classes], which stops at the row's end."""
    B, M, C = 2, 40, 6
    pred = random_dense(B, M, C, seed=9)
    want = orc.postprocess(pred, C, 0.2, NMS)
    for off in (0, 1):
        x = at_residue(pred, off)
        same = [None if r is None else r.cpu().numpy() for r in yb.postprocess(x, C, 0.2, NMS)]
        assert_lists_bit_equal(same, want, what="num_classes = C")
        assert_lists_bit_equal(yb.postprocess(x, C + 7, 0.2, NMS), same, what="num_classes = C + 7")
        with pytest.raises(_cabi.YoloHeadError):
            yb.postprocess(x, 0, 0.2, NMS)

"""The NMS back end (everything yl_nms_ex2 launches after the filter: k_segment_nms_bins, k_segment_nms_big, k_select_topk,
k_segment_nms_agnostic, k_gather_rows) at exact IoU decisions, across box scales, on every tier and routing branch.

Every case runs through the C ABI (yl_post_reset, yl_filter_dense, then yl_nms_ex2 per image group) into a rows buffer filled
with a canary, and checks:
  * rows [0, min(K_b, cap_out)) of every image are those of the literal fp32 NMS bit for bit (the C oracle per class,
    diou_spec for DIoU, agnostic_spec for agnostic, cap_spec on top for max_det), the rest of the image's slot and everything
    past the buffer's end still hold the canary, meta[b] = K_b and meta[B+b], meta[2B+b] are the literal filter's counts;
  * tier routing, read from the workspace (post_layout of yl_common.cuh, restated in nms_edge_cases.layout): big_count of the
    group (at its first image) and big_list list exactly the segments the small tier must pass on (more than 256 records,
    !(thr > 0), or a warp's pair queue over 512 pairs), so each case provably reaches the tier it is named for."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from yolov4_b200 import _cabi                                         # noqa: E402

import agnostic_spec                                                  # noqa: E402
import cap_spec                                                       # noqa: E402
import diou_spec                                                      # noqa: E402
import nms_edge_cases as nec                                          # noqa: E402
from oracle import oracle as orc                                      # noqa: E402  (checker only)
from test_gpu_parity import bit_equal                                 # noqa: E402

F32 = np.float32
CANARY = 0x7FC0DEAD                                                   # a NaN no kernel writes
PAD = 64                                                              # canary words past the rows buffer
VARIANTS = ("iou", "diou", "agnostic", "max_det")
FRESH = os.environ.get("YL_NMS_BACK_END_FRESH") == "1"


def _pow2(n):
    p = 1
    while p < n:
        p <<= 1
    return p


def run_cabi(pred, thr, cap_seg, cap_out, groups, diou=0, agnostic=0, max_det=0):
    """One yl_filter_dense over the batch, then yl_nms_ex2 per (img_first, img_count) group into one workspace.  Returns (rows
    [B*cap_out*7 + PAD] uint32, meta [3B], {img_first: sorted big_list entries of the group})."""
    B, M, nch = pred.shape
    C = nch - 5
    L = _cabi.lib()
    nb = L.yl_post_workspace_bytes_ex(B, M, C, cap_seg, agnostic)
    ws = torch.zeros(nb, dtype=torch.uint8, device="cuda")
    x = torch.from_numpy(np.ascontiguousarray(pred)).cuda()
    rows = torch.full((B * cap_out * 7 + PAD,), CANARY, dtype=torch.int32, device="cuda")
    meta = torch.full((3 * B,), -7, dtype=torch.int32, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    _cabi.check(L.yl_post_reset(ws.data_ptr(), nb, B, M, C, cap_seg, st))
    _cabi.check(L.yl_filter_dense(x.data_ptr(), B, M, C, C, float(nec.CONF), ws.data_ptr(), nb, cap_seg, 0, B, st))
    for i0, n in groups:
        _cabi.check(L.yl_nms_ex2(ws.data_ptr(), nb, B, M, C, cap_seg, float(thr), max_det, agnostic, diou, rows.data_ptr(), cap_out,
                                 meta.data_ptr(), None, i0, n, st))
    torch.cuda.synchronize()
    w = ws.cpu().numpy()
    lay = nec.layout(B, M, C, cap_seg)
    big = {}
    for i0, _ in groups:
        cnt = int(w[lay["big_count"] + 4 * i0:lay["big_count"] + 4 * i0 + 4].view(np.uint32)[0])
        assert cnt <= B * C, "big_count of group %d: %d" % (i0, cnt)
        o = lay["big_list"] + 4 * i0 * C
        big[i0] = sorted(w[o:o + 4 * cnt].view(np.uint32).tolist())
    return rows.cpu().numpy().view(np.uint32), meta.cpu().numpy(), big


def expected_rows(pred, thr, variant, max_det=0):
    C = pred.shape[2] - 5
    if variant == "diou":
        return diou_spec.postprocess(pred, C, nec.CONF, thr)
    if variant == "agnostic":
        return agnostic_spec.postprocess(pred, C, nec.CONF, thr)
    want = orc.postprocess(pred, C, nec.CONF, thr, nthreads=8)
    return cap_spec.cap_detections(want, max_det) if max_det else want


def expected_big(pred, thr, cap_seg, groups):
    """{img_first: sorted segment ids} the small tier must pass on (nec.must_go_big), per group."""
    C = pred.shape[2] - 5
    out = {}
    for i0, n in groups:
        segs = []
        for b in range(i0, i0 + n):
            cand = agnostic_spec.candidates(pred[b], C, nec.CONF)
            for c in np.unique(cand["cls"]):
                sel = np.nonzero(cand["cls"] == c)[0]
                box = cand["box"][sel[np.lexsort((-cand["row"][sel], -cand["s"][sel]))]]
                if nec.must_go_big(box, thr, cap_seg):
                    segs.append(b * C + int(c))
        out[i0] = sorted(segs)
    return out


def check(pred, thr, variant="iou", cap_seg=None, cap_out=None, groups=None, what=""):
    """Runs pred at thr through the variant (with max_det: once per distinct value K_b - 1) and asserts rows, canaries, meta and
    routing.  Returns ({img_first: big_list} of the last run, the uncapped oracle rows)."""
    pred = np.ascontiguousarray(pred, np.float32)
    B, C = pred.shape[0], pred.shape[2] - 5
    tot, seg = [], []
    for p in pred:
        cls = agnostic_spec.candidates(p, C, nec.CONF)["cls"]
        tot.append(len(cls))
        seg.append(int(np.bincount(cls).max()) if len(cls) else 0)
    cap_seg = cap_seg or _pow2(max(16, max(seg)))
    groups = groups or [(0, B)]
    base = expected_rows(pred, thr, "iou" if variant == "max_det" else variant)
    kept = [0 if r is None else len(r) for r in base]
    cap_out = cap_out or max(16, max(kept) + 3)
    runs = [(0, base)]
    if variant == "max_det":
        runs = [(m, cap_spec.cap_detections(base, m)) for m in sorted({max(1, k - 1) for k in kept})]
    want_big = expected_big(pred, thr, cap_seg, groups) if variant != "agnostic" else {i0: [] for i0, _ in groups}
    for max_det, want in runs:
        rows, meta, big = run_cabi(pred, thr, cap_seg, cap_out, groups, diou=int(variant == "diou"),
                                   agnostic=int(variant == "agnostic"), max_det=max_det)
        tag = "%s thr %r %s max_det %d:" % (what, float(thr), variant, max_det)
        img = rows[:B * cap_out * 7].reshape(B, cap_out, 7)
        for b in range(B):
            k = 0 if want[b] is None else len(want[b])
            assert meta[b] == k, "%s image %d: meta[b] %d, literal NMS %d" % (tag, b, meta[b], k)
            assert meta[B + b] == seg[b] and meta[2 * B + b] == tot[b], "%s image %d: meta %s" % (tag, b, meta)
            nw = min(k, cap_out)
            if nw:
                got = img[b, :nw].copy().view(np.float32)
                if not bit_equal(got, want[b][:nw]):
                    bad = np.argwhere(~((got.view(np.uint32) == want[b][:nw].view(np.uint32)) | (np.isnan(got) & np.isnan(want[b][:nw]))))
                    raise AssertionError("%s image %d: %d words differ, first row %d: %s vs %s" % (
                        tag, b, len(bad), bad[0][0], got[bad[0][0]], want[b][bad[0][0]]))
            assert (img[b, nw:] == CANARY).all(), "%s image %d: rows past %d were written" % (tag, b, nw)
        assert (rows[B * cap_out * 7:] == CANARY).all(), "%s written past the rows buffer" % tag
        assert big == want_big, "%s segments passed to the big tier %s, must be %s" % (tag, big, want_big)
    return big, base


def _variant_params(variants=VARIANTS):
    return pytest.mark.parametrize("variant", variants)


# ------------------------------------------------------------------------------------------------ exact decisions x scales
PAIR_CASES = [(n, side, tier) for n in nec.BASE_PAIRS for side in ("q", "below", "above") for tier in nec.FILLER]


@pytest.mark.parametrize("name,side,tier", PAIR_CASES, ids=["%s-%s-%s" % c for c in PAIR_CASES])
def test_exact_pair_on_every_scale(name, side, tier):
    """The pair's literal IoU q at scale 1 as the threshold, and one ulp either side; one copy per segment at scales 2^-80 ..
    2^67 (subnormal areas and intersections, both area-bin clamps, the +-1e6 coordinate clamp, overflowing areas and unions).
    With filler, the segments exceed 256 (big tier, shared memory) or 1024 records (global memory, cap_seg 2048)."""
    images, C, where = nec.pair_images(name, tier)
    q, thrs = nec.pair_threshold(name)
    thr = thrs[side]
    pred = nec.make_pred(images, C, seed=len(name))
    cap_seg = {"small": 16, "big": 512, "global": 2048}[tier]
    big, want = check(pred, thr, cap_seg=cap_seg, what="%s %s" % (name, tier))
    n_big = sum(len(v) for v in big.values())
    assert n_big == (0 if tier == "small" and thr > 0 else len(where)), "tier %s reached by %d segments" % (tier, n_big)
    # at scale 1 the pair decides as q says: at q and below it B is suppressed, above it B is kept (at thr <= 0 every box of
    # the segment has IoU >= thr with the first one)
    b1, c1 = [bc for bc, k in where.items() if k == 0][0]
    rows1 = want[b1][want[b1][:, 6] == c1]
    assert len(rows1) == (len(nec.BASE_PAIRS[name][2]) + nec.FILLER[tier] + (1 if side != "above" else 2) if thr > 0 else 1)


@pytest.mark.parametrize("variant", ("diou", "agnostic", "max_det"))
@pytest.mark.parametrize("name,side", [(n, s) for n in nec.BASE_PAIRS for s in ("q", "below", "above")])
def test_exact_pair_variants(name, side, variant):
    """The small-tier pair segments again with the DIoU decision, class-agnostic NMS and a detection cap of K_b - 1."""
    images, C, _ = nec.pair_images(name, "small")
    thr = nec.pair_threshold(name)[1][side]
    check(nec.make_pred(images, C, seed=len(name)), thr, variant, cap_seg=16, what=name)


# ------------------------------------------------------------------------------------------------ area-bin gaps
GAP_THRESHOLDS = nec.gap_change_thresholds() + nec.gap_pair_thresholds()


@pytest.mark.parametrize("thr", GAP_THRESHOLDS, ids=["%.9g" % t for t in GAP_THRESHOLDS])
def test_area_bin_gap_pairs(thr):
    """Contained pairs at the tightest spot of area-bin gaps K - 1, K and K + 1 (K = area_bin_gap(thr)) at each in-octave
    position, at thresholds on both sides of every change of K and at the IoU of each gap's tightest pair."""
    images, C, _ = nec.area_gap_images(thr)
    check(nec.make_pred(images, C), thr, cap_seg=16, what="area gaps")


# ------------------------------------------------------------------------------------------------ thresholds
def threshold_case():
    """Two images: the base pairs, a scattered segment, a tie segment, a queue cluster, invalid boxes and identical boxes (in
    one bin because of a tiny range and because of the +-1e6 clamp)."""
    img0 = {}
    for c, name in enumerate(nec.BASE_PAIRS):
        a, b, anchors = nec.BASE_PAIRS[name]
        img0[c] = ([a, b] + list(anchors), nec.descending_scores(2 + len(anchors)))
    img1 = {0: nec.routing_segment(90, 3), 1: nec.tie_segment(40, 4), 2: nec.queue_cluster(1), 3: nec.invalid_segment(),
            4: nec.identical_segment(40, "tiny"), 5: nec.identical_segment(40, "huge")}
    return nec.make_pred([img0, img1], len(nec.BASE_PAIRS), seed=5)


THR_CASE = None


@_variant_params()
@pytest.mark.parametrize("thr", nec.THRESHOLDS, ids=[repr(float(t)) for t in nec.THRESHOLDS])
def test_threshold_classes(thr, variant):
    """Every threshold class (subnormal, tiny, ordinary, near 1, 1, above 1, inf, +-0, negative, NaN): !(thr > 0) sends every
    segment to the big tier's literal formula, the others stay in the small tier."""
    global THR_CASE
    if THR_CASE is None:
        THR_CASE = threshold_case()
    big, _ = check(THR_CASE, thr, variant, what="threshold classes")
    if variant != "agnostic":
        n_seg = len(nec.BASE_PAIRS) + 6
        assert sum(len(v) for v in big.values()) == (n_seg if not thr > 0 else 0)


# ------------------------------------------------------------------------------------------------ routing sizes
SIZES = (1, 2, 63, 64, 65, 127, 128, 129, 255, 256, 257, 1023, 1024, 1025)


@_variant_params()
@pytest.mark.parametrize("cap", ("n", "pow2"))
@pytest.mark.parametrize("n", SIZES)
def test_segment_sizes(n, cap, variant):
    """A segment of n records beside one of up to 3, with cap_seg = n and a power of two above n: the small tier up to 256, the
    big tier in shared memory up to 1024, in global memory beyond (where kept_scratch exists only because cap_seg > 1024)."""
    pred = nec.make_pred([{0: nec.routing_segment(n, n), 1: nec.routing_segment(min(n, 3), 7)}], 2, seed=n)
    cap_seg = n if cap == "n" else _pow2(n + 1)
    big, _ = check(pred, F32(0.45), variant, cap_seg=cap_seg, what="n %d cap_seg %d" % (n, cap_seg))
    if variant != "agnostic":
        assert big == {0: [0] if n > nec.SMALL_R else []}


@_variant_params()
@pytest.mark.parametrize("n", (130, 200, 256))
def test_score_ties_across_record_128(n, variant):
    """Pairs of overlapping boxes sharing a score, all along the order: the split rank (records 128 and up) collides and the
    64-bit (score, row) re-rank decides which box of each pair is kept."""
    big, _ = check(nec.make_pred([{0: nec.tie_segment(n, n)}], 1, seed=n), F32(0.45), variant, what="ties n %d" % n)
    if variant != "agnostic":
        assert big == {0: []}


@_variant_params()
@pytest.mark.parametrize("pairs", (512, 513))
def test_pair_queue_boundary(pairs, variant):
    """One warp's queue holds exactly 512 candidate pairs (the small tier resolves the segment) or 513 (it overflows and the
    big tier takes the segment)."""
    boxes, scores = nec.queue_cluster(pairs - 511)
    assert nec.small_tier_queues(boxes, F32(0.45))[0] == pairs
    big, _ = check(nec.make_pred([{0: (boxes, scores), 1: nec.routing_segment(20, 1)}], 2, seed=pairs), F32(0.45), variant,
                   what="queue %d" % pairs)
    if variant != "agnostic":
        assert big == {0: [0] if pairs > nec.QCAP_W else []}


# ------------------------------------------------------------------------------------------------ output shape
def truncation_case():
    """Three images of four classes, up to 16 records per segment (cap_seg 16: the gather's speculative loads stop at 32
    float4), different kept totals."""
    images = []
    for b, sizes in enumerate(((5, 16, 9, 3), (16, 2, 0, 11), (7, 7, 7, 1))):
        images.append({c: nec.routing_segment(n, 10 * b + c) for c, n in enumerate(sizes) if n})
    return nec.make_pred(images, 4, seed=9)


CAP_OUT_CASES = ("first_row", "inside_class", "last_row", "kept", "above")


@_variant_params(("iou", "diou", "max_det"))
@pytest.mark.parametrize("groups", ("one_call", "groups"))
@pytest.mark.parametrize("where", CAP_OUT_CASES)
def test_cap_out_truncation(where, groups, variant):
    """cap_out on the first row, inside image 0's second class segment, on its last kept row, equal to it and above every
    image's total; meta[b] stays the true count and nothing past cap_out is written.  "groups": yl_nms_ex2 once per image
    group ([0, 1) and [1, 3)) into one workspace, so the second group's big_count lives at image 1."""
    pred = truncation_case()
    want = orc.postprocess(pred, 4, nec.CONF, F32(0.45), nthreads=4)
    k0 = len(want[0])
    c0 = int((want[0][:, 6] == want[0][0, 6]).sum())
    cap_out = {"first_row": 1, "inside_class": c0 + 1, "last_row": k0 - 1, "kept": k0,
               "above": max(len(w) for w in want) + 3}[where]
    assert 1 <= cap_out and (where != "inside_class" or c0 + 1 < k0)
    if variant == "max_det":
        # max_det <= cap_out is the ABI's rule: the cap runs at K_b - 1 wherever that fits
        ks = sorted({len(w) - 1 for w in want if 1 <= len(w) - 1 <= cap_out}) or [1]
        for m in ks:
            _check_capped(pred, m, cap_out, groups)
        return
    check(pred, F32(0.45), variant, cap_seg=16, cap_out=cap_out, groups=[(0, 3)] if groups == "one_call" else [(0, 1), (1, 2)],
          what="cap_out %d" % cap_out)


def _check_capped(pred, max_det, cap_out, groups):
    B = pred.shape[0]
    want = cap_spec.cap_detections(orc.postprocess(pred, 4, nec.CONF, F32(0.45), nthreads=4), max_det)
    rows, meta, _ = run_cabi(pred, F32(0.45), 16, cap_out, [(0, 3)] if groups == "one_call" else [(0, 1), (1, 2)], max_det=max_det)
    img = rows[:B * cap_out * 7].reshape(B, cap_out, 7)
    for b in range(B):
        k = len(want[b])
        assert meta[b] == k
        nw = min(k, cap_out)
        assert bit_equal(img[b, :nw].copy().view(np.float32), want[b][:nw]), "max_det %d image %d" % (max_det, b)
        assert (img[b, nw:] == CANARY).all()
    assert (rows[B * cap_out * 7:] == CANARY).all()


# ------------------------------------------------------------------------------------------------ without PDL
def test_without_pdl_in_a_fresh_process():
    """The four back-end kernels form a PDL chain: the threshold, size, tie, queue and truncation cases again in a fresh process
    with YL_PDL=0 (read when the library loads) must give the same bytes, which the checks above pin to the literal NMS."""
    if FRESH:
        pytest.skip("already in the fresh process")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, YL_PDL="0", YL_NMS_BACK_END_FRESH="1")
    p = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider", os.path.abspath(__file__),
                        "-k", "threshold_classes or segment_sizes or ties or queue_boundary or truncation"],
                       cwd=root, env=env, capture_output=True, text=True, timeout=1500)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-2000:]
    passed = re.search(r"(\d+) passed", p.stdout)
    assert passed and int(passed.group(1)) >= 200 and "skipped" not in p.stdout, p.stdout[-1000:]

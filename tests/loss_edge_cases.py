"""Hostile label sets for build_target and the fused loss, shared by the CPU spec test and the GPU tests.

Every case is a dict: name, C, img, labels [B,K,5] fp32 (pixels), raws (three numpy heads [B,3(5+C),F,F]), mask (ANCHOR_MASK),
thrs (ignore thresholds) and error.  `error` cases hold a matched GT that the reference's
indexing rejects (IndexError): only that is checked on them.  Coordinates stay within +-32767 grid units, where the
reference's float -> int16 cast is defined.
"""
import functools

import numpy as np

from oracle import oracle as orc
from yolov4_b200.synth import synth_head_outputs

ALT_MASK = [[2, 1, 0], [5, 4, 3], [8, 7, 6]]
# box sizes (px) whose best anchor is 1, 4 and 7 of the default anchors: one per layer
SIZES = [(20.0, 30.0), (70.0, 60.0), (190.0, 240.0)]


def heads(B, img, C, seed, fg_prob=0.05):
    return [r.numpy().copy() for r in synth_head_outputs(B, img, C, seed=seed, fg_prob=fg_prob, clustered=True)]


def plant_box(raws, C, mask, b, layer, a, box_px):
    """Sets the tx, ty, tw, th logits of image b, slot a of `layer` at the cell holding the box centre so that the decoded
    train-mode box is close to box_px (xc, yc, w, h); boxes outside the grid are skipped."""
    raw = raws[layer]
    F, s = raw.shape[2], float(orc.STRIDES[layer])
    x, y, w, h = (float(v) for v in box_px)
    if not all(np.isfinite([x, y, w, h])) or w <= 0 or h <= 0 or not (0 <= x < F * s and 0 <= y < F * s):
        return
    i, j = int(x / s), int(y / s)
    anc = orc.masked_anchors_grid(layer, orc.ANCHORS_PX, mask)[a]
    fx, fy = [min(max(v, 0.02), 0.98) for v in (x / s - i, y / s - j)]
    nch = 5 + C
    raw[b, a * nch + 0, j, i] = np.log(fx / (1 - fx))
    raw[b, a * nch + 1, j, i] = np.log(fy / (1 - fy))
    raw[b, a * nch + 2, j, i] = np.log(w / s / anc[0])
    raw[b, a * nch + 3, j, i] = np.log(h / s / anc[1])


def plant_near_gts(raws, labels, C, mask, every=2):
    """Predictions planted on / near every `every`-th GT on all three layers: non-trivial ignore masks."""
    for b in range(labels.shape[0]):
        for t in range(0, labels.shape[1], every):
            if labels[b, t].sum() > 0:
                box = labels[b, t, :4] * np.float32(1.0 + 0.02 * (t % 5))
                box[:2] = labels[b, t, :2]
                for l in range(3):
                    plant_box(raws, C, mask, b, l, t % 3, box)


def case(name, C, img, labels, raws, mask=orc.ANCHOR_MASK, thrs=(0.7,), error=False):
    return dict(name=name, C=C, img=img, labels=np.ascontiguousarray(labels, np.float32), raws=raws, mask=mask,
                thrs=tuple(thrs), error=error)


class _Cells:
    """Hands out distinct cells per layer, so that boxes meant to be alone on their cell are."""

    def __init__(self, img):
        self.img, self.next = img, [0, 0, 0]

    def centre(self, layer, fx=0.37, fy=0.61):
        s = orc.STRIDES[layer]
        F = self.img // s
        k = self.next[layer]
        self.next[layer] += 1
        q = (k * 7) % (F * F)
        assert k < F * F, "out of cells"
        return ((q % F) + fx) * s, ((q // F) + fy) * s


def class_id_rows(C, img, ids, seed=0):
    """Every id on an isolated cell, as the last GT of a collided cell and as a non-last GT of one.  The two GTs of a collided
    cell are 40 rows apart, so different slices of the kernels own them."""
    rng = np.random.RandomState(seed)
    cells = _Cells(img)
    iso, first, second = [], [], []
    for k, cid in enumerate(ids):
        l = k % 3
        w, h = SIZES[l]
        x, y = cells.centre(l)
        iso.append((x, y, w, h, cid))
        for last in (True, False):
            x, y = cells.centre(l, 0.2 + 0.6 * rng.rand(), 0.2 + 0.6 * rng.rand())
            partner = (x + 0.05 * orc.STRIDES[l], y, w * 1.04, h * 0.97, float(k % C))
            mine = (x, y, w, h, cid)
            first.append(partner if last else mine)
            second.append(mine if last else partner)
    filler = []
    while len(first) + len(filler) < 40:
        x, y = cells.centre(0, 0.5, 0.5)
        filler.append((x, y, 12.0, 14.0, float(len(filler) % C)))
    return iso + first + filler + second


def labels_of(rows_per_image, K):
    B = len(rows_per_image)
    lab = np.zeros((B, K, 5), np.float32)
    for b, rows in enumerate(rows_per_image):
        lab[b, :len(rows)] = np.array(rows, np.float32)
    return lab


def class_ids(C=4, img=160, seed=11):
    """Every class id in [-(10+C), -1], fractional ids, and the ordinary ones."""
    ids = [float(v) for v in range(-(10 + C), 0)] + [2.7, -0.5, 0.0, float(C - 1)]
    rows = class_id_rows(C, img, ids, seed)
    lab = labels_of([rows, rows[::-1]], len(rows) + 8)
    raws = heads(2, img, C, seed)
    plant_near_gts(raws, lab, C, orc.ANCHOR_MASK, every=3)
    return case("class_ids_C%d" % C, C, img, lab, raws)


def bad_class(cid, C=4, img=96, seed=12):
    """One matched GT whose class id indexes outside the target row."""
    rows = [(30.0, 40.0, 20.0, 30.0, 1.0), (50.5, 60.5, 20.0, 30.0, cid), (70.0, 20.0, 70.0, 60.0, 2.0)]
    return case("bad_class_%g" % cid, C, img, labels_of([rows], 6), heads(1, img, C, seed), error=True)


def collisions(C=6, img=96, seed=13):
    """41 GTs of mixed (also negative) classes on one cell of layer 0 (two-word ballots), pairs on other cells, and a second
    image whose 16 GTs all share one layer-1 cell."""
    rng = np.random.RandomState(seed)
    ids = list(range(-(10 + C), C))
    rows = []
    for k in range(41):
        rows.append((44.5 + rng.rand() * 3, 27.0 + rng.rand() * 3, 20.0 * (1 + 0.002 * k), 30.0, float(ids[k % len(ids)])))
        if k % 4 == 0:
            rows.append((8.0 + 16 * (k // 8), 84.0, 18.0, 28.0, float(ids[(5 * k) % len(ids)])))
    rows2 = [(50.0 + 0.3 * k, 40.0, 70.0, 60.0, float(ids[(3 * k) % len(ids)])) for k in range(16)]
    lab = labels_of([rows, rows2], 64)
    raws = heads(2, img, C, seed)
    plant_near_gts(raws, lab, C, orc.ANCHOR_MASK, every=5)
    return case("collisions", C, img, lab, raws)


def full_k256(C=5, img=96, seed=14):
    """K = 256 label slots, every one used: random boxes of all sizes and classes in [-(10+C), C)."""
    rng = np.random.RandomState(seed)
    lab = np.zeros((2, 256, 5), np.float32)
    lab[..., 0:2] = rng.uniform(0, img, (2, 256, 2))
    lab[..., 2:4] = np.exp(rng.uniform(np.log(3.0), np.log(110.0), (2, 256, 2)))
    lab[..., 4] = rng.randint(-(10 + C), C, (2, 256))
    raws = heads(2, img, C, seed)
    plant_near_gts(raws, lab, C, orc.ANCHOR_MASK, every=7)
    return case("full_k256", C, img, lab, raws, thrs=(0.7, 0.3))


def first_n_rows(C=3, img=128, seed=15):
    """Zero rows and rows with a sum <= 0 among the first n (n counts the rows with a sum > 0, the first n rows are used)."""
    r0 = [(30.0, 40.0, 20.0, 30.0, 1.0), (60.0, 70.0, 70.0, 60.0, 2.0), (0.0, 0.0, 0.0, 0.0, 0.0),
          (-50.0, -30.0, 20.0, 30.0, 2.0), (90.0, 20.0, 20.0, 30.0, 0.0), (0.0, 0.0, 0.0, 0.0, 0.0),
          (100.0, 100.0, 18.0, 25.0, 1.0), (-80.0, 40.0, 30.0, 5.0, 0.0), (20.0, 110.0, 20.0, 30.0, 2.0)]
    r1 = [(0.0, 0.0, 0.0, 0.0, 0.0), (-10.0, -10.0, 5.0, 5.0, 1.0), (64.0, 64.0, 20.0, 30.0, 1.0),
          (30.0, 30.0, 70.0, 60.0, 0.0), (0.0, 0.0, 0.0, 0.0, 0.0), (100.0, 60.0, 20.0, 30.0, 2.0)]
    lab = labels_of([r0, r1], 12)
    raws = heads(2, img, C, seed)
    plant_near_gts(raws, lab, C, orc.ANCHOR_MASK)
    return case("first_n_rows", C, img, lab, raws)


def geometry(C=3, img=160, seed=16):
    """Centres on cell edges, at 0 and one ulp below the image size, negative centres (a negative xy target, and one that
    wraps to the far side of the grid), boxes of 1e-3 px."""
    below = float(np.nextafter(np.float32(img), np.float32(0)))
    rows = [(8.0, 16.0, 20.0, 30.0, 0.0), (32.0, 64.0, 70.0, 60.0, 1.0), (64.0, 96.0, 190.0, 240.0, 2.0),
            (0.0, 0.0, 20.0, 30.0, 1.0), (0.0, 50.0, 70.0, 60.0, 2.0), (0.0, 0.0, 190.0, 240.0, 0.0),
            (below, below, 20.0, 30.0, 2.0), (below, 3.0, 70.0, 60.0, 0.0), (below, below, 190.0, 240.0, 1.0),
            (-5.0, 50.0, 20.0, 30.0, 0.0), (50.0, -3.0, 70.0, 60.0, 1.0), (-20.0, 60.0, 20.0, 30.0, 2.0),
            (70.0, -40.0, 70.0, 60.0, 0.0), (-60.0, 60.0, 190.0, 240.0, 1.0),
            (77.7, 33.3, 1e-3, 1e-3, 1.0), (120.2, 99.9, 1e-3, 2e-3, 2.0), (40.0, 140.0, 1e-3, 40.0, 0.0)]
    lab = labels_of([rows], 20)
    raws = heads(1, img, C, seed)
    plant_near_gts(raws, lab, C, orc.ANCHOR_MASK)
    return case("geometry", C, img, lab, raws, thrs=(0.7, 0.0))


def out_of_grid(C=3, img=160, seed=17):
    """A matched centre at exactly the image size: one past the last cell."""
    rows = [(50.0, 50.0, 20.0, 30.0, 0.0), (float(img), 70.0, 20.0, 30.0, 1.0)]
    return case("out_of_grid", C, img, labels_of([rows], 4), heads(1, img, C, seed), error=True)


def huge_box(C=3, img=160, seed=18):
    """w h > 2 F^2 on layer 2 (5x5 at 160 px): tgt_scale = sqrt(negative) = NaN."""
    rows = [(80.0, 80.0, 300.0, 300.0, 1.0), (30.0, 40.0, 20.0, 30.0, 0.0), (100.0, 60.0, 70.0, 60.0, 2.0)]
    return case("huge_box", C, img, labels_of([rows], 4), heads(1, img, C, seed))


def degenerate(C=8, img=160, seed=5):
    """The zero / negative / inf / 1e30 / NaN extents of the pathological build_target test among ordinary boxes."""
    B, K, n = 2, 16, 12
    rng = np.random.RandomState(seed)
    lab = np.zeros((B, K, 5), np.float32)
    for b in range(B):
        lab[b, :n, 0:2] = rng.uniform(4, img - 4, (n, 2))
        lab[b, :n, 2:4] = np.exp(rng.uniform(np.log(4.0), np.log(img * 0.8), (n, 2)))
        lab[b, :n, 4] = rng.randint(0, 8, n)
    lab[0, 2, 2:4] = lab[0, 1, 2:4]
    lab[1, 1, 2] = np.inf
    lab[1, 4, 3] = 1e30
    lab[1, 5, 2] = 0.0
    lab[0, 6, 2] = -20.0
    lab[0, 7, 2:4] = (-20.0, -30.0)
    lab[1, 8, 3] = np.nan
    raws = heads(B, img, C, seed)
    plant_near_gts(raws, lab, C, orc.ANCHOR_MASK)
    return case("degenerate", C, img, lab, raws, thrs=(0.7, 0.0))


def mixed(C, img=128, seed=19, mask=orc.ANCHOR_MASK, B=2, n=24, thrs=(0.7,), name=None):
    """Ordinary boxes of all sizes with classes in [-(10+C), C), a few collisions, predictions planted near the GTs."""
    rng = np.random.RandomState(seed)
    lab = np.zeros((B, n + 4, 5), np.float32)
    lab[:, :n, 0:2] = rng.uniform(1, img - 1, (B, n, 2))
    lab[:, :n, 2:4] = np.exp(rng.uniform(np.log(4.0), np.log(img * 1.5), (B, n, 2)))
    lab[:, :n, 4] = rng.randint(-(10 + C), C, (B, n))
    lab[:, 5, :4] = lab[:, 1, :4]                         # collisions 4 and 8 rows apart
    lab[:, 9, :4] = lab[:, 1, :4] * np.float32(1.01)
    lab[:, 9, :2] = lab[:, 1, :2]
    raws = heads(B, img, C, seed)
    plant_near_gts(raws, lab, C, mask)
    return case(name or "mixed_C%d" % C, C, img, lab, raws, mask=mask, thrs=thrs)


def ignore_thresholds(C=4, img=160, seed=20):
    return mixed(C, img, seed, thrs=(0.7, 0.3, 0.0, -0.5, 1.0), name="ignore_thresholds")


def _boundary_scene(C, img, seed, contained):
    """One GT on layer 0 and a prediction at the same cell in another anchor slot (not matched), with a large objectness
    logit: the prediction either overlaps the GT or contains it.  Returns (labels, raws, (b, a, j, i), v) with v the fp32
    IoU of the decoded prediction and the GT, as the ignore test computes it."""
    gt = np.array([75.3, 83.1, 22.0, 33.0], np.float32)
    lab = labels_of([[tuple(gt) + (1.0,)]], 2)
    raws = heads(1, img, C, seed, fg_prob=0.0)
    s = np.float32(8)
    out, pred = orc.decode_train(raws[0], 0, C)
    target, _, tgt_mask, _ = orc.build_target(pred, lab, 0, C, 0.7)
    ga, gj, gi = [int(v[0]) for v in np.nonzero(tgt_mask[0, ..., 0])]
    a = (ga + 1) % 3
    box = gt * np.float32(1.6 if contained else 1.08)
    box[:2] = gt[:2] + (np.float32(0.0) if contained else np.float32(1.3))
    plant_box(raws, C, orc.ANCHOR_MASK, 0, 0, a, box)
    raws[0][0, a * (5 + C) + 4, gj, gi] = 6.0
    _, pred = orc.decode_train(raws[0], 0, C)
    v = orc.bboxes_iou(pred[0, a, gj, gi][None], (gt / s)[None], xyxy=False)[0, 0]
    return lab, raws, (0, a, gj, gi), np.float32(v)


def ignore_boundary(contained, C=4, img=160, seed=21):
    """thr = v keeps the planted cell (IoU > thr is false), thr = the float below v ignores it.  With the GT inside the
    prediction, IoU is the area ratio and thresholds around ratio / 0.99 put the GT at the edge of the ignore test's
    area run."""
    lab, raws, cell, v = _boundary_scene(C, img, seed, contained)
    thrs = [v, np.nextafter(v, np.float32(-np.inf))]
    if contained:
        e = np.float32(v / np.float32(0.99))
        thrs += [e, np.nextafter(e, np.float32(-np.inf)), np.nextafter(e, np.float32(np.inf))]
    c = case("ignore_boundary_%s" % ("contained" if contained else "overlap"), C, img, lab, raws,
             thrs=[float(t) for t in thrs])
    c["cell"], c["v"] = cell, v
    return c


def with_special_logits(c, seed=22):
    """Special logits planted where the reference's value is defined: +-17 / +-88 / +-104 / +-inf in every channel of matched
    cells except +-inf in tw / th (an infinite wh term), +-104 / +-inf in the objectness of ignored and plain cells, and NaN
    in the objectness of one plain cell.  (A non-finite box or class logit at an unmatched cell, or NaN at an ignored one,
    becomes NaN * 0 in the reference's masked products, which the fused loss never forms: those cells contribute exactly 0
    there.)"""
    rng = np.random.RandomState(seed)
    C, mask, lab = c["C"], c["mask"], c["labels"]
    nch = 5 + C
    vals = np.array([17, -17, 88, -88, 104, -104, np.inf, -np.inf], np.float32)
    raws = [r.copy() for r in c["raws"]]
    for l, raw in enumerate(raws):
        _, pred = orc.decode_train(raw, l, C, mask=mask)
        _, obj_mask, tgt_mask, _ = orc.build_target(pred, lab, l, C, c["thrs"][0], mask=mask)
        matched = tgt_mask[..., 0] == 1
        ignored = (obj_mask == 0) & ~matched
        for b, a, j, i in np.argwhere(matched):
            for ch in range(nch):
                v = vals[rng.randint(len(vals))]
                if ch in (2, 3) and not np.isfinite(v):
                    v = np.float32(104.0 if v > 0 else -104.0)
                raw[b, a * nch + ch, j, i] = v
        for b, a, j, i in np.argwhere(ignored):
            raw[b, a * nch + 4, j, i] = vals[4 + rng.randint(4)]
        plain = np.argwhere(~matched & (obj_mask == 1))
        for b, a, j, i in plain[rng.choice(len(plain), min(12, len(plain)), replace=False)]:
            raw[b, a * nch + 4, j, i] = vals[4 + rng.randint(4)]
        if l == 0:
            b, a, j, i = plain[0]
            raw[b, a * nch + 4, j, i] = np.nan
    return dict(c, name=c["name"] + "_special_logits", raws=raws)


def big_wh_logit(c):
    """One matched cell of each layer with tw = 1e9: its wh gradient, times an upstream gradient of 1e30, overflows fp32."""
    C, mask, lab = c["C"], c["mask"], c["labels"]
    raws = [r.copy() for r in c["raws"]]
    for l, raw in enumerate(raws):
        _, pred = orc.decode_train(raw, l, C, mask=mask)
        _, _, tgt_mask, _ = orc.build_target(pred, lab, l, C, c["thrs"][0], mask=mask)
        m = np.argwhere(tgt_mask[..., 0] == 1)
        if len(m):
            b, a, j, i = m[0]
            raw[b, a * (5 + C) + 2, j, i] = 1e9
    return dict(c, name=c["name"] + "_big_wh", raws=raws)


VALID = {
    "class_ids": class_ids, "collisions": collisions, "full_k256": full_k256, "first_n_rows": first_n_rows,
    "geometry": geometry, "huge_box": huge_box, "degenerate": degenerate, "ignore_thresholds": ignore_thresholds,
    "ignore_boundary_overlap": lambda: ignore_boundary(False), "ignore_boundary_contained": lambda: ignore_boundary(True),
    "mixed_C1": lambda: mixed(1, seed=23), "mixed_C28": lambda: mixed(28, seed=24), "mixed_C29": lambda: mixed(29, seed=25),
    "mixed_C80": lambda: mixed(80, img=160, seed=26),
    "alt_anchor_mask": lambda: mixed(4, seed=27, mask=ALT_MASK, name="alt_anchor_mask"),
    "mixed_608": lambda: mixed(80, img=608, seed=28, n=50, name="mixed_608"),
    "special_logits": lambda: with_special_logits(mixed(6, seed=29, name="logits")),
}
"""The label sets on which the reference runs to the end, by name."""

# The sets whose BCE inputs and targets all lie in [0, 1] and whose loss is finite: the unfused torch path runs on these (ATen's
# BCE asserts on the device outside [0, 1]).
UNFUSED = ("alt_anchor_mask", "class_ids", "collisions", "full_k256", "ignore_boundary_contained", "ignore_boundary_overlap",
           "ignore_thresholds", "mixed_608", "mixed_C1", "mixed_C28", "mixed_C29", "mixed_C80")

ERROR = {"bad_class_%d" % v: functools.partial(bad_class, float(v)) for v in (4, 7, -15, -24)}
ERROR["out_of_grid"] = out_of_grid
"""Label sets with a matched GT that the reference's indexing rejects (C = 4 for the class ids)."""


@functools.lru_cache(maxsize=None)
def get(name):
    return VALID[name]() if name in VALID else ERROR[name]()

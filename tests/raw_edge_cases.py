"""Raw head tensors for the fused front end (yl_filter_raw_typed: a flag kernel, k_flag_tma or k_flag_raw, then k_emit_flagged)
at its edges, and a model of which flag kernel a call dispatches to.

  heads            random heads [B, 3*(5+C), F, F] for an explicit grid list (synth derives only floor(img / stride))
  t_star           the smallest logit of an element type that passes the spec's exact test fl32(obj * sigmoid(t)) >= conf
  threshold_case   heads whose only candidates are planted t* pairs at class, lane, tile and scale edges
  plant_specials   NaN, +-inf, +-0 and +-1e30 in the objectness, class and box planes of live and dead boxes
"""
import math
import os

import numpy as np

from oracle import oracle as orc

F32 = np.float32
SPECIALS = [F32(np.nan), F32(np.inf), F32(-np.inf), F32(0.0), F32(-0.0), F32(1e30), F32(-1e30)]
CLASS_EDGES = (0, 7, 8, 31, 32, 63, 64, 127)              # flag-chunk (8 classes) and flag-word (32 classes) edges
WT_KC, FT_STAGES = 8, 3                                   # k_flag_tma: classes per ring stage, ring stages


def row_offsets(Fs):
    """First row of every scale in the concatenated [M] axis (yolov4.py:324)."""
    out, r = [], 0
    for f in Fs:
        out.append(r)
        r += 3 * f * f
    return out


def heads(B, Fs, C, seed):
    """Random heads: background boxes with objectness logits around -6 and class logits around -8 (at conf 1e-3 under one per
    cent of their pairs pass, so the oracle's NMS stays quick on 75x75 grids), and six per cent foreground boxes with a live
    objectness and two strong classes."""
    rng = np.random.RandomState(seed)
    out = []
    for f in Fs:
        h = np.empty((B, 3, 5 + C, f, f), F32)
        h[:, :, 0:2] = rng.randn(B, 3, 2, f, f)
        h[:, :, 2:4] = 0.5 * rng.randn(B, 3, 2, f, f)
        h[:, :, 4] = 2 * rng.randn(B, 3, f, f) - 6
        h[:, :, 5:] = 2.5 * rng.randn(B, 3, C, f, f) - 8
        fg = np.argwhere(rng.rand(B, 3, f, f) < 0.06)         # foreground: live objectness, two strong classes
        for b, a, y, x in fg:
            h[b, a, 4, y, x] = 1 + rng.randn()
            h[b, a, 5 + rng.randint(C, size=2), y, x] = 2 + rng.randn(2)
        out.append(h.reshape(B, 3 * (5 + C), f, f))
    return out


def plant_specials(raws, C, seed):
    """Every special value as the objectness of a box, as a class logit of a live box (objectness logit 4) and of a dead one
    (objectness logit -inf or -30), and as tx / tw of a live box.  A dead box flags nothing whatever its class logits are; a
    NaN class logit of a live box drops the whole row (utils.py:139-145)."""
    rng = np.random.RandomState(seed)
    for h in raws:
        B, _, f, _ = h.shape
        v = h.reshape(B, 3, 5 + C, f * f)
        for k, s in enumerate(SPECIALS):
            for what in range(5):
                b, a, p = rng.randint(B), rng.randint(3), rng.randint(f * f)
                c = 5 + rng.randint(C)
                if what == 0:
                    v[b, a, 4, p] = s
                    v[b, a, 5:, p] = 2.0                  # classes that would pass: the objectness decides
                elif what == 1:
                    v[b, a, 4, p] = 4.0
                    v[b, a, c, p] = s
                elif what == 2:
                    v[b, a, 4, p] = -np.inf if k % 2 else -30.0
                    v[b, a, c, p] = s
                    v[b, a, 5 + (c - 4) % C, p] = np.inf
                else:
                    v[b, a, 4, p] = 4.0
                    v[b, a, 5:, p] = 3.0
                    v[b, a, 0 if what == 3 else 2, p] = s
    return raws


# ------------------------------------------------------------------------------------------------ element types
DTYPES = ("f32", "f16", "bf16")


def to_elem(x, dt):
    """x rounded to nearest in the element type, returned widened to float32 (exact)."""
    x = np.asarray(x, F32)
    if dt == "f32":
        return x.copy()
    if dt == "f16":
        return x.astype(np.float16).astype(F32)
    b = x.view(np.uint32).astype(np.uint64)
    r = ((b + 0x7FFF + ((b >> 16) & 1)) >> 16).astype(np.uint32)        # round to nearest even (no NaN inputs here)
    return (r << 16).view(F32)


def _bits(dt):
    return {"f32": (32, 0x7F800000), "f16": (16, 0x7C00), "bf16": (16, 0x7F80)}[dt]


def _key_to_value(k, dt):
    n, _ = _bits(dt)
    sign = 1 << (n - 1)
    bits = k if k >= 0 else (-k) | sign
    if dt == "f32":
        return np.array([bits], np.uint32).view(F32)[0]
    if dt == "f16":
        return F32(np.array([bits], np.uint16).view(np.float16)[0])
    return np.array([bits << 16], np.uint32).view(F32)[0]


def sigmoid(t):
    """The fp32 spec sigmoid (DESIGN.md section 4) of one value."""
    return F32(orc.lib().orc_sigmoidf(float(t)))


def passes(obj, t, conf):
    """The spec's exact per-class test fl32(obj * sigmoid(t)) >= conf."""
    return bool(F32(obj) * sigmoid(t) >= F32(conf))


def t_star(obj, conf, dt):
    """(t*, pred(t*)) in the element type dt: t* the smallest value with passes(obj, t*, conf), pred its predecessor, found by
    bisection on the ordered integer encoding (-inf .. +inf; -0 is skipped, it equals +0).  None when even +inf fails."""
    _, inf = _bits(dt)
    lo, hi = -inf, inf
    if not passes(obj, _key_to_value(hi, dt), conf):
        return None
    assert not passes(obj, _key_to_value(lo, dt), conf), "conf <= 0: every logit passes"
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if passes(obj, _key_to_value(mid, dt), conf):
            hi = mid
        else:
            lo = mid
    return _key_to_value(hi, dt), _key_to_value(lo, dt)


def _value_to_key(t, dt):
    n_bits, _ = _bits(dt)
    sign = 1 << (n_bits - 1)
    if dt == "f16":
        b = int(np.array([t], np.float16).view(np.uint16)[0])
    else:
        b = int(np.array([t], F32).view(np.uint32)[0]) >> (0 if dt == "f32" else 16)
    return b if b < sign else -(b & (sign - 1))


def values_below(t, n, dt):
    """The n values of the element type directly below t (ordered encoding)."""
    _, inf = _bits(dt)
    k = _value_to_key(t, dt)
    return [_key_to_value(j, dt) for j in range(max(-inf, k - n), k)]


def next_up(t, dt):
    """The value of the element type directly above t."""
    _, inf = _bits(dt)
    return _key_to_value(min(_value_to_key(t, dt) + 1, inf), dt)


# ------------------------------------------------------------------------------------------------ exact-threshold cases
THRESHOLD_CONFS = (1e-4, 1e-3, 0.005, float(np.nextafter(F32(0.02), F32(0))), 0.02, 0.2, 0.5, 0.9, 0.999, 1e-30,
                   float(np.array([0x00012345], np.uint32).view(F32)[0]))          # the last one subnormal (1.04e-40)
# conf / obj: 1 (obj = conf where reachable), both sides of the 0.9 cap of class_logit_bound, ..., and obj = 1 (None)
RATIOS = (1.0, 0.9 / (1 - 1e-5) * (1 + 1e-6), 0.9 / (1 - 1e-5) * (1 - 1e-6), 0.9001, 0.8999, 0.5, 1e-2, 1e-4, 1e-8, None)


def _objectness_logit(conf, ratio, dt):
    """(to, obj): an objectness logit of the element type and its sigmoid with obj >= conf near conf / ratio, or None."""
    if ratio is None:
        to = to_elem(F32(30.0), dt)
        return float(to), sigmoid(to)
    target = float(F32(conf)) / ratio
    if target > 1.0:
        return None
    to = F32(30.0) if target >= 1.0 else to_elem(F32(math.log(target) - math.log1p(-target)), dt)
    for _ in range(64):                                   # ratio 1: step up until sigmoid(to) reaches conf
        if sigmoid(to) >= F32(conf):
            break
        to = next_up(to, dt)
    if not sigmoid(to) >= F32(conf):
        return None
    return float(to), sigmoid(to)


def threshold_regimes(conf, dt):
    """[(ratio, to, obj, t*, pred)] of every reachable regime of conf."""
    out = []
    for r in RATIOS:
        o = _objectness_logit(conf, r, dt)
        if o is None:
            continue
        ts = t_star(o[1], conf, dt)
        if ts is not None:
            out.append((r, o[0], o[1]) + ts)
    return out


def edge_positions(F2):
    """Box positions at lane (4 boxes), warp tile (32 / 128 boxes), CTA tile and scale edges."""
    return sorted({p for p in (0, 3, 4, 31, 32, 127, 128, 511, 512, F2 - 1) if 0 <= p < F2})


def threshold_case(Fs, C, conf, dt, B=2):
    """Heads (float32 arrays holding values of dt) in which every (image, scale, anchor, edge position) holds a planted box;
    the rest are dead (objectness logit -inf).  Planted boxes alternate between a pair box (t* as class k1, pred(t*) as class
    k2, every other class -inf) and an all-pred box (every class pred(t*)), cycling through the regimes of conf and the class
    edges.  Returns (raws, expected) with expected the sorted (image, row, class) list of the only candidates: the t* pairs."""
    regimes = threshold_regimes(conf, dt)
    assert regimes, "conf %r has no reachable regime" % conf
    edges = [k for k in CLASS_EDGES if k < C] + ([C - 1] if C - 1 not in CLASS_EDGES else [])
    raws = [np.zeros((B, 3, 5 + C, f * f), F32) for f in Fs]
    for v in raws:
        v[:, :, 4] = -np.inf
        v[:, :, 5:] = -np.inf
    offs = row_offsets(Fs)
    expected, i = [], 0
    for b in range(B):
        for l, f in enumerate(Fs):
            for a in range(3):
                for p in edge_positions(f * f):
                    _, to, _, ts, pr = regimes[(i // 2) % len(regimes)]
                    v = raws[l][b, a]
                    v[4, p] = to
                    if (i + b) % 2 == 0:
                        k1 = edges[(i // 2) % len(edges)]
                        k2 = edges[(i // 2 + 1) % len(edges)] if len(edges) > 1 else None
                        v[5 + k1, p] = ts
                        if k2 is not None:
                            v[5 + k2, p] = pr
                        expected.append((b, offs[l] + a * f * f + p, k1))
                    else:
                        v[5:, p] = pr
                    i += 1
    return [v.reshape(B, 3 * (5 + C), f, f) for v, f in zip(raws, Fs)], sorted(expected)


# ------------------------------------------------------------------------------------------------ dispatch model
def flag_kernel(Fs, C, conf, dt, bases=None, flag_env=None):
    """The kernels yl_filter_raw_typed launches for a case, as ('tma', NW) or ('raw', dt, NW) for the flag pass, plus the
    emit kernel's (dt, NW) and the vector width of every scale.  bases: the heads' data_ptr() % 16 (default all 0).  A scale is
    a vector scale when F^2 % 4 == 0, its base is 16-byte (fp32) or 8-byte (16-bit) aligned and its table rows start at a
    multiple of 4; k_flag_tma streams the fp32 vector scales when the threshold is below 0.02 and there are at least three
    8-class chunks, unless YL_FLAG selects the register-staged kernel."""
    bases = bases or [0] * len(Fs)
    flag_env = os.environ.get("YL_FLAG") if flag_env is None else flag_env
    nw = (C + 31) // 32
    align = 16 if dt == "f32" else 8
    vec = [4 if (f * f) % 4 == 0 and base % align == 0 and off % 4 == 0 else 1
           for f, base, off in zip(Fs, bases, row_offsets(Fs))]
    sparse = F32(conf) >= F32(0.02)
    tma = (flag_env is None or flag_env == "tma") and dt == "f32" and not sparse and \
        any(v == 4 for v in vec) and (C + WT_KC - 1) // WT_KC >= FT_STAGES
    flag = ("tma", nw) if tma else ("raw", dt, nw)
    return flag, (dt, nw), vec

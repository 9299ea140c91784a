"""The IoU box term of the fused loss (`fused_yolo_loss(..., iou_loss='giou' | 'diou' | 'ciou', iou_normalizer=n)`), stated three
ways:

  box_loss        the term and d term / d (px, py, pw, ph) in float64 torch with autograd, on the xyxy corners x +- w / 2:
                  torchvision 0.26's generalized_ / distance_ / complete_box_iou_loss (eps 1e-7), alpha of CIoU under no_grad,
                  torch.maximum / torch.minimum (half the gradient to each side of an exact tie).  A NaN term gives NaN in all
                  four derivatives.
  layer_spec      one layer of the fused loss: the four components and d loss / d raw.  Components 2 and 3 and the gradient
                  channels 4.. are orc.yolo_loss_layer's; the box term replaces components 0 and 1 (0 becomes n * sum of the
                  terms, 1 is 0) and box channels 0..3 (n * d term / d raw at the matched cells, 0 elsewhere).  p is
                  orc.decode_train's train-mode box, g the cell's LAST matched GT (label / stride), the assignment
                  tests/target_spec.py's.
  box_loss_fp32   a NumPy model of the kernel (yl_loss.cu, iou_box_loss) in its operation order: the linear geometry in
                  float64, everything else one fp32 rounding per operation.  It establishes the gradient bound
                  (GRAD_REL, GRAD_ABS) on the CPU.
"""
import numpy as np
import torch

from oracle import oracle as orc

KINDS = ("giou", "diou", "ciou")
EPS = 1e-7
# |g - g64| <= GRAD_REL |g64| + GRAD_ABS * n per entry of d loss / d raw (n = iou_normalizer); DESIGN.md section 1
GRAD_REL, GRAD_ABS = 1e-4, 1e-6
# Predicted extents outside [EXTENT_MIN, EXTENT_MAX] grid units (|tw| or |th| of ~70 and more): there the literal expression's
# aspect derivative is 0 * inf (a zero height) or needs more range than fp32 has, so the gradient bound does not apply; those
# cells are checked for their term and for NaN in all four entries where the term is NaN (extreme_extent)
EXTENT_MIN, EXTENT_MAX = 1e-30, 1e30


def extreme_extent(p):
    """Rows of p [N, 4] whose predicted width or height lies outside [EXTENT_MIN, EXTENT_MAX] (NaN included)."""
    wh = np.abs(np.asarray(p, np.float64)[:, 2:4])
    return ~((wh >= EXTENT_MIN) & (wh <= EXTENT_MAX)).all(1)


# ------------------------------------------------------------------------------------------------ float64 torch spec
def _terms(kind, p, g):
    """torchvision's expressions on [N, 4] (cx, cy, w, h) float64 tensors.  Both boxes are first moved by the prediction's centre
    (a constant for autograd): every term is translation-invariant, and the prediction's corners +- w / 2 stay exact in float64,
    so a tiny predicted extent is not rounded away against a large grid coordinate."""
    o = p[:, :2].detach()
    pc, gc = p[:, :2] - o, g[:, :2] - o
    x1, x2 = pc[:, 0] - p[:, 2] / 2, pc[:, 0] + p[:, 2] / 2
    y1, y2 = pc[:, 1] - p[:, 3] / 2, pc[:, 1] + p[:, 3] / 2
    x1g, x2g = gc[:, 0] - g[:, 2] / 2, gc[:, 0] + g[:, 2] / 2
    y1g, y2g = gc[:, 1] - g[:, 3] / 2, gc[:, 1] + g[:, 3] / 2
    xk1, yk1, xk2, yk2 = torch.maximum(x1, x1g), torch.maximum(y1, y1g), torch.minimum(x2, x2g), torch.minimum(y2, y2g)
    mask = (yk2 > yk1) & (xk2 > xk1)
    inter = torch.where(mask, (xk2 - xk1) * (yk2 - yk1), torch.zeros_like(x1))
    union = (x2 - x1) * (y2 - y1) + (x2g - x1g) * (y2g - y1g) - inter
    iou = inter / (union + EPS)
    xc1, yc1, xc2, yc2 = torch.minimum(x1, x1g), torch.minimum(y1, y1g), torch.maximum(x2, x2g), torch.maximum(y2, y2g)
    if kind == "giou":
        area_c = (xc2 - xc1) * (yc2 - yc1)
        return 1 - (iou - (area_c - union) / (area_c + EPS))
    diag = (xc2 - xc1) ** 2 + (yc2 - yc1) ** 2 + EPS
    cen = ((x2 + x1) / 2 - (x1g + x2g) / 2) ** 2 + ((y2 + y1) / 2 - (y1g + y2g) / 2) ** 2
    loss = 1 - iou + cen / diag
    if kind == "diou":
        return loss
    v = (4 / torch.pi ** 2) * torch.pow(torch.atan((x2g - x1g) / (y2g - y1g)) - torch.atan((x2 - x1) / (y2 - y1)), 2)
    with torch.no_grad():
        alpha = v / (1 - iou + v + EPS)
    return loss + alpha * v


def box_loss(kind, p, g):
    """kind in KINDS; p, g [N, 4] (cx, cy, w, h) -> (term float64 [N], d term / d p float64 [N, 4])."""
    p = torch.as_tensor(np.asarray(p, np.float64)).reshape(-1, 4).clone().requires_grad_(True)
    g = torch.as_tensor(np.asarray(g, np.float64)).reshape(-1, 4)
    with np.errstate(all="ignore"):
        loss = _terms(kind, p, g)
        (grad,) = torch.autograd.grad(loss.sum(), p)
    loss, grad = loss.detach().numpy(), grad.numpy().copy()
    grad[np.isnan(loss)] = np.nan
    return loss, grad


# ------------------------------------------------------------------------------------------------ assignment
def last_gt_per_cell(labels, layer_no, F, anchors=orc.ANCHORS_PX, mask=orc.ANCHOR_MASK):
    """{(b, a, j, i): t} -- the last GT t that tests/target_spec.py's scatter writes into each matched cell of the layer."""
    labels = np.asarray(labels, np.float32)
    stride = np.float32(orc.STRIDES[layer_no])
    ref = np.zeros((9, 4), np.float32)
    ref[:, 2:] = np.array([[w / float(stride), h / float(stride)] for w, h in anchors], np.float64).astype(np.float32)
    s = labels[:, :, 0]
    for c in range(1, 5):
        s = s + labels[:, :, c]
    nlabel = (s > 0).sum(1)
    tb = labels[:, :, :4] / stride
    with np.errstate(invalid="ignore"):
        ti, tj = tb[..., 0].astype(np.int16), tb[..., 1].astype(np.int16)
    owner = {}
    for b in range(labels.shape[0]):
        n = int(nlabel[b])
        if n == 0:
            continue
        box = np.zeros((n, 4), np.float32)
        box[:, 2], box[:, 3] = tb[b, :n, 2], tb[b, :n, 3]
        best = np.argmax(orc.bboxes_iou(box, ref, xyxy=True), axis=1)
        for t in range(n):
            if best[t] not in mask[layer_no]:
                continue
            i, j = int(ti[b, t]), int(tj[b, t])
            if not (-F <= i < F and -F <= j < F):
                raise IndexError("a matched GT indexes outside the grid")
            owner[(b, int(best[t] % 3), j % F, i % F)] = t
    return owner


def matched_pairs(raw, labels, layer_no, C, anchors=orc.ANCHORS_PX, mask=orc.ANCHOR_MASK):
    """(cells [M, 4] (b, a, j, i), p [M, 4] fp32, g [M, 4] fp32, s [M, 2] fp32 sigmoids of tx, ty) of the layer's matched cells."""
    output, pred = orc.decode_train(raw, layer_no, C, anchors, mask)
    F = pred.shape[2]
    owner = last_gt_per_cell(labels, layer_no, F, anchors, mask)
    cells = np.array(sorted(owner), np.int64).reshape(-1, 4)
    tb = (np.asarray(labels, np.float32)[..., :4] / np.float32(orc.STRIDES[layer_no])).astype(np.float32)
    p = np.array([pred[b, a, j, i] for b, a, j, i in cells], np.float32).reshape(-1, 4)
    g = np.array([tb[b, owner[(b, a, j, i)]] for b, a, j, i in cells], np.float32).reshape(-1, 4)
    s = np.array([output[b, a, j, i, :2] for b, a, j, i in cells], np.float32).reshape(-1, 2)
    return cells, p, g, s


def raw_chain(dp, p, s):
    """d / d p -> d / d raw: s (1 - s) for x, y (s the fp32 sigmoid), pw, ph for w, h (float64)."""
    s64, p64 = s.astype(np.float64), p.astype(np.float64)
    return dp * np.concatenate([s64 * (1.0 - s64), p64[:, 2:4]], 1)


def layer_spec(raw, labels, layer_no, C, thr, kind, norm=1.0, anchors=orc.ANCHORS_PX, mask=orc.ANCHOR_MASK):
    """One layer: (components float64 [4], d loss / d raw float64 [B, 3(5+C), F, F], per-cell (cells, term, d term / d raw, p))."""
    comps, grad = orc.yolo_loss_layer(raw, labels, layer_no, C, thr, anchors, mask)
    cells, p, g, s = matched_pairs(raw, labels, layer_no, C, anchors, mask)
    term, dp = box_loss(kind, p, g)
    with np.errstate(invalid="ignore", over="ignore"):
        graw = norm * raw_chain(dp, p, s)
        comps = np.array([norm * term.sum(), 0.0, comps[2], comps[3]])
    grad = np.array(grad)
    nch = 5 + C
    for a in range(3):
        grad[:, a * nch:a * nch + 4] = 0.0
    for (b, a, j, i), gr in zip(cells, graw):
        grad[b, a * nch:a * nch + 4, j, i] = gr
    return comps, grad, (cells, norm * term, graw, p)


# ------------------------------------------------------------------------------------------------ fp32 model of the kernel
def _axis(pc, pw, gc, gw):
    d = pc.astype(np.float64) - gc.astype(np.float64)
    hp, hg = 0.5 * pw.astype(np.float64), 0.5 * gw.astype(np.float64)
    lo, hi = d - hp, d + hp
    iw = np.minimum(hi, hg) - np.maximum(lo, -hg)
    cw = np.maximum(hi, hg) - np.minimum(lo, -hg)

    def share(a, b):
        return np.where(a > b, 1.0, np.where(a == b, 0.5, 0.0)).astype(np.float32)

    aR, aL, bR, bL = share(hg, hi), share(lo, -hg), share(hi, hg), share(-hg, lo)
    h = np.float32(0.5)
    return ((d + (hp - hp) + (hg - hg)).astype(np.float32), iw > 0, iw.astype(np.float32), cw.astype(np.float32), aR - aL, (aR + aL) * h,
            bR - bL, (bR + bL) * h)


def box_loss_fp32(kind, p, g):
    """The kernel's term and d term / d p on fp32 [N, 4] inputs (reciprocals as correctly rounded fp32 divisions; the kernel's
    MUFU.RCP is within 1 ulp of them)."""
    f = np.float32
    p, g = np.asarray(p, f).reshape(-1, 4), np.asarray(g, f).reshape(-1, 4)
    px, py, pw, ph = p.T
    gx, gy, gw, gh = g.T
    one, eps = f(1), f(EPS)
    with np.errstate(all="ignore"):
        xd, xov, xiw, xcw, xdi, xdip, xdc, xdcp = _axis(px, pw, gx, gw)
        yd, yov, yiw, ycw, ydi, ydip, ydc, ydcp = _axis(py, ph, gy, gh)
        ov = xov & yov
        I = np.where(ov, xiw * yiw, f(0))
        ap, ag = pw * ph, gw * gh
        U = (ap + ag) - I
        Ue = U + eps
        rUe = one / Ue
        iou = I * rUe
        omi = np.where(np.isinf(Ue), one - iou, (((ap - I) + (ag - I)) + eps) * rUe)
        kx, ky = np.where(ov, yiw, f(0)), np.where(ov, xiw, f(0))
        dI = [kx * xdi, ky * ydi, kx * xdip, ky * ydip]
        dU = [f(0) - dI[0], f(0) - dI[1], ph - dI[2], pw - dI[3]]
        d = [(iou * dU[k] - dI[k]) * rUe for k in range(4)]
        L = omi
        if kind == "giou":
            Cc = xcw * ycw
            Ce = Cc + eps
            rCe = one / Ce
            L = L + (Cc - U) * rCe
            dC = [ycw * xdc, xcw * ydc, ycw * xdcp, xcw * ydcp]
            q = Ue * rCe
            d = [d[k] + (dC[k] * q - dU[k]) * rCe for k in range(4)]
        else:
            rho2 = xd * xd + yd * yd
            D = (xcw * xcw + ycw * ycw) + eps
            rD = one / D
            P = rho2 * rD
            L = L + P
            tcx, tcy = f(2) * xcw, f(2) * ycw
            dD = [tcx * xdc, tcy * ydc, tcx * xdcp, tcy * ydcp]
            dr = [f(2) * xd, f(2) * yd, f(0) * xd, f(0) * yd]
            d = [d[k] + (dr[k] - P * dD[k]) * rD for k in range(4)]
            if kind == "ciou":
                r = pw * (one / ph)
                da = np.arctan(gw * (one / gh)) - np.arctan(r)
                v = f(0.405284735) * (da * da)
                alpha = v * (one / ((omi + v) + eps))
                L = L + alpha * v
                wide = np.abs(pw) > np.abs(ph)
                inv = one / np.where(wide, pw, ph)
                t = np.where(wide, ph, pw) * inv
                ik = inv * (one / (one + t * t))
                dik = ik * t
                c = alpha * (f(-0.810569469) * da)
                d[2] = d[2] + c * np.where(wide, dik, ik)
                d[3] = d[3] - c * np.where(wide, ik, dik)
        d = np.stack(d, 1).astype(f)
        d[np.isnan(L)] = np.nan
    return L.astype(f), d


def raw_grad_fp32(kind, p, g, s, norm=1.0):
    """The kernel's mgrad[..., 0:4] entries: fp32 (n * d) * s * (1 - s) for x, y and (n * d) * pw, ph for w, h."""
    f = np.float32
    _, d = box_loss_fp32(kind, p, g)
    n = f(norm)
    with np.errstate(all="ignore"):
        dn = d * n
        s = np.asarray(s, f)
        out = np.empty_like(dn)
        out[:, :2] = (dn[:, :2] * s) * (f(1) - s)
        out[:, 2:] = dn[:, 2:] * np.asarray(p, f)[:, 2:]
    return out


def within_bound(got, want, norm=1.0, rel=GRAD_REL, abs_=GRAD_ABS):
    """Boolean mask: NaN where want is NaN, the same infinities, finite entries within rel |want| + abs_ * norm."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    with np.errstate(invalid="ignore"):
        ok = np.abs(got - want) <= rel * np.abs(want) + abs_ * norm
    ok |= np.isnan(got) & np.isnan(want)
    ok |= np.isinf(want) & (got == want)
    return ok & (np.isnan(got) == np.isnan(want))

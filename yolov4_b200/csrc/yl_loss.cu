// yl_loss.cu -- N2 (SURVEY.md 8f): YOLOLoss.forward (yolo/model/yololoss.py:373-443) for one layer, fused with the
// train-mode YOLOLayer (yololayer.py:122-145) and build_target (:118-371), straight from the raw head tensor.
//
// The reference materialises, per layer and step, the dense `output`, `pred`, `target`, `tgt_mask`, `tgt_scale` and `obj_mask`
// tensors and runs ~15 elementwise passes plus four reductions over them.  But outside the <= K matched cells of an
// image every masked term is exactly 0 (tgt_mask = 0 => BCE(0, 0) = 0, MSE(0, 0) = 0), and the objectness term of a cell
// needs only its five box / objectness logits.  So:
//
//   k_loss_match   per image: GT -> cell assignment (:249-265), then for every matched cell (last writer per cell, class
//                  one-hots accumulated over colliding GTs, SURVEY.md 7-9) the xy / wh / cls terms of :417-427 and their
//                  derivatives with respect to the raw logits, kept in a compact per-GT table.  A class id sets channel
//                  5 + cls with Python's negative-index wrap, as build_target does (class_channel): a negative id marks
//                  another class, or overwrites the last GT's x / y / w / h target with 1 (channel 4 stays 1).
//   k_loss_obj     per cell: decode the box from tx,ty,tw,th (5 of the 85 planes are read), ignore mask (:276-294),
//                  objectness BCE (:425) and d/d(raw objectness).
//   k_loss_bwd_*   grad_raw = upstream * (objectness plane from k_loss_obj, matched cells from the table); the rest of
//                  grad_raw is the zero background (cudaMemsetAsync).
//
// 16-bit heads (fp16 / bf16): the forward kernels widen every element on load (yl_common.cuh: every 16-bit value has an exact
// fp32 image) and the fp32 arithmetic below applies unchanged; the backward kernels form the same fp32 product and round it once
// into the head's element type, so a 16-bit gradient is the fp32 path's gradient on the widened head, rounded to nearest-even.
//
// IoU box regression (iou_loss = GIoU / DIoU / CIoU, k_loss_match<T, IOU>, yl_loss_forward_ex): the xy BCE and wh MSE of every
// matched cell are replaced by iou_normalizer * torchvision's box-IoU loss of the decoded prediction and the cell's last GT, in
// grid units (DESIGN.md sections 1 and 5.9).  Lanes 0..3 evaluate the term redundantly and keep their own channel's derivative;
// k_loss_obj, the class terms and the backward kernels do not change.  The IOU = 0 instantiations are the plain loss, unchanged.
//
// Per-term arithmetic is fp32 like the reference's (ATen binary_cross_entropy: (t-1) max(log(1-x), -100) - t max(log x, -100),
// backward (x-t)/max((1-x) x, 1e-12); mse_loss); sums are accumulated in fp64.  Parity: loss and gradient within 1e-5 /
// 2e-5 relative of the reference (tests/golden/loss.npz), not bit-exact (the reference's reduction order is unspecified).
#include "yl_target.cuh"
#include "../../include/yolo_head.h"

namespace yl {

constexpr int LS_THREADS = 256;

// The clamps propagate NaN (nanmaxf, not fmaxf): a NaN probability gives a NaN term, as the max of ATen's CPU kernel does,
// and as the NaN gradient of the same cell already says.
__device__ __forceinline__ float bce_term(float x, float t)
{
    const float lx = nanmaxf(spec_logf(x), -100.0f), l1x = nanmaxf(spec_logf(__fsub_rn(1.0f, x)), -100.0f);
    return __fsub_rn(__fmul_rn(__fsub_rn(t, 1.0f), l1x), __fmul_rn(t, lx));
}
// bce_term for t = 1 (one) or t = 0: the other logarithm is clamped to [-100, 0] and multiplied by zero, so the term is
// -max(log x, -100) resp. -max(log(1 - x), -100) -- the same value (NaN included) for one spec_logf instead of two.
__device__ __forceinline__ float bce_term01(float x, bool one)
{
    const float l = nanmaxf(spec_logf(one ? x : __fsub_rn(1.0f, x)), -100.0f);
    return __fsub_rn(0.0f, l);
}
__device__ __forceinline__ float bce_grad(float x, float t)
{
    return __fdiv_rn(__fsub_rn(x, t), fmaxf(__fmul_rn(__fsub_rn(1.0f, x), x), 1e-12f));
}

// ---- IoU box losses (iou_loss = giou / diou / ciou): torchvision's generalized_ / distance_ / complete_box_iou_loss with
// eps = 1e-7 on the xyxy corners x +- w / 2 of the predicted box p and the GT g (grid units), and d loss / d (px, py, pw, ph) of
// that float64 expression: alpha of CIoU is a constant (torchvision computes it under no_grad) and an exact tie of
// torch.maximum / torch.minimum gives half the gradient to each side.
constexpr float IOU_EPS = 1e-7f;

// NaN-propagating min / max of fp64 edges (torch.minimum / maximum propagate NaN)
__device__ __forceinline__ double edge_min(double a, double b) { return (a != a) ? a : ((b != b) ? b : (a < b ? a : b)); }
__device__ __forceinline__ double edge_max(double a, double b) { return (a != a) ? a : ((b != b) ? b : (a > b ? a : b)); }
// 1 / x within 1 ulp (MUFU.RCP; a subnormal x counts as 0 and gives inf, +inf gives 0, NaN stays NaN).  The IoU term is a
// tolerance contract, and unlike __fdiv_rn this has no slow-path call, whose register save would spill.
__device__ __forceinline__ float rcp_approx(float x)
{
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// the first operand's share of the gradient of max(a, b) (or of min(b, a)): 1, 1/2 at a tie, 0
__device__ __forceinline__ float share_gt(double a, double b) { return a > b ? 1.0f : (a == b ? 0.5f : 0.0f); }

// One axis of the box pair: the prediction's edges relative to the GT's centre.  The fp64 difference of two fp32 values is
// exact and every edge is within 2^-53 of its real value, so the min / max decisions (ties included) are the float64 spec's,
// and the widths and the centre distance below are each ONE fp32 rounding away from the exact value, whether the boxes sit
// in cell 0 or cell 75 and however small they are.
struct IouAxis { float d, iw, cw, di, dip, dc, dcp; bool ov; };
__device__ __forceinline__ IouAxis iou_axis(float pc, float pw, float gc, float gw)
{
    const double d = (double)pc - (double)gc, hp = 0.5 * (double)pw, hg = 0.5 * (double)gw;
    const double l = d - hp, r = d + hp;
    const double iw = edge_min(r, hg) - edge_max(l, -hg), cw = edge_max(r, hg) - edge_min(l, -hg);
    IouAxis x;
    x.d = (float)(d + (hp - hp) + (hg - hg));                              // the spec's (x1 + x2) / 2 is NaN for an infinite width
    x.ov = iw > 0.0;                                                       // torchvision: overlap strictly positive
    x.iw = (float)iw;
    x.cw = (float)cw;
    const float aR = share_gt(hg, r), aL = share_gt(l, -hg);               // p's share in min(right edges), max(left edges)
    const float bR = share_gt(r, hg), bL = share_gt(-hg, l);               // p's share in max(right edges), min(left edges)
    x.di = __fsub_rn(aR, aL);                                              // d iw / d pc, d iw / d pw
    x.dip = __fmul_rn(__fadd_rn(aR, aL), 0.5f);
    x.dc = __fsub_rn(bR, bL);                                              // d cw / d pc, d cw / d pw
    x.dcp = __fmul_rn(__fadd_rn(bR, bL), 0.5f);
    return x;
}

// L(p, g) and d L / d (px, py, pw, ph) in d.  IOU: 1 GIoU, 2 DIoU, 3 CIoU.  A NaN term gives NaN in all four derivatives.
template <int IOU>
__device__ __forceinline__ float iou_box_loss(float px, float py, float pw, float ph, float gx, float gy, float gw, float gh,
                                              float (&d)[4])
{
    const IouAxis X = iou_axis(px, pw, gx, gw), Y = iou_axis(py, ph, gy, gh);
    const bool ov = X.ov && Y.ov;
    const float I = ov ? __fmul_rn(X.iw, Y.iw) : 0.0f;
    const float ap = __fmul_rn(pw, ph), ag = __fmul_rn(gw, gh);
    const float U = __fsub_rn(__fadd_rn(ap, ag), I), Ue = __fadd_rn(U, IOU_EPS);
    const float rUe = rcp_approx(Ue), iou = __fmul_rn(I, rUe);
    // 1 - iou as ((ap - I) + (ag - I) + eps) / Ue: no cancellation near iou = 1 (exactly eps / Ue for p == g); an infinite
    // area makes that inf / inf, where 1 - iou is exact instead
    const float omi = isinf(Ue) ? __fsub_rn(1.0f, iou)
                                : __fmul_rn(__fadd_rn(__fadd_rn(__fsub_rn(ap, I), __fsub_rn(ag, I)), IOU_EPS), rUe);
    // d I / d p (zero without overlap); d U = (0, 0, ph, pw) - d I; d (1 - iou) = (iou d U - d I) / Ue
    const float kx = ov ? Y.iw : 0.0f, ky = ov ? X.iw : 0.0f;
    const float dI[4] = {__fmul_rn(kx, X.di), __fmul_rn(ky, Y.di), __fmul_rn(kx, X.dip), __fmul_rn(ky, Y.dip)};
    const float dU[4] = {__fsub_rn(0.0f, dI[0]), __fsub_rn(0.0f, dI[1]), __fsub_rn(ph, dI[2]), __fsub_rn(pw, dI[3])};
#pragma unroll
    for (int k = 0; k < 4; ++k) d[k] = __fmul_rn(__fsub_rn(__fmul_rn(iou, dU[k]), dI[k]), rUe);
    float L = omi;
    if (IOU == 1) {                                                        // GIoU: + (C - U) / (C + eps)
        const float C = __fmul_rn(X.cw, Y.cw), Ce = __fadd_rn(C, IOU_EPS);
        L = __fadd_rn(L, __fmul_rn(__fsub_rn(C, U), rcp_approx(Ce)));
        const float dC[4] = {__fmul_rn(Y.cw, X.dc), __fmul_rn(X.cw, Y.dc), __fmul_rn(Y.cw, X.dcp), __fmul_rn(X.cw, Y.dcp)};
        const float rCe = rcp_approx(Ce), q = __fmul_rn(Ue, rCe);     // d = (dC (U + eps) / Ce - dU) / Ce
#pragma unroll
        for (int k = 0; k < 4; ++k) d[k] = __fadd_rn(d[k], __fmul_rn(__fsub_rn(__fmul_rn(dC[k], q), dU[k]), rCe));
    } else {                                                               // DIoU / CIoU: + rho^2 / (cw^2 + ch^2 + eps)
        const float rho2 = __fadd_rn(__fmul_rn(X.d, X.d), __fmul_rn(Y.d, Y.d));
        const float D = __fadd_rn(__fadd_rn(__fmul_rn(X.cw, X.cw), __fmul_rn(Y.cw, Y.cw)), IOU_EPS);
        const float rD = rcp_approx(D), P = __fmul_rn(rho2, rD);
        L = __fadd_rn(L, P);
        const float tcx = __fmul_rn(2.0f, X.cw), tcy = __fmul_rn(2.0f, Y.cw);
        const float dD[4] = {__fmul_rn(tcx, X.dc), __fmul_rn(tcy, Y.dc), __fmul_rn(tcx, X.dcp), __fmul_rn(tcy, Y.dcp)};
        const float dr[4] = {__fmul_rn(2.0f, X.d), __fmul_rn(2.0f, Y.d), 0.0f, 0.0f};
#pragma unroll
        for (int k = 0; k < 4; ++k) d[k] = __fadd_rn(d[k], __fmul_rn(__fsub_rn(dr[k], __fmul_rn(P, dD[k])), rD));
        if (IOU == 3) {                                                    // CIoU: + alpha v, alpha constant
            const float r = __fmul_rn(pw, rcp_approx(ph));
            const float da = __fsub_rn(atanf(__fmul_rn(gw, rcp_approx(gh))), atanf(r));
            const float v = __fmul_rn(0.405284735f, __fmul_rn(da, da));     // 4 / pi^2
            const float alpha = __fmul_rn(v, rcp_approx(__fadd_rn(__fadd_rn(omi, v), IOU_EPS)));
            L = __fadd_rn(L, __fmul_rn(alpha, v));
            // d atan(pw / ph) = (ph d pw - pw d ph) / (pw^2 + ph^2), through the ratio t = min / max of the two extents (|t| <= 1),
            // so that nothing overflows or underflows for extents in [1e-30, 1e30];  d v = -(8 / pi^2) da d atan(pw / ph)
            const bool wide = fabsf(pw) > fabsf(ph);
            const float inv = rcp_approx(wide ? pw : ph), t = __fmul_rn(wide ? ph : pw, inv);
            const float ik = __fmul_rn(inv, rcp_approx(__fadd_rn(1.0f, __fmul_rn(t, t))));
            const float dik = __fmul_rn(ik, t);
            const float c = __fmul_rn(alpha, __fmul_rn(-0.810569469f, da));  // 8 / pi^2
            d[2] = __fadd_rn(d[2], __fmul_rn(c, wide ? dik : ik));
            d[3] = __fsub_rn(d[3], __fmul_rn(c, wide ? ik : dik));
        }
    }
    if (L != L) {
#pragma unroll
        for (int k = 0; k < 4; ++k) d[k] = L;
    }
    return L;
}

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

struct LossAnchors { AnchorSet an; float maw[3], mah[3]; };          // all nine / the layer's three anchors, grid units

// fp32 -> element type of the gradient, round to nearest-even (overflow to +-inf)
__device__ __forceinline__ float narrow(float x, float *) { return x; }
__device__ __forceinline__ __half narrow(float x, __half *) { return __float2half_rn(x); }
__device__ __forceinline__ __nv_bfloat16 narrow(float x, __nv_bfloat16 *) { return __float2bfloat16_rn(x); }

// IOU (YL_IOU_LOSS_*): 0 is the reference's xy BCE / wh MSE box term; 1..3 replace it by iou_norm * L(p, g) of the matched
// cell (iou_box_loss), with p decoded from the cell's four box logits exactly as k_loss_obj decodes it and g its last GT.
// iou_norm is the last parameter so that the IOU = 0 instantiations keep the parameter layout (and code) they always had.  The
// IoU instantiations ask for one resident CTA per SM at least (in place of ptxas's occupancy target), which lets them hold the
// box term's ~80 live values without spilling; the grid has 8 B CTAs of which a few hundred fit on 148 SMs at any count.
template <typename T, int IOU>
__global__ void __launch_bounds__(LS_THREADS, IOU == 0 ? 0 : 1)
k_loss_match(const T *__restrict__ raw, const float *__restrict__ labels, int F, int K, int C, float stride, LossAnchors A,
             double *__restrict__ loss4, int *__restrict__ tcell_all, int *__restrict__ mcell, float *__restrict__ mgrad,
             int *__restrict__ status, float iou_norm, float sxy, float beta)
{
    __shared__ float tb[TG_MAXK][4];
    __shared__ float tcls[TG_MAXK];
    __shared__ int tcell[TG_MAXK];
    __shared__ int tanc[TG_MAXK];
    __shared__ int sh_n;
    pdl_trigger();
    // grid (image, slice): every CTA of an image repeats the cheap assignment, then its warps take the GTs of its slice
    const int b = blockIdx.x;
    const int n = load_truth(labels, b, K, stride, tb, tcls, &sh_n);
    for (int t = threadIdx.x; t < K; t += LS_THREADS) {
        int cell = -1, anc = 0;
        if (t < n) cell = match_truth(tb[t], F, A.an, &anc, status);
        tcell[t] = cell;
        tanc[t] = anc;
        if (blockIdx.y == 0) tcell_all[(size_t)b * K + t] = cell;
        // the slice that owns GT slot t (see the loop below) initialises its entry of the table, before its own barrier
        if ((t % ((int)gridDim.y * (LS_THREADS / 32))) / (LS_THREADS / 32) == (int)blockIdx.y) mcell[(size_t)b * K + t] = -1;
    }
    __syncthreads();
    const int nch = 5 + C, F2 = F * F, nk = 4 + C;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double acc_xy = 0.0, acc_wh = 0.0, acc_cls = 0.0;
    for (int t = blockIdx.y * (LS_THREADS / 32) + warp; t < n; t += gridDim.y * (LS_THREADS / 32)) {
        const int cell = tcell[t];
        if (cell < 0) continue;
        bool overridden = false;                                       // a later matched GT lands on the same cell: it owns the cell
        for (int u = t + 1 + lane; u < n; u += 32) overridden |= (tcell[u] == cell);
        if (__any_sync(0xFFFFFFFFu, overridden)) continue;
        const int a = cell / F2, r = cell - a * F2;
        const T *cp = raw + ((size_t)(b * 3 + a) * nch) * F2 + r;       // channel k of this cell at cp[k * F2]
        const float tw = tb[t][2], th = tb[t][3];
        const float sc = __fsqrt_rn(__fsub_rn(2.0f, __fdiv_rn(__fdiv_rn(__fmul_rn(tw, th), (float)F), (float)F)));   // :337
        const float w2 = __fmul_rn(sc, sc);                                                                          // :417
        float *gout = mgrad + ((size_t)b * K + t) * nk;
        if (lane == 0) mcell[(size_t)b * K + t] = cell;
        // GTs that share the cell (usually just this one): bit u of same[u >> 5]
        unsigned same[TG_MAXK / 32];
        bool bad_class = false;
#pragma unroll
        for (int w = 0; w < TG_MAXK / 32; ++w) {
            const int u = 32 * w + lane;
            const bool s = u < n && tcell[u] == cell;
            same[w] = (32 * w < n) ? __ballot_sync(0xFFFFFFFFu, s) : 0u;
            if (s) {
                const int ku = class_channel(tcls[u], nch);
                bad_class |= (ku < 0 || ku >= nch);
            }
        }
        if (bad_class && status) atomicExch(status, 1);                // the reference raises IndexError at :369
        // The cell's last GT (this one) writes the xy / wh targets; its class channel overwrites one of them when its id
        // wraps onto 0..3, and wrapping onto 4 (objectness, already 1) changes nothing.
        const int kt = class_channel(tcls[t], nch);
        for (int kk = lane; kk < nk; kk += 32) {
            if constexpr (IOU != 0) {
                if (kk < 4) {                                          // IoU term: lanes 0..3 each evaluate it, keep their channel
                    const float t0 = widen(cp[0]), t1 = widen(cp[(size_t)F2]), t2 = widen(cp[2 * (size_t)F2]), t3 = widen(cp[3 * (size_t)F2]);
                    const int j = r / F, i = r - j * F;
                    const float sx = spec_sigmoidf(t0), sy = spec_sigmoidf(t1);
                    const float pw = __fmul_rn(spec_expf(t2), A.maw[a]), ph = __fmul_rn(spec_expf(t3), A.mah[a]);
                    float dl[4];
                    // scale_x_y: centre fl(fl(fl(s * sxy) + beta) + cell); sxy = 1, beta = -0 is fl(s + cell), bit for bit
                    const float term = iou_box_loss<IOU>(__fadd_rn(__fadd_rn(__fmul_rn(sx, sxy), beta), (float)i),
                                                         __fadd_rn(__fadd_rn(__fmul_rn(sy, sxy), beta), (float)j), pw, ph,
                                                         tb[t][0], tb[t][1], tb[t][2], tb[t][3], dl);
                    if (kk == 0) acc_xy += (double)__fmul_rn(iou_norm, term);
                    const float dn = __fmul_rn(iou_norm, kk == 0 ? dl[0] : kk == 1 ? dl[1] : kk == 2 ? dl[2] : dl[3]);
                    const float s = kk == 0 ? sx : sy;                 // x, y: through sxy s (1 - s); w, h: through pw, ph
                    gout[kk] = kk < 2 ? __fmul_rn(__fmul_rn(__fmul_rn(dn, sxy), s), __fsub_rn(1.0f, s)) : __fmul_rn(dn, kk == 2 ? pw : ph);
                    continue;
                }
            }
            const int k = kk < 4 ? kk : kk + 1;
            const float v = widen(cp[(size_t)k * F2]);
            float g;
            if (kk < 2) {                                              // xy: weighted BCE (:421)
                const float x = spec_sigmoidf(v);
                const float tg = (kt == kk) ? 1.0f : __fsub_rn(tb[t][kk], (float)(short)(int)tb[t][kk]);              // :346,349
                acc_xy += (double)__fmul_rn(bce_term(x, tg), w2);
                g = __fmul_rn(__fmul_rn(__fmul_rn(bce_grad(x, tg), w2), x), __fsub_rn(1.0f, x));
            } else if (kk < 4) {                                       // wh: MSE / 2 on the scaled raw logits (:423)
                const float anc = (kk == 2) ? A.maw[tanc[t]] : A.mah[tanc[t]];
                const float tg = (kt == kk) ? 1.0f : spec_logf(__fadd_rn(__fdiv_rn(kk == 2 ? tw : th, anc), 1e-16f)); // :362,365
                const float d = __fsub_rn(__fmul_rn(v, sc), __fmul_rn(tg, sc));
                acc_wh += 0.5 * (double)d * (double)d;
                g = __fmul_rn(d, sc);
            } else {                                                   // classes: BCE against the union of the cell's one-hots (:427)
                const int kc = kk + 1;                                 // channel 5 + class
                float tg = 0.0f;
#pragma unroll
                for (int w = 0; w < TG_MAXK / 32; ++w) {
                    unsigned m = same[w];
                    while (m) {
                        const int u = 32 * w + __ffs(m) - 1;
                        m &= m - 1u;
                        if (class_channel(tcls[u], nch) == kc) tg = 1.0f;                                             // :369
                    }
                }
                const float x = spec_sigmoidf(v);
                acc_cls += (double)bce_term(x, tg);
                g = __fmul_rn(__fmul_rn(bce_grad(x, tg), x), __fsub_rn(1.0f, x));
            }
            gout[kk] = g;
        }
    }
    acc_xy = warp_sum(acc_xy); acc_wh = warp_sum(acc_wh); acc_cls = warp_sum(acc_cls);
    if (lane == 0) {
        if (acc_xy != 0.0) atomicAdd(&loss4[0], acc_xy);
        if (acc_wh != 0.0) atomicAdd(&loss4[1], acc_wh);
        if (acc_cls != 0.0) atomicAdd(&loss4[3], acc_cls);
    }
    // Nothing here reads the output of the kernel before it on the stream (the previous scale's k_loss_obj), so the
    // two overlap; waiting at the end keeps completion ordered along the chain for whatever follows the last kernel.
    pdl_wait();
}

// SXY: the ignore test's predicted centre takes the grid-sensitivity decode (scale_x_y); otherwise sxy / beta are not read.
template <typename T, bool SXY>
__global__ void __launch_bounds__(LS_THREADS)
k_loss_obj(const T *__restrict__ raw, const float *__restrict__ labels, int F, int K, int C, float stride, LossAnchors A,
           float ignore_thre, const int *__restrict__ tcell_all, double *__restrict__ loss4, float *__restrict__ gobj, float sxy,
           float beta)
{
    __shared__ __align__(16) float tb[TG_MAXK][4];
    __shared__ __align__(16) float tc[TG_MAXK][4];
    __shared__ float tcls[TG_MAXK];
    __shared__ float tarea[TG_MAXK];
    __shared__ unsigned char tns[TG_MAXK];
    __shared__ float tkey[TG_MAXK];
    __shared__ int sh_n, sh_ns;
    __shared__ double sh_acc[LS_THREADS / 32];
    __shared__ unsigned sh_hit[LS_THREADS / 32];
    const int b = blockIdx.y;
    const int F2 = F * F, cells = 3 * F2, nch = 5 + C;
    pdl_trigger();
    const int n = load_truth(labels, b, K, stride, tb, tcls, &sh_n);
    if (threadIdx.x < LS_THREADS / 32) sh_hit[threadIdx.x] = 0u;
    if (n > 0) prep_truth(n, tb, tc, tarea, tns, tkey, &sh_ns);
    const int cell = blockIdx.x * LS_THREADS + threadIdx.x;
    double term = 0.0;
    float t4 = 0.0f;
    bool ignored = false;
    if (cell < cells) {
        const int a = cell / F2, r = cell - a * F2;
        const int j = r / F, i = r - j * F;
        const T *cp = raw + ((size_t)(b * 3 + a) * nch) * F2 + r;
        const float t0 = widen(cp[0]), t1 = widen(cp[(size_t)F2]), t2 = widen(cp[2 * (size_t)F2]), t3 = widen(cp[3 * (size_t)F2]);
        t4 = widen(cp[4 * (size_t)F2]);
        if (n > 0) {                                                   // :225-227: no labels => obj_mask stays 1
            // pred exactly as the train-mode YOLOLayer forms it (yololayer.py:126-134): grid units, no stride
            float sx, sy, ew, eh;
            spec_sigmoid2(t0, t1, sx, sy);                             // packed fp32x2 forms: the same bits as the scalar calls
            spec_exp2(t2, t3, ew, eh);
            if constexpr (SXY) {
                sx = __fadd_rn(__fmul_rn(sx, sxy), beta);
                sy = __fadd_rn(__fmul_rn(sy, sxy), beta);
            }
            const float ax = __fadd_rn(sx, (float)i), ay = __fadd_rn(sy, (float)j);
            const float aw = __fmul_rn(ew, A.maw[a]), ah = __fmul_rn(eh, A.mah[a]);
            ignored = iou_max_above(ax, ay, aw, ah, n, tb, tc, tarea, tns, sh_ns, ignore_thre);
        }
    }
    // Everything above is independent of k_loss_match (launched just before this kernel with programmatic dependent
    // launch): only the matched cells need its output.  Bitmap of the matched cells among this CTA's LS_THREADS cells.
    __syncthreads();
    pdl_wait();
    for (int t = threadIdx.x; t < n; t += LS_THREADS) {
        const int rel = tcell_all[(size_t)b * K + t] - (int)blockIdx.x * LS_THREADS;
        if (rel >= 0 && rel < LS_THREADS) atomicOr(&sh_hit[rel >> 5], 1u << (rel & 31));
    }
    __syncthreads();
    if (cell < cells) {
        const bool matched = (sh_hit[threadIdx.x >> 5] >> (threadIdx.x & 31)) & 1u;
        if (matched) ignored = false;                                  // matched cells are never ignored (:330)
        const float x = spec_sigmoidf(t4);
        float g = 0.0f;
        if (!ignored) {                                                // obj_mask = 1: BCE(x, t) with t = 1 on matched cells (:330,367,425)
            const float tg = matched ? 1.0f : 0.0f;
            term = (double)bce_term01(x, matched);
            g = __fmul_rn(__fmul_rn(bce_grad(x, tg), x), __fsub_rn(1.0f, x));
        }
        gobj[(size_t)b * cells + cell] = g;
    }
    term = warp_sum(term);
    if ((threadIdx.x & 31) == 0) sh_acc[threadIdx.x >> 5] = term;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < LS_THREADS / 32; ++w) s += sh_acc[w];
        if (s != 0.0) atomicAdd(&loss4[2], s);
    }
}

template <typename T>
__global__ void __launch_bounds__(LS_THREADS)
k_loss_bwd_obj(const float *__restrict__ gobj, const float *__restrict__ upstream, int F2, int C, long n_cells,
               T *__restrict__ grad_raw)
{
    const long c = (long)blockIdx.x * LS_THREADS + threadIdx.x;       // cell index over [B*3, F2]
    if (c >= n_cells) return;
    const long ba = c / F2;
    const int r = (int)(c - ba * F2);
    grad_raw[((size_t)ba * (5 + C) + 4) * F2 + r] = narrow(__fmul_rn(gobj[c], upstream[0]), grad_raw);
}

template <typename T>
__global__ void __launch_bounds__(LS_THREADS)
k_loss_bwd_sparse(const int *__restrict__ mcell, const float *__restrict__ mgrad, const float *__restrict__ upstream,
                  int F2, int K, int C, int n_gt, T *__restrict__ grad_raw)
{
    const int gt = blockIdx.x * (LS_THREADS / 32) + (threadIdx.x >> 5);   // one warp per (image, GT slot)
    if (gt >= n_gt) return;
    const int cell = mcell[gt];
    if (cell < 0) return;
    const int lane = threadIdx.x & 31, b = gt / K, nch = 5 + C, nk = 4 + C;
    const int a = cell / F2, r = cell - a * F2;
    T *gp = grad_raw + ((size_t)(b * 3 + a) * nch) * F2 + r;
    const float up = upstream[0];
    for (int kk = lane; kk < nk; kk += 32) gp[(size_t)(kk < 4 ? kk : kk + 1) * F2] = narrow(__fmul_rn(mgrad[(size_t)gt * nk + kk], up), gp);
}

static int fill_anchors(LossAnchors &A, const float *anchors_px, const int *anchor_mask3, float stride)
{
    for (int q = 0; q < 9; ++q) {                                                             // yololoss.py:139-150
        A.an.w[q] = (float)((double)anchors_px[2 * q] / (double)stride);
        A.an.h[q] = (float)((double)anchors_px[2 * q + 1] / (double)stride);
    }
    for (int a = 0; a < 3; ++a) {
        if (anchor_mask3[a] < 0 || anchor_mask3[a] > 8) return YL_ERR_ARG;
        A.an.mask[a] = anchor_mask3[a];
        A.maw[a] = A.an.w[anchor_mask3[a]];
        A.mah[a] = A.an.h[anchor_mask3[a]];
    }
    return YL_OK;
}

}  // namespace yl

using namespace yl;

template <typename T>
static int loss_forward_impl(const T *raw, const float *labels, int B, int F, int K, int C, int layer_no,
                             const float *anchors_px, const int *anchor_mask3, float ignore_thre, int iou_loss, float iou_norm,
                             float sxy, double *loss4, float *gobj, int *tcell_all, int *mcell, float *mgrad, int *status,
                             int chained, yl_stream_t stream)
{
    if (!raw || !labels || !anchors_px || !anchor_mask3 || !loss4 || !gobj || !tcell_all || !mcell || !mgrad) return YL_ERR_ARG;
    if (B <= 0 || F <= 0 || K <= 0 || K > TG_MAXK || C <= 0 || layer_no < 0 || layer_no > 2) return YL_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const float stride = (float)(8 << layer_no);
    LossAnchors A;
    const int rc = fill_anchors(A, anchors_px, anchor_mask3, stride);
    if (rc != YL_OK) return rc;
    // programmatic dependent launch along match(l) -> obj(l) -> match(l+1) -> ...: the latency-bound match kernels and the
    // small scales' obj kernels fill the tails of their neighbours (see the waits in the kernels).  k_loss_match reads raw /
    // labels and adds into loss4 / status BEFORE it waits, so it may only be launched programmatically behind this library's
    // own k_loss_obj (chained != 0): behind a foreign kernel (the producer of raw or labels, the fill of loss4) it is a
    // normal launch, fully ordered after everything earlier on the stream.
    const bool pdl = pdl_enabled();
    auto match = iou_loss == YL_IOU_LOSS_GIOU ? k_loss_match<T, YL_IOU_LOSS_GIOU>
               : iou_loss == YL_IOU_LOSS_DIOU ? k_loss_match<T, YL_IOU_LOSS_DIOU>
               : iou_loss == YL_IOU_LOSS_CIOU ? k_loss_match<T, YL_IOU_LOSS_CIOU> : k_loss_match<T, YL_IOU_LOSS_NONE>;
    const float beta = scale_xy_beta(sxy);
    YL_CUDA_TRY(launch_after(match, dim3(B, 8), dim3(LS_THREADS), 0, st, pdl && chained != 0, raw, labels, F, K, C, stride, A,
                             loss4, tcell_all, mcell, mgrad, status, iou_norm, sxy, beta));
    dim3 grid((3 * F * F + LS_THREADS - 1) / LS_THREADS, B);
    // a scale of exactly 1 is the unscaled objectness kernel (the same launches and bytes as without scale_x_y)
    YL_CUDA_TRY(launch_after(sxy != 1.0f ? k_loss_obj<T, true> : k_loss_obj<T, false>, grid, dim3(LS_THREADS), 0, st, pdl, raw,
                             labels, F, K, C, stride, A, ignore_thre, (const int *)tcell_all, loss4, gobj, sxy, beta));
    return YL_OK;
}

static int loss_forward_typed(const void *raw, int dtype, const float *labels, int B, int F, int K, int C, int layer_no,
                              const float *anchors_px, const int *anchor_mask3, float ignore_thre, int iou_loss, float iou_norm,
                              float sxy, double *loss4, float *gobj, int *tcell_all, int *mcell, float *mgrad, int *status,
                              int chained, yl_stream_t stream)
{
    if (iou_loss < YL_IOU_LOSS_NONE || iou_loss > YL_IOU_LOSS_CIOU || !(iou_norm >= 0.0f) || isinf(iou_norm)) return YL_ERR_ARG;
    // scale_x_y moves the predicted centre of the IoU box term; the BCE xy term has no scaled counterpart
    if (!scale_xy_valid(sxy) || (sxy != 1.0f && iou_loss == YL_IOU_LOSS_NONE)) return YL_ERR_ARG;
    switch (dtype) {
    case YL_DTYPE_F32:
        return loss_forward_impl((const float *)raw, labels, B, F, K, C, layer_no, anchors_px, anchor_mask3, ignore_thre, iou_loss,
                                 iou_norm, sxy, loss4, gobj, tcell_all, mcell, mgrad, status, chained, stream);
    case YL_DTYPE_F16:
        return loss_forward_impl((const __half *)raw, labels, B, F, K, C, layer_no, anchors_px, anchor_mask3, ignore_thre, iou_loss,
                                 iou_norm, sxy, loss4, gobj, tcell_all, mcell, mgrad, status, chained, stream);
    case YL_DTYPE_BF16:
        return loss_forward_impl((const __nv_bfloat16 *)raw, labels, B, F, K, C, layer_no, anchors_px, anchor_mask3, ignore_thre,
                                 iou_loss, iou_norm, sxy, loss4, gobj, tcell_all, mcell, mgrad, status, chained, stream);
    default:
        return YL_ERR_ARG;
    }
}

extern "C" int yl_loss_forward_ex2(const void *raw, int dtype, const float *labels, int B, int F, int K, int C, int layer_no,
                                   const float *anchors_px, const int *anchor_mask3, float ignore_thre, int iou_loss,
                                   float iou_normalizer, float scale_x_y, int chained, double *loss4, float *gobj, int *tcell_all,
                                   int *mcell, float *mgrad, int *status, yl_stream_t stream)
{
    return loss_forward_typed(raw, dtype, labels, B, F, K, C, layer_no, anchors_px, anchor_mask3, ignore_thre, iou_loss,
                              iou_normalizer, scale_x_y, loss4, gobj, tcell_all, mcell, mgrad, status, chained, stream);
}

extern "C" int yl_loss_forward_ex(const void *raw, int dtype, const float *labels, int B, int F, int K, int C, int layer_no,
                                  const float *anchors_px, const int *anchor_mask3, float ignore_thre, int iou_loss,
                                  float iou_normalizer, int chained, double *loss4, float *gobj, int *tcell_all, int *mcell,
                                  float *mgrad, int *status, yl_stream_t stream)
{
    return yl_loss_forward_ex2(raw, dtype, labels, B, F, K, C, layer_no, anchors_px, anchor_mask3, ignore_thre, iou_loss,
                               iou_normalizer, 1.0f, chained, loss4, gobj, tcell_all, mcell, mgrad, status, stream);
}

extern "C" int yl_loss_forward(const float *raw, const float *labels, int B, int F, int K, int C, int layer_no,
                               const float *anchors_px, const int *anchor_mask3, float ignore_thre,
                               double *loss4, float *gobj, int *tcell_all, int *mcell, float *mgrad, int *status,
                               yl_stream_t stream)
{
    return yl_loss_forward_ex(raw, YL_DTYPE_F32, labels, B, F, K, C, layer_no, anchors_px, anchor_mask3, ignore_thre,
                              YL_IOU_LOSS_NONE, 1.0f, 0, loss4, gobj, tcell_all, mcell, mgrad, status, stream);
}

extern "C" int yl_loss_forward_chained(const float *raw, const float *labels, int B, int F, int K, int C, int layer_no,
                                       const float *anchors_px, const int *anchor_mask3, float ignore_thre,
                                       double *loss4, float *gobj, int *tcell_all, int *mcell, float *mgrad, int *status,
                                       yl_stream_t stream)
{
    return yl_loss_forward_ex(raw, YL_DTYPE_F32, labels, B, F, K, C, layer_no, anchors_px, anchor_mask3, ignore_thre,
                              YL_IOU_LOSS_NONE, 1.0f, 1, loss4, gobj, tcell_all, mcell, mgrad, status, stream);
}

extern "C" int yl_loss_forward_typed(const void *raw, int dtype, const float *labels, int B, int F, int K, int C, int layer_no,
                                     const float *anchors_px, const int *anchor_mask3, float ignore_thre,
                                     double *loss4, float *gobj, int *tcell_all, int *mcell, float *mgrad, int *status,
                                     yl_stream_t stream)
{
    return yl_loss_forward_ex(raw, dtype, labels, B, F, K, C, layer_no, anchors_px, anchor_mask3, ignore_thre,
                              YL_IOU_LOSS_NONE, 1.0f, 0, loss4, gobj, tcell_all, mcell, mgrad, status, stream);
}

extern "C" int yl_loss_forward_chained_typed(const void *raw, int dtype, const float *labels, int B, int F, int K, int C,
                                             int layer_no, const float *anchors_px, const int *anchor_mask3, float ignore_thre,
                                             double *loss4, float *gobj, int *tcell_all, int *mcell, float *mgrad, int *status,
                                             yl_stream_t stream)
{
    return yl_loss_forward_ex(raw, dtype, labels, B, F, K, C, layer_no, anchors_px, anchor_mask3, ignore_thre,
                              YL_IOU_LOSS_NONE, 1.0f, 1, loss4, gobj, tcell_all, mcell, mgrad, status, stream);
}

template <typename T>
static int loss_backward_impl(const float *gobj, const int *mcell, const float *mgrad, const float *upstream,
                              int B, int F, int K, int C, T *grad_raw, cudaStream_t st)
{
    const int F2 = F * F;
    const long n_cells = (long)B * 3 * F2;
    YL_CUDA_TRY(cudaMemsetAsync(grad_raw, 0, sizeof(T) * (size_t)n_cells * (5 + C), st));
    k_loss_bwd_obj<T><<<(unsigned)((n_cells + LS_THREADS - 1) / LS_THREADS), LS_THREADS, 0, st>>>(gobj, upstream, F2, C, n_cells, grad_raw);
    YL_LAUNCH_CHECK();
    const int n_gt = B * K;
    k_loss_bwd_sparse<T><<<(n_gt + LS_THREADS / 32 - 1) / (LS_THREADS / 32), LS_THREADS, 0, st>>>(mcell, mgrad, upstream, F2, K, C, n_gt,
                                                                                                grad_raw);
    YL_LAUNCH_CHECK();
    return YL_OK;
}

extern "C" int yl_loss_backward_typed(const float *gobj, const int *mcell, const float *mgrad, const float *upstream,
                                      int B, int F, int K, int C, void *grad_raw, int dtype, yl_stream_t stream)
{
    if (dtype != YL_DTYPE_F32 && dtype != YL_DTYPE_F16 && dtype != YL_DTYPE_BF16) return YL_ERR_ARG;
    if (!gobj || !mcell || !mgrad || !upstream || !grad_raw || B <= 0 || F <= 0 || K <= 0 || C <= 0) return YL_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == YL_DTYPE_F16) return loss_backward_impl(gobj, mcell, mgrad, upstream, B, F, K, C, (__half *)grad_raw, st);
    if (dtype == YL_DTYPE_BF16) return loss_backward_impl(gobj, mcell, mgrad, upstream, B, F, K, C, (__nv_bfloat16 *)grad_raw, st);
    return loss_backward_impl(gobj, mcell, mgrad, upstream, B, F, K, C, (float *)grad_raw, st);
}

extern "C" int yl_loss_backward(const float *gobj, const int *mcell, const float *mgrad, const float *upstream,
                                int B, int F, int K, int C, float *grad_raw, yl_stream_t stream)
{
    return yl_loss_backward_typed(gobj, mcell, mgrad, upstream, B, F, K, C, grad_raw, YL_DTYPE_F32, stream);
}

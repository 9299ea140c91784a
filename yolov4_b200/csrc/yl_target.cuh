// yl_target.cuh -- device helpers shared by build_target (yl_target.cu) and the fused loss (yl_loss.cu): label loading,
// the literal bboxes_iou(xywh) of yolo/model/yololoss.py:16-91, and the GT -> cell assignment of :249-265.
#pragma once
#include "yl_common.cuh"

namespace yl {

constexpr int TG_THREADS = 256;
constexpr int TG_MAXK = 256;       // labels per image held in shared memory (cfg DATA.MAX_NUM_LABELS is 60)

// Loads image b's labels, counts nlabel = #(row sum > 0) (:219) and converts the FIRST n rows to grid units (:196-202).
__device__ __forceinline__ int load_truth(const float *__restrict__ labels, int b, int K, float stride, float (*tb)[4], float *cls, int *sh_n)
{
    if (threadIdx.x == 0) *sh_n = 0;
    __syncthreads();
    const float *lab = labels + (size_t)b * K * 5;
    for (int t = threadIdx.x; t < K; t += blockDim.x) {
        const float l0 = lab[5 * t], l1 = lab[5 * t + 1], l2 = lab[5 * t + 2], l3 = lab[5 * t + 3], l4 = lab[5 * t + 4];
        const float s = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(l0, l1), l2), l3), l4);
        if (s > 0.0f) atomicAdd(sh_n, 1);
        tb[t][0] = __fdiv_rn(l0, stride); tb[t][1] = __fdiv_rn(l1, stride);
        tb[t][2] = __fdiv_rn(l2, stride); tb[t][3] = __fdiv_rn(l3, stride);
        cls[t] = l4;
    }
    __syncthreads();
    return *sh_n;
}

// bboxes_iou(..., xyxy=False) for one pair, literal NaN-propagating form (:64-91)
__device__ __forceinline__ float iou_xywh(float ax, float ay, float aw, float ah, float bx, float by, float bw, float bh)
{
    const float ahw = __fmul_rn(aw, 0.5f), ahh = __fmul_rn(ah, 0.5f), bhw = __fmul_rn(bw, 0.5f), bhh = __fmul_rn(bh, 0.5f);
    const float tlx = nanmaxf(__fsub_rn(ax, ahw), __fsub_rn(bx, bhw)), tly = nanmaxf(__fsub_rn(ay, ahh), __fsub_rn(by, bhh));
    const float brx = nanminf(__fadd_rn(ax, ahw), __fadd_rn(bx, bhw)), bry = nanminf(__fadd_rn(ay, ahh), __fadd_rn(by, bhh));
    const float en = __fmul_rn((tlx < brx) ? 1.0f : 0.0f, (tly < bry) ? 1.0f : 0.0f);
    const float ai = __fmul_rn(__fmul_rn(__fsub_rn(brx, tlx), __fsub_rn(bry, tly)), en);
    return __fdiv_rn(ai, __fsub_rn(__fadd_rn(__fmul_rn(aw, ah), __fmul_rn(bw, bh)), ai));
}

__device__ __forceinline__ bool bounded(float v) { return fabsf(v) <= 1e18f; }   // false for NaN / inf / huge

struct AnchorSet { float w[9], h[9]; int mask[3]; };

// Channel of a GT's class one-hot in its cell's 5+C target row, target[..., 5 + cls] = 1 (:369): int16 truncation of the
// class id, then Python's negative-index wrap, so negative ids land on channels nch-1..0 (0..4: the box / objectness
// targets).  Valid when 0 <= channel < nch; the reference raises IndexError otherwise.
__device__ __forceinline__ int class_channel(float cls, int nch)
{
    const int k = 5 + (int)(short)(int)cls;
    return k < 0 ? k + nch : k;
}

// GT t of an image -> the cell it is assigned to on this layer, or -1 (yololoss.py:249-265, :206-207, :257): IoU of
// (0,0,w,h) against the nine (0,0,aw,ah) reference anchors, xyxy=True form; first max wins, NaN counts as the maximum
// (torch.argmax); the GT belongs to the layer when the best anchor is one of the layer's three; int16 truncation of the
// cell coordinates with Python's negative-index wrap.  *anc = best_n % 3.
__device__ __forceinline__ int match_truth(const float (&tbt)[4], int F, const AnchorSet &an, int *anc, int *status)
{
    const float w = tbt[2], h = tbt[3];
    const float area_a = __fmul_rn(__fsub_rn(w, 0.0f), __fsub_rn(h, 0.0f));
    int best_n = 0;
    float best = 0.0f;
    for (int q = 0; q < 9; ++q) {
        const float tlx = nanmaxf(0.0f, 0.0f), tly = tlx;
        const float brx = nanminf(w, an.w[q]), bry = nanminf(h, an.h[q]);
        const float en = __fmul_rn((tlx < brx) ? 1.0f : 0.0f, (tly < bry) ? 1.0f : 0.0f);
        const float ai = __fmul_rn(__fmul_rn(__fsub_rn(brx, tlx), __fsub_rn(bry, tly)), en);
        const float area_b = __fmul_rn(__fsub_rn(an.w[q], 0.0f), __fsub_rn(an.h[q], 0.0f));
        const float v = __fdiv_rn(ai, __fsub_rn(__fadd_rn(area_a, area_b), ai));
        if (q == 0) { best = v; best_n = 0; }
        else if (best == best && (v != v || v > best)) { best = v; best_n = q; }
    }
    int cell = -1;
    if (best_n == an.mask[0] || best_n == an.mask[1] || best_n == an.mask[2]) {          // :264-265
        int i = (int)(short)(int)tbt[0];                                                  // :206-207 int16 truncation
        int j = (int)(short)(int)tbt[1];
        if (i < 0) i += F;                                                                // python negative indexing
        if (j < 0) j += F;
        if (i < 0 || i >= F || j < 0 || j >= F) { if (status) atomicExch(status, 1); }
        else cell = ((best_n % 3) * F + j) * F + i;                                       // :257
    }
    *anc = best_n % 3;
    return cell;
}


// Per-GT data of the ignore test, derived once per CTA from tb (grid units).  A GT is "simple" when all its values are
// finite and bounded and its area is >= 0.  The simple GTs are stored SORTED BY AREA (tc = corners, tarea = areas, n - ns
// entries); tns lists the ns GTs that are not simple.  Must be called by every thread of the CTA; ends synchronised.
__device__ __forceinline__ void prep_truth(int n, const float (*tb)[4], float (*tc)[4], float *tarea, unsigned char *tns,
                                           float *tkey, int *sh_ns)
{
    if (threadIdx.x == 0) *sh_ns = 0;
    for (int t = threadIdx.x; t < n; t += (int)blockDim.x) {
        const bool simple = bounded(tb[t][0]) && bounded(tb[t][1]) && bounded(tb[t][2]) && bounded(tb[t][3]) &&
                            (__fmul_rn(tb[t][2], tb[t][3]) >= 0.0f);    // union = area_a + area_b stays > 0
        tkey[t] = simple ? __fmul_rn(tb[t][2], tb[t][3]) : -1.0f;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < n; t += (int)blockDim.x) {
        const float key = tkey[t];
        int below = 0, ns_before = 0;
        for (int u = 0; u < n; ++u) {
            const float ku = tkey[u];
            below += (ku >= 0.0f && (ku < key || (ku == key && u < t))) ? 1 : 0;
            ns_before += (ku < 0.0f && u < t) ? 1 : 0;
        }
        if (key >= 0.0f) {
            const float bhw = __fmul_rn(tb[t][2], 0.5f), bhh = __fmul_rn(tb[t][3], 0.5f);
            tc[below][0] = __fsub_rn(tb[t][0], bhw); tc[below][1] = __fsub_rn(tb[t][1], bhh);
            tc[below][2] = __fadd_rn(tb[t][0], bhw); tc[below][3] = __fadd_rn(tb[t][1], bhh);
            tarea[below] = key;
        } else {
            tns[ns_before] = (unsigned char)t;
            atomicAdd(sh_ns, 1);
        }
    }
    __syncthreads();
}

// First index q in [0, m) with v[q] >= x (UPPER: v[q] > x); v ascending.
template <bool UPPER>
__device__ __forceinline__ int area_bound(const float *v, int m, float x)
{
    int lo = 0, len = m;
    while (len > 0) {
        const int half = len >> 1;
        const float y = v[lo + half];
        const bool right = UPPER ? !(x < y) : (y < x);
        lo = right ? lo + half + 1 : lo;
        len = right ? len - half - 1 : half;
    }
    return lo;
}

// obj_mask = !(max_n IoU(box, GT_n) > ignore_thre) for one predicted box (ax, ay, aw, ah) in grid units (yololoss.py:276-294):
// returns true when the maximum is above the threshold.
__device__ __forceinline__ bool iou_max_above(float ax, float ay, float aw, float ah, int n, const float (*tb)[4],
                                              const float (*tc)[4], const float *tarea, const unsigned char *tns, int ns,
                                              float ignore_thre)
{
    // Fast path: with all coordinates finite and bounded and a strictly positive pred area, a GT that does not
    // overlap the cell's box has IoU exactly +0 (no NaN, no overflow), so only overlapping pairs need the division.
    // (and a non-negative threshold: an IoU of exactly 0 must not count as "above")
    const bool csimple = bounded(ax) && bounded(ay) && bounded(aw) && bounded(ah) && (__fmul_rn(aw, ah) > 0.0f) &&
                         (ignore_thre >= 0.0f);
    // max_n IoU > thr (:283-286) == "some IoU > thr and no IoU is NaN" (torch.max propagates NaN, and NaN > thr is False)
    bool above = false, nan_seen = false;
    if (!csimple) {
        for (int t = 0; t < n; ++t) {
            const float v = iou_xywh(ax, ay, aw, ah, tb[t][0], tb[t][1], tb[t][2], tb[t][3]);
            nan_seen |= (v != v);
            above |= (v > ignore_thre);
        }
        return above && !nan_seen;
    }
    for (int q = 0; q < ns; ++q) {
        const int t = tns[q];
        const float v = iou_xywh(ax, ay, aw, ah, tb[t][0], tb[t][1], tb[t][2], tb[t][3]);
        nan_seen |= (v != v);
        above |= (v > ignore_thre);
    }
    const float ahw = __fmul_rn(aw, 0.5f), ahh = __fmul_rn(ah, 0.5f);
    const float ax1 = __fsub_rn(ax, ahw), ay1 = __fsub_rn(ay, ahh), ax2 = __fadd_rn(ax, ahw), ay2 = __fadd_rn(ay, ahh);
    const float area_a = __fmul_rn(aw, ah);
    // IoU <= min(area) / max(area) (up to fp32 rounding, ~1e-6 relative): a simple GT whose area lies outside
    // [0.99 thr area_a, area_a / (0.99 thr)] cannot reach the threshold, and contributes neither a NaN nor an "above".
    // The simple GTs are sorted by area, so the pairs worth testing are one contiguous run found by two binary searches
    // (thr = 0: the whole list).
    const int m = n - ns;
    const float k = 0.99f * ignore_thre;
    const int q0 = area_bound<false>(tarea, m, k * area_a);
    const int q1 = (k > 0.0f) ? area_bound<true>(tarea, m, area_a / k) : m;
    for (int q = q0; q < q1; ++q) {
        const float4 g = *reinterpret_cast<const float4 *>(tc[q]);
        const float tlx = fmaxf(ax1, g.x), brx = fminf(ax2, g.z);
        const float tly = fmaxf(ay1, g.y), bry = fminf(ay2, g.w);
        if (tlx < brx && tly < bry) {
            // same operations as iou_xywh with en == 1; the quotient is only formed when the comparison is within
            // 0.1 % of the threshold (its rounding error is 6e-8)
            const float ai = __fmul_rn(__fsub_rn(brx, tlx), __fsub_rn(bry, tly));
            const float uni = __fsub_rn(__fadd_rn(area_a, tarea[q]), ai);
            const float tu = __fmul_rn(ignore_thre, uni);
            bool d;
            if (uni > 0.0f && uni < 3.0e38f && ai > 1.001f * tu && ai < 3.0e38f) d = true;
            else if (uni > 0.0f && uni < 3.0e38f && ai < 0.999f * tu) d = false;
            else d = __fdiv_rn(ai, uni) > ignore_thre;
            above |= d;
        }
    }
    return above && !nan_seen;
}

}  // namespace yl

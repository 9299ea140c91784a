// yl_nms.cu -- back end of the postprocess pipeline.
//
//   k_segment_nms_bins  one CTA per (image,class) candidate segment of up to SMALL_R records: sort by
//                       (score desc, box row desc) [utils.py:58 with stable tie order], greedy NMS dropping a box when
//                       IoU >= thr with any already kept box [utils.py:67-84]; the kept detections are written as
//                       finished 7-float rows at the front of the segment.
//   k_segment_nms_big   persistent CTAs over the queue of segments the small tier passes on (more than SMALL_R
//                       candidates, dense overlap graphs, thr <= 0): bitonic sort + 64-wide chunked bitmask NMS in
//                       shared memory (<= SMEM_R) or in place in global memory (degenerate all-ties inputs, SURVEY 7-2).
//   k_gather_rows       class-ascending concatenation of the kept rows of an image [utils.py:191-220] into
//                       out_rows[b] = (x1,y1,x2,y2,obj,cls_conf,cls) and the per-image counts.
//   k_select_topk       per-image detection cap (max_det), between the NMS tiers and the gather.
//   k_segment_nms_agnostic  class-agnostic NMS, one CTA per image, in place of the two NMS tiers (yl_nms_ex).
// The three NMS kernels take a template flag DIOU: the DIoU-NMS pair decision in place of IoU >= thr (yl_nms_ex2).
//
// Candidate record (written by the filter kernels, yl_filter.cu): two uint4,
//   A = {score bits, box row, cls_conf bits, obj_conf bits}    B = {x1, y1, x2, y2}
// so a segment is self-contained and the back end reads nothing but its own 32-byte records.
#include <math.h>
#include <stdlib.h>

#include "yl_common.cuh"
#include "../../include/yolo_head.h"

namespace yl {

constexpr int NMS_THREADS = 128;
constexpr int SMEM_R = kSmemR;
constexpr int CHUNK = 64;

// DIoU penalty (Zheng et al., AAAI 2020) of candidate a against kept box b, pen = num / den: squared distance of the box
// centres over the squared diagonal of the smallest box enclosing both, every operation one fp32 rounding in this order,
// max / min propagating NaN.  pen is >= 0 or NaN, so fl(iou - pen) >= thr implies fl(iou) >= thr: every conservative IoU
// pruning stays exact.  num and den are returned apart so that the boxes need not stay live until the division.
__device__ __forceinline__ float2 diou_terms(const float4 &a, const float4 &b)
{
    const float dx = __fsub_rn(__fmul_rn(__fadd_rn(a.x, a.z), 0.5f), __fmul_rn(__fadd_rn(b.x, b.z), 0.5f));
    const float dy = __fsub_rn(__fmul_rn(__fadd_rn(a.y, a.w), 0.5f), __fmul_rn(__fadd_rn(b.y, b.w), 0.5f));
    const float cw = __fsub_rn(nanmaxf(a.z, b.z), nanminf(a.x, b.x));
    const float ch = __fsub_rn(nanmaxf(a.w, b.w), nanminf(a.y, b.y));
    return make_float2(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fadd_rn(__fmul_rn(cw, cw), __fmul_rn(ch, ch)));
}

// IoU >= thr decision, bit-equal to utils.py:71-77 (fp32, separate roundings, (area_a + area_b) - inter, IEEE divide).
// Fast path (thr > 0, boxes sanitised so that NaN coordinates can never overlap): a pair whose intersection
// is empty has iou = 0 or NaN, neither of which is >= thr, so only overlapping pairs pay for the division.
// DIOU: the decision fl(iou - fl(num / den)) >= thr (diou_terms).  Every early `return false` holds for it too; the `return
// true` shortcut does not, so such a pair takes the exact quotient and the penalty.
template <bool DIOU = false>
__device__ __forceinline__ bool suppresses_pos(const float4 &a, float area_a, const float4 &b, float area_b, float thr)
{
    const float tlx = fmaxf(a.x, b.x), tly = fmaxf(a.y, b.y);
    const float brx = fminf(a.z, b.z), bry = fminf(a.w, b.w);
    if (!(tlx < brx && tly < bry)) return false;
    // Overlapping boxes have positive extents, so fl(inter) <= min(area) and union >= max(area): boxes whose areas
    // differ by more than the threshold ratio cannot reach it (common across anchor scales), no matter the overlap.
    {
        const float amin = fminf(area_a, area_b), amax = fmaxf(area_a, area_b);
        if (amax < 3.0e38f && amin < 0.999f * thr * amax) return false;
    }
    const float2 pen = DIOU ? diou_terms(a, b) : make_float2(0.0f, 0.0f);
    const float inter = __fmul_rn(__fsub_rn(brx, tlx), __fsub_rn(bry, tly));
    const float uni = __fsub_rn(__fadd_rn(area_a, area_b), inter);
    // fl(inter/uni) >= thr is decided without the division when inter is not within 0.1% of thr*uni (the quotient's
    // rounding error is 6e-8): only the rare near-threshold pair pays for the IEEE divide.
    if (uni > 0.0f && uni < 3.0e38f) {
        const float tu = thr * uni;
        if (inter < 0.999f * tu) return false;
        if (!DIOU && inter > 1.001f * tu && inter < 3.0e38f) return true;
    }
    if (DIOU) return __fsub_rn(__fdiv_rn(inter, uni), __fdiv_rn(pen.x, pen.y)) >= thr;
    return __fdiv_rn(inter, uni) >= thr;
}

// General path (thr <= 0 or unsanitised boxes): literal NaN-propagating formula.
template <bool DIOU = false>
__device__ __forceinline__ bool suppresses_any(const float4 &a, float area_a, const float4 &b, float area_b, float thr)
{
    const float tlx = nanmaxf(a.x, b.x), tly = nanmaxf(a.y, b.y);
    const float brx = nanminf(a.z, b.z), bry = nanminf(a.w, b.w);
    const float en = (tlx < brx && tly < bry) ? 1.0f : 0.0f;
    const float inter = __fmul_rn(__fmul_rn(__fsub_rn(brx, tlx), __fsub_rn(bry, tly)), en);
    const float iou = __fdiv_rn(inter, __fsub_rn(__fadd_rn(area_a, area_b), inter));
    if (DIOU) {
        const float2 pen = diou_terms(a, b);
        return __fsub_rn(iou, __fdiv_rn(pen.x, pen.y)) >= thr;
    }
    return iou >= thr;
}

__device__ __forceinline__ float box_area(const float4 &b) { return __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y)); }

__device__ __forceinline__ float4 sanitise(const float4 &b)
{
    // A box with a NaN coordinate never suppresses and is never suppressed (np.maximum/np.minimum propagate the
    // NaN, (tl < br) is False, iou is NaN).  Give it an empty extent so the fmaxf/fminf fast path agrees.
    if (b.x != b.x || b.y != b.y || b.z != b.z || b.w != b.w) return make_float4(kInf, kInf, -kInf, -kInf);
    return b;
}

__device__ __forceinline__ float4 as_float4(const uint4 &u)
{
    return make_float4(__uint_as_float(u.x), __uint_as_float(u.y), __uint_as_float(u.z), __uint_as_float(u.w));
}

// One finished output row (utils.py:177-184): (x1, y1, x2, y2, obj_conf, cls_conf, cls_idx as float).
__device__ __forceinline__ void store_row(float *o, const float4 &box, unsigned conf_bits, unsigned obj_bits, float fc)
{
    o[0] = box.x; o[1] = box.y; o[2] = box.z; o[3] = box.w;
    o[4] = __uint_as_float(obj_bits); o[5] = __uint_as_float(conf_bits); o[6] = fc;
}

// ---------------------------------------------------------------------------------------------------------------
// Small tier (the common case: ~150 candidates per (image,class) at conf 1e-4).  Everything in ~21 KB of shared memory.
//   1. rank by bucket sort: the 32-bit score keys are spread over RB buckets by their offset from the segment's smallest
//      key (monotone, so a bucket's records come after every record of lower buckets); a record's rank is its bucket's
//      first position plus the number of smaller unique 64-bit keys (score desc, row desc) in its own bucket;
//   2. candidate pairs by table lookup instead of an all-pairs loop: boxes are binned on x1, x2, y1, y2 (NBIN bins over
//      the segment's coordinate range) and on log2(area) (4 bins per octave); six prefix tables hold, per bin, the set
//      (bitmask over sorted positions) of boxes that CANNOT overlap / reach the IoU threshold with a box of that bin:
//         x1_i > x2_j | x2_i < x1_j | y1_i > y2_j | y2_i < y1_j | area_i >> area_j | area_i << area_j
//      so the candidate set of row j is one 6-way OR per 64 earlier boxes.  Binning is monotone, hence conservative: a
//      pair that overlaps (tl < br on both axes) and whose area ratio allows IoU >= thr is never excluded;
//   3. the surviving (i, j) pairs (~2 % of all pairs) are queued, then tested exactly by all threads (no divergence);
//   4. pairs with IoU >= thr set a bit in the transposed suppression matrix T[j]; one warp walks only the rows that
//      have such a bit, in score order: kept[j] = (T[j] & kept) == 0                       (utils.py:67-84);
//   5. the kept detections are staged in shared memory and stored as one contiguous run of 7-float rows.
// Segments with more than SMALL_R candidates, with more queued pairs than the queue holds, or with thr <= 0 (where
// every pair must go through the literal NaN-propagating formula) are passed on to the big tier.
// ---------------------------------------------------------------------------------------------------------------
constexpr int SMALL_R = 256;
constexpr int SMALL_W = SMALL_R / 32;
#ifndef YL_NMS_THREADS
#define YL_NMS_THREADS 128
#endif
constexpr int SMALL_THREADS = YL_NMS_THREADS;          // a multiple of 32
constexpr int SMALL_WARPS = SMALL_THREADS / 32;
constexpr int SMALL_EPT = (SMALL_R + SMALL_THREADS - 1) / SMALL_THREADS;      // records per thread, at most
#ifndef YL_NMS_NBIN
#define YL_NMS_NBIN 48
#endif
constexpr int NBIN = YL_NMS_NBIN;                     // bins per table (at most 64: bin numbers are packed in 6 bits)
#ifndef YL_NMS_QCAP
#define YL_NMS_QCAP 512
#endif
constexpr int QCAP_W = YL_NMS_QCAP;                     // queued pairs per warp
#ifndef YL_NMS_MINB
#define YL_NMS_MINB 10
#endif
constexpr int RB_LOG2 = 7, RB = 1 << RB_LOG2;           // rank buckets
constexpr int AREA_BIN_OFF = (127 + 4) << 2;            // float bits >> 21 of 16.0f: areas below 16 px^2 share bin 0

// Phase probe (tools/nms_phase_probe.py; never defined in the library build).  YL_NMS_PROBE: thread 0 of every CTA adds the
// clock64() cycles of each phase (closed by a barrier) to yl_nms_probe_acc[phase] and counts segments, queued
// pairs, rows with a suppressor and kept rows in the slots after the phases.  YL_NMS_PROBE_STOP=k: the CTA returns after phase
// k (the results are then wrong; only the kernel's time means something).
#if defined(YL_NMS_PROBE) || defined(YL_NMS_PROBE_STOP)
__device__ unsigned long long yl_nms_probe_acc[16];
extern "C" int yl_nms_probe_read(unsigned long long *host, int reset)
{
    cudaError_t e = cudaMemcpyFromSymbol(host, yl_nms_probe_acc, sizeof(yl_nms_probe_acc));
    if (e == cudaSuccess && reset) {
        static const unsigned long long zero[16] = {};
        e = cudaMemcpyToSymbol(yl_nms_probe_acc, zero, sizeof(zero));
    }
    return (int)e;
}
#endif
#ifdef YL_NMS_PROBE
#define NMS_PHASE(k)                                                                                                    \
    do {                                                                                                               \
        __syncthreads();                                                                                               \
        if (threadIdx.x == 0) {                                                                                        \
            const long long t_ = clock64();                                                                            \
            atomicAdd(&yl_nms_probe_acc[k], (unsigned long long)(t_ - probe_t));                                       \
            probe_t = t_;                                                                                              \
        }                                                                                                              \
    } while (0)
#define NMS_COUNT(k, v) do { if (threadIdx.x == 0) atomicAdd(&yl_nms_probe_acc[k], (unsigned long long)(v)); } while (0)
#elif defined(YL_NMS_PROBE_STOP)
#define NMS_PHASE(k) do { if ((k) == YL_NMS_PROBE_STOP) return; } while (0)
#define NMS_COUNT(k, v) do {} while (0)
#else
#define NMS_PHASE(k) do {} while (0)
#define NMS_COUNT(k, v) do {} while (0)
#endif

struct alignas(16) BinsSmem {
    union {
        struct {
            unsigned long long key[SMALL_R];            // (score key, ~row), grouped by bucket
            unsigned base[RB + 1];                      // records per bucket, then the bucket's first position
        } s;
        unsigned short queue[SMALL_WARPS][QCAP_W];      // (j << 8) | i candidate pairs, one queue per warp
    } a;
    float4 box[SMALL_R];                                // sorted
    uint2 co[SMALL_R];                                  // sorted {cls_conf bits, obj_conf bits}
    unsigned bins[SMALL_R];                             // sorted: bx1 | bx2<<6 | by1<<12 | by2<<18 | barea<<24 | invalid<<31
    union {
        unsigned long long tab[6][SMALL_W / 2][NBIN + 1];   // exclusion sets per bin, two 32-box words per entry (+1: conflict-free scan)
        unsigned T[SMALL_R][SMALL_W];                   // transposed suppression matrix
        float stage[SMALL_R * 7];                       // finished rows
    } b;
    float red[2][SMALL_WARPS];
    unsigned kred[2][SMALL_WARPS];
    unsigned qn[SMALL_WARPS];
    unsigned dirty[SMALL_W], keptw[SMALL_W], pref[SMALL_W + 1];
};

__device__ __forceinline__ int coord_bin(float v, float lo, float scale)
{
    // monotone in v: fp subtraction, multiplication by a non-negative constant, floor and clamping all are
    const int q = __float2int_rd(__fmul_rn(__fsub_rn(v, lo), scale));      // saturates on +-inf, 0 on NaN
    return min(max(q, 0), NBIN - 1);
}

// DIOU selects the DIoU decision for the exact tests of step 5; the bin tables stay exact for it (DIoU >= thr needs IoU >= thr).
template <bool DIOU>
__global__ void __launch_bounds__(SMALL_THREADS, YL_NMS_MINB)
k_segment_nms_bins(uint4 *__restrict__ cand, const unsigned *__restrict__ seg_count, unsigned *__restrict__ kept_count,
                   int C, int cap_seg, float thr, int area_k, int seg_first,
                   unsigned *__restrict__ big_count, unsigned *__restrict__ big_list)
{
    __shared__ BinsSmem S;
    const unsigned FULL = 0xFFFFFFFFu;
    const int seg = seg_first + blockIdx.x;
#ifdef YL_NMS_PROBE
    long long probe_t = clock64();
#endif
    pdl_trigger();
    {
        // zero the exclusion tables: independent of the input, so a CTA launched early (PDL) does it while the filter
        // kernel is still draining, and otherwise while the record loads are in flight
        uint4 *z = reinterpret_cast<uint4 *>(&S.b.tab[0][0][0]);
        constexpr int NZ = (int)(sizeof(S.b.tab) / sizeof(uint4));
        for (int i = threadIdx.x; i < NZ; i += SMALL_THREADS) z[i] = make_uint4(0u, 0u, 0u, 0u);
        for (int i = threadIdx.x; i < RB; i += SMALL_THREADS) S.a.s.base[i] = 0u;
        if (threadIdx.x < SMALL_WARPS) S.qn[threadIdx.x] = 0u;
        if (threadIdx.x < SMALL_W) S.dirty[threadIdx.x] = 0u;
    }
    pdl_wait();                                                 // segment counts and records of the filter kernel
    const unsigned cnt = seg_count[seg];
    if (cnt == 0u) return;                                      // kept_count was zeroed by yl_post_reset
    if (cnt > (unsigned)cap_seg) return;                        // overflow: reported through meta[], caller re-runs
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (cnt > (unsigned)SMALL_R || !(thr > 0.0f)) {
        if (tid == 0) big_list[atomicAdd(big_count, 1u)] = (unsigned)seg;
        return;
    }
    const int n = (int)cnt;
    const int nw = (n + 31) >> 5, nwp = (nw + 1) >> 1;
    uint4 *rec = cand + (size_t)seg * cap_seg * 2;
    NMS_PHASE(0);
    NMS_COUNT(9, 1);
    NMS_COUNT(12, n);

    // ---- 1. records -> registers; score keys -> shared memory; coordinate range of the segment ----
    uint4 ra[SMALL_EPT];
    float4 rb[SMALL_EPT];
#pragma unroll
    for (int u = 0; u < SMALL_EPT; ++u) {
        const int e = tid + u * SMALL_THREADS;
        ra[u] = make_uint4(0u, 0u, 0u, 0u);
        rb[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (e < n) { ra[u] = rec[2 * e]; rb[u] = as_float4(rec[2 * e + 1]); }
    }
    unsigned long long key[SMALL_EPT];
    bool valid[SMALL_EPT];
    float lo = kInf, hi = -kInf;
    unsigned kmin = 0xFFFFFFFFu, kmax = 0u;
#pragma unroll
    for (int u = 0; u < SMALL_EPT; ++u) {
        const int e = tid + u * SMALL_THREADS;
        key[u] = ~0ull;
        valid[u] = false;
        if (e < n) {
            const unsigned k32 = score_desc_bits(ra[u].x);
            key[u] = ((unsigned long long)k32 << 32) | (unsigned)(~ra[u].y);
            kmin = min(kmin, k32);
            kmax = max(kmax, k32);
            // only boxes with positive extents (hence no NaN) can overlap anything (suppresses_pos: tl < br on both axes)
            valid[u] = rb[u].x < rb[u].z && rb[u].y < rb[u].w;
            if (valid[u]) { lo = fminf(lo, fminf(rb[u].x, rb[u].y)); hi = fmaxf(hi, fmaxf(rb[u].z, rb[u].w)); }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fminf(lo, __shfl_xor_sync(FULL, lo, o));
        hi = fmaxf(hi, __shfl_xor_sync(FULL, hi, o));
    }
    kmin = __reduce_min_sync(FULL, kmin);
    kmax = __reduce_max_sync(FULL, kmax);
    if (lane == 0) { S.red[0][warp] = lo; S.red[1][warp] = hi; S.kred[0][warp] = kmin; S.kred[1][warp] = kmax; }
    __syncthreads();
    NMS_PHASE(1);

    // ---- 2. rank: bucket = (score key - smallest key) >> sh, sh such that every key of the segment has a bucket below RB ----
    int bk[SMALL_EPT], rank[SMALL_EPT];
    {
#pragma unroll
        for (int wq = 1; wq < SMALL_WARPS; ++wq) { kmin = min(kmin, S.kred[0][wq]); kmax = max(kmax, S.kred[1][wq]); }
        kmin = min(kmin, S.kred[0][0]);                         // kmin / kmax already hold this thread's own warp
        kmax = max(kmax, S.kred[1][0]);
        const int sh = max(0, (32 - __clz((int)(kmax - kmin))) - RB_LOG2);
#pragma unroll
        for (int u = 0; u < SMALL_EPT; ++u) {
            bk[u] = 0;
            rank[u] = 0;
            if (tid + u * SMALL_THREADS < n) {
                bk[u] = (int)(((unsigned)(key[u] >> 32) - kmin) >> sh);
                rank[u] = (int)atomicAdd(&S.a.s.base[bk[u]], 1u);     // position inside the bucket, for the scatter
            }
        }
    }
    __syncthreads();
    if (warp == 0) {
        // exclusive prefix of the bucket counts, RB / 32 buckets per lane
        constexpr int BL = RB / 32;
        unsigned c[BL], sum = 0u;
#pragma unroll
        for (int k = 0; k < BL; ++k) { c[k] = S.a.s.base[BL * lane + k]; sum += c[k]; }
        unsigned incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned v = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += v;
        }
        unsigned run = incl - sum;
#pragma unroll
        for (int k = 0; k < BL; ++k) { S.a.s.base[BL * lane + k] = run; run += c[k]; }
        if (lane == 31) S.a.s.base[RB] = incl;
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < SMALL_EPT; ++u)
        if (tid + u * SMALL_THREADS < n) S.a.s.key[S.a.s.base[bk[u]] + rank[u]] = key[u];
    __syncthreads();
#pragma unroll
    for (int u = 0; u < SMALL_EPT; ++u) {
        if (tid + u * SMALL_THREADS < n) {
            const int b0 = (int)S.a.s.base[bk[u]], b1 = (int)S.a.s.base[bk[u] + 1];
            int r = b0;
            for (int m = b0; m < b1; ++m) r += (S.a.s.key[m] < key[u]) ? 1 : 0;     // equal scores: ordered by ~row
            rank[u] = r;
        }
    }

    NMS_PHASE(2);

    // ---- 3. sorted arrays, bins, table inserts ----
    {
        lo = S.red[0][0]; hi = S.red[1][0];
#pragma unroll
        for (int wq = 1; wq < SMALL_WARPS; ++wq) { lo = fminf(lo, S.red[0][wq]); hi = fmaxf(hi, S.red[1][wq]); }
        lo = fmaxf(lo, -1.0e6f);
        hi = fminf(hi, 1.0e6f);
        float scale = __fdiv_rn((float)NBIN, __fsub_rn(hi, lo));
        if (!(scale > 0.0f && scale < 3.0e38f)) scale = 0.0f;  // empty / degenerate range: one bin, nothing is excluded
#pragma unroll
        for (int u = 0; u < SMALL_EPT; ++u) {
            const int e = tid + u * SMALL_THREADS;
            if (e < n) {
                const int r = rank[u];
                S.box[r] = rb[u];
                S.co[r] = make_uint2(ra[u].z, ra[u].w);
                const unsigned bit = 1u << (r & 31);
                const int wp = r >> 6, half = (r >> 5) & 1;
                unsigned bn = 0x80000000u;
                if (valid[u]) {
                    const int bx1 = coord_bin(rb[u].x, lo, scale), bx2 = coord_bin(rb[u].z, lo, scale);
                    const int by1 = coord_bin(rb[u].y, lo, scale), by2 = coord_bin(rb[u].w, lo, scale);
                    const int ab = min(max((int)(__float_as_uint(box_area(rb[u])) >> 21) - AREA_BIN_OFF, 0), NBIN - 1);
                    bn = (unsigned)bx1 | ((unsigned)bx2 << 6) | ((unsigned)by1 << 12) | ((unsigned)by2 << 18) | ((unsigned)ab << 24);
                    // tab[0][.][b] (suffix-OR) = { i : bx1_i - 1 >= b }  -> lookup at bx2_j gives x1_i > x2_j (in bins)
                    // tab[1][.][b] (prefix-OR) = { i : bx2_i + 1 <= b }  -> lookup at bx1_j gives x2_i < x1_j
                    if (bx1 >= 1) atomicOr(reinterpret_cast<unsigned *>(&S.b.tab[0][wp][bx1 - 1]) + half, bit);
                    if (bx2 + 1 < NBIN) atomicOr(reinterpret_cast<unsigned *>(&S.b.tab[1][wp][bx2 + 1]) + half, bit);
                    if (by1 >= 1) atomicOr(reinterpret_cast<unsigned *>(&S.b.tab[2][wp][by1 - 1]) + half, bit);
                    if (by2 + 1 < NBIN) atomicOr(reinterpret_cast<unsigned *>(&S.b.tab[3][wp][by2 + 1]) + half, bit);
                    // tab[4][.][b] (suffix-OR) = { i : ab_i - K >= b }   -> lookup at ab_j gives area_i too large for IoU >= thr
                    // tab[5][.][b] (prefix-OR) = { i : ab_i + K <= b }   -> lookup at ab_j gives area_i too small
                    if (ab - area_k >= 0) atomicOr(reinterpret_cast<unsigned *>(&S.b.tab[4][wp][ab - area_k]) + half, bit);
                    if (ab + area_k < NBIN) atomicOr(reinterpret_cast<unsigned *>(&S.b.tab[5][wp][ab + area_k]) + half, bit);
                } else {
                    atomicOr(reinterpret_cast<unsigned *>(&S.b.tab[1][wp][0]) + half, bit);     // in every prefix set: never a candidate
                }
                S.bins[r] = bn;
            }
        }
    }
    __syncthreads();
    NMS_PHASE(3);
    // prefix / suffix OR over the bins of 6 tables x nwp word pairs.  Eight lanes share a chain: each ORs its own run of
    // bins (independent loads), a 3-step shuffle scan over the eight run totals gives every lane its carry, and the runs
    // are stored back -- about 15 dependent steps where one lane per chain walked NBIN of them while three warps waited.
    {
        constexpr int BPL = (NBIN + 7) / 8;                     // bins per lane
        const int nchain = 6 * nwp;
        const int sub = tid & 7;
        for (int c0 = 0; c0 < nchain; c0 += SMALL_THREADS / 8) {    // CTA-uniform trip count: the shuffles run with a full mask
            const int c = c0 + (tid >> 3);
            const bool valid = c < nchain;
            const int t = valid ? c / nwp : 0, wp = valid ? c - t * nwp : 0;
            unsigned long long *p = &S.b.tab[t][wp][0];
            const bool fwd = (t & 1) != 0;                      // odd tables are prefix sets, even ones suffix sets
            unsigned long long v[BPL];
#pragma unroll
            for (int k = 0; k < BPL; ++k) {
                const int i = BPL * sub + k;                    // position along the scan direction
                v[k] = (valid && i < NBIN) ? p[fwd ? i : NBIN - 1 - i] : 0ull;
            }
#pragma unroll
            for (int k = 1; k < BPL; ++k) v[k] |= v[k - 1];
            unsigned long long incl = v[BPL - 1];
#pragma unroll
            for (int o = 1; o < 8; o <<= 1) {
                const unsigned long long y = __shfl_up_sync(FULL, incl, o, 8);
                if (sub >= o) incl |= y;
            }
            unsigned long long carry = __shfl_up_sync(FULL, incl, 1, 8);
            if (sub == 0) carry = 0ull;
#pragma unroll
            for (int k = 0; k < BPL; ++k) {
                const int i = BPL * sub + k;
                if (valid && i < NBIN) p[fwd ? i : NBIN - 1 - i] = v[k] | carry;
            }
        }
    }
    __syncthreads();
    NMS_PHASE(4);

    // ---- 4. candidate pairs (i < j) -> this warp's queue ----
    const int wbase = tid & ~31;
    unsigned qcount = 0u;
    bool overflow = false;
    {
        unsigned short *myq = S.a.queue[warp];
        const unsigned lt = (1u << lane) - 1u;
#pragma unroll
        for (int u = 0; u < SMALL_EPT; ++u) {
            const int j0 = wbase + u * SMALL_THREADS;           // first row of this warp's block of 32 (warp-uniform)
            if (j0 < n) {
                const int j = j0 + lane;
                const unsigned bn = (j < n) ? S.bins[j] : 0x80000000u;
                const bool act = !(bn >> 31);
                const int bx1 = bn & 63, bx2 = (bn >> 6) & 63, by1 = (bn >> 12) & 63, by2 = (bn >> 18) & 63, ab = (bn >> 24) & 63;
                const int wpj = j0 >> 6;
                for (int wp = 0; wp <= wpj; ++wp) {
                    const unsigned long long ex = S.b.tab[0][wp][bx2] | S.b.tab[1][wp][bx1] | S.b.tab[2][wp][by2] |
                                                  S.b.tab[3][wp][by1] | S.b.tab[4][wp][ab] | S.b.tab[5][wp][ab];
                    const int rel = j - 64 * wp;                 // rows of this warp lie in one 64-block: rel >= 0
                    const unsigned long long lim = (rel >= 64) ? ~0ull : ((1ull << rel) - 1ull);
                    const unsigned long long cw = act ? (~ex & lim) : 0ull;
                    unsigned c0 = (unsigned)cw, c1 = (unsigned)(cw >> 32);
                    const int ibase = 64 * wp;
                    while (__any_sync(FULL, (c0 | c1) != 0u)) {  // one pair per lane and round, low word first
                        const bool has = (c0 | c1) != 0u;
                        const unsigned m = __ballot_sync(FULL, has);
                        if (has) {
                            int ii;
                            if (c0) { ii = __ffs(c0) - 1; c0 &= c0 - 1u; }
                            else { ii = 32 + __ffs(c1) - 1; c1 &= c1 - 1u; }
                            const unsigned slot = qcount + __popc(m & lt);
                            if (slot < (unsigned)QCAP_W) myq[slot] = (unsigned short)((j << 8) | (ibase + ii));
                            else overflow = true;
                        }
                        qcount += __popc(m);
                    }
                }
            }
        }
        if (lane == 0) S.qn[warp] = min(qcount, (unsigned)QCAP_W);
    }
    if (__syncthreads_or(overflow)) {
        // dense overlap graph: more candidate pairs than the queue holds -- the chunked big tier takes the segment
        if (tid == 0) big_list[atomicAdd(big_count, 1u)] = (unsigned)seg;
        return;
    }
    unsigned qtotal = 0u;
#pragma unroll
    for (int wq = 0; wq < SMALL_WARPS; ++wq) qtotal += S.qn[wq];
    NMS_PHASE(5);
    NMS_COUNT(11, qtotal);

    // ---- 5. exact tests on the queued pairs, suppression matrix, resolve ----
    bool any_edges = false;
    if (qtotal != 0u) {                                          // CTA-uniform
        uint4 *z = reinterpret_cast<uint4 *>(&S.b.T[0][0]);
        for (int i = tid; i < n * (SMALL_W / 4); i += SMALL_THREADS) z[i] = make_uint4(0u, 0u, 0u, 0u);
        __syncthreads();
        bool found = false;
        // the queues laid end to end, so that the ~110 pairs of a typical segment take one round of the whole CTA rather
        // than one round of the first warp per queue
        for (unsigned p = tid; p < qtotal; p += SMALL_THREADS) {
            unsigned q = p;
            int wq = 0;
#pragma unroll
            for (int k = 0; k < SMALL_WARPS - 1; ++k) {
                const unsigned cq = S.qn[k];
                if (wq == k && q >= cq) { q -= cq; wq = k + 1; }
            }
            const unsigned e = S.a.queue[wq][q];
            const int j = e >> 8, i = e & 255;
            const float4 bj = S.box[j], bi = S.box[i];
            if (suppresses_pos<DIOU>(bj, box_area(bj), bi, box_area(bi), thr)) {
                atomicOr(&S.b.T[j][i >> 5], 1u << (i & 31));
                atomicOr(&S.dirty[j >> 5], 1u << (j & 31));
                found = true;
            }
        }
        any_edges = __syncthreads_or(found) != 0;
    }
    NMS_PHASE(6);
    if (tid < 32) {
        // lane w owns kept word w; only rows with a suppressor are visited, in score order (utils.py:67-84)
        unsigned keptw = 0u;
        if (lane < nw) keptw = (lane == nw - 1 && (n & 31)) ? ((1u << (n & 31)) - 1u) : FULL;
        if (any_edges) {
            for (int w = 0; w < nw; ++w) {
                unsigned d = S.dirty[w];
                while (d) {
                    const int jj = __ffs(d) - 1;
                    d &= d - 1u;
                    const unsigned t = (lane <= w) ? S.b.T[32 * w + jj][lane & (SMALL_W - 1)] : 0u;
                    if (__any_sync(FULL, (t & keptw) != 0u) && lane == w) keptw &= ~(1u << jj);
                }
            }
        }
        int c = __popc(keptw), incl = c;
#pragma unroll
        for (int o = 1; o < SMALL_W; o <<= 1) {
            const int v = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane < SMALL_W) { S.keptw[lane] = keptw; S.pref[lane] = (unsigned)(incl - c); }
        if (lane == SMALL_W - 1) { S.pref[SMALL_W] = (unsigned)incl; kept_count[seg] = (unsigned)incl; }
    }
    __syncthreads();
    NMS_PHASE(7);
    NMS_COUNT(13, __popc(S.dirty[0]) + __popc(S.dirty[1]) + __popc(S.dirty[2]) + __popc(S.dirty[3]) + __popc(S.dirty[4]) +
                  __popc(S.dirty[5]) + __popc(S.dirty[6]) + __popc(S.dirty[7]));
    NMS_COUNT(14, S.pref[SMALL_W]);

    // ---- 6. finished rows: stage in shared memory (the tables / T are dead), store as one contiguous run ----
    const float fc = (float)(seg % C);                           // utils.py:183 class id stored as float
    for (int j = tid; j < n; j += SMALL_THREADS) {
        const unsigned kw = S.keptw[j >> 5];
        if ((kw >> (j & 31)) & 1u) {
            const unsigned q = S.pref[j >> 5] + __popc(kw & ((1u << (j & 31)) - 1u));
            const uint2 co = S.co[j];
            store_row(S.b.stage + q * 7, S.box[j], co.x, co.y, fc);
        }
    }
    __syncthreads();
    {
        const int nf = (int)S.pref[SMALL_W] * 7;
        float4 *dst4 = reinterpret_cast<float4 *>(rec);
        const float4 *src4 = reinterpret_cast<const float4 *>(S.b.stage);
        for (int i = tid; i < (nf >> 2); i += SMALL_THREADS) dst4[i] = src4[i];
        const int tail = nf & ~3;
        if (tid < (nf & 3)) reinterpret_cast<float *>(rec)[tail + tid] = S.b.stage[tail + tid];
    }
    NMS_PHASE(8);
}

// ---- big tier ---------------------------------------------------------------------------------------------
struct SmemStore {
    unsigned long long *key;   // ascending sort key: (~score order bits) << 32 | ~row
    unsigned short *idx;       // sorted position -> record index
    const float4 *ubox;        // record order, original boxes
    bool pos;
    __device__ __forceinline__ void cswap(int i, int j)
    {
        const unsigned long long a = key[i], b = key[j];
        if (b < a) { key[i] = b; key[j] = a; const unsigned short t = idx[i]; idx[i] = idx[j]; idx[j] = t; }
    }
    __device__ __forceinline__ float4 get_box(int i) const { const float4 b = ubox[idx[i]]; return pos ? sanitise(b) : b; }
    __device__ __forceinline__ float get_area(int i) const { return box_area(ubox[idx[i]]); }
};

struct GlobalStore {
    uint4 *rec;                // record i: rec[2i] = {key hi, key lo, conf, obj}, rec[2i+1] = box
    bool pos;
    __device__ __forceinline__ void cswap(int i, int j)
    {
        const uint4 a = rec[2 * i], b = rec[2 * j];
        const unsigned long long ka = ((unsigned long long)a.x << 32) | a.y, kb = ((unsigned long long)b.x << 32) | b.y;
        if (kb < ka) {
            const uint4 ab = rec[2 * i + 1], bb = rec[2 * j + 1];
            rec[2 * i] = b; rec[2 * j] = a; rec[2 * i + 1] = bb; rec[2 * j + 1] = ab;
        }
    }
    __device__ __forceinline__ float4 get_box(int i) const
    {
        const float4 b = as_float4(rec[2 * i + 1]);
        return pos ? sanitise(b) : b;
    }
    __device__ __forceinline__ float get_area(int i) const { return box_area(as_float4(rec[2 * i + 1])); }
};

// Bitonic network in the "flip" formulation: every compare-exchange orders ascending, so virtual +inf padding
// beyond n never moves and non-power-of-two n works by skipping out-of-range partners.
template <class Store, int NT = NMS_THREADS>
__device__ void bitonic_sort(Store &s, int n)
{
    int P = 1;
    while (P < n) P <<= 1;
    for (int k = 2; k <= P; k <<= 1) {
        for (int i = threadIdx.x; i < n; i += NT) {
            const int l = i ^ (k - 1);
            if (l > i && l < n) s.cswap(i, l);
        }
        __syncthreads();
        for (int j = k >> 2; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n; i += NT) {
                const int l = i ^ j;
                if (l > i && l < n) s.cswap(i, l);
            }
            __syncthreads();
        }
    }
}

// Greedy NMS over the sorted segment, 64 candidates at a time:
//   (1) each chunk member is tested against every box kept so far (all threads, pairs in parallel)
//   (2) the 64x64 intra-chunk suppression matrix is built as one 64-bit row per member
//   (3) warp 0 resolves the chunk serially with the rows in registers
//   (4) survivors are appended to the kept list (compacted in place: a kept box never moves to a higher index)
// kept_of[q] = sorted position of the q-th kept box.  Returns the number kept.  DIOU selects the DIoU pair decision.
template <bool POS, bool DIOU, class Store, int NT = NMS_THREADS>
__device__ int greedy_nms(Store &s, int n, float thr, unsigned short *kept_s, unsigned *kept_g,
                          unsigned *sh_supp /*[2]*/, unsigned long long *sh_rows /*[64]*/, int *sh_nk)
{
    const int tid = threadIdx.x;
    if (tid == 0) *sh_nk = 0;
    __syncthreads();
    for (int c0 = 0; c0 < n; c0 += CHUNK) {
        const int cn = min(CHUNK, n - c0);
        const int nk = *sh_nk;
        if (tid < 2) sh_supp[tid] = 0u;
        if (tid < CHUNK) sh_rows[tid] = 0ull;
        __syncthreads();
        // (1) chunk x kept
        {
            const int i = tid & (CHUNK - 1);
            if (i < cn) {
                const float4 bi = s.get_box(c0 + i);
                const float ai = s.get_area(c0 + i);
                bool dead = false;
                for (int q = tid / CHUNK; q < nk && !dead; q += NT / CHUNK) {
                    const int kq = kept_s ? (int)kept_s[q] : (int)kept_g[q];
                    const float4 bk = s.get_box(kq);
                    const float ak = s.get_area(kq);
                    dead = POS ? suppresses_pos<DIOU>(bi, ai, bk, ak, thr) : suppresses_any<DIOU>(bi, ai, bk, ak, thr);
                }
                if (dead) atomicOr(&sh_supp[i >> 5], 1u << (i & 31));
            }
        }
        // (2) intra-chunk rows: row i has bit j set (j > i) when i suppresses j
        for (int pr = tid; pr < CHUNK * CHUNK; pr += NT) {
            const int i = pr / CHUNK, j = pr - i * CHUNK;
            if (j > i && j < cn) {
                const float4 bi = s.get_box(c0 + i), bj = s.get_box(c0 + j);
                const bool sup = POS ? suppresses_pos<DIOU>(bj, s.get_area(c0 + j), bi, s.get_area(c0 + i), thr)
                                     : suppresses_any<DIOU>(bj, s.get_area(c0 + j), bi, s.get_area(c0 + i), thr);
                if (sup) atomicOr(&sh_rows[i], 1ull << j);
            }
        }
        __syncthreads();
        // (3) serial resolve by warp 0
        if (tid < 32) {
            const unsigned long long r0 = sh_rows[tid], r1 = sh_rows[tid + 32];
            unsigned long long removed = ((unsigned long long)sh_supp[1] << 32) | sh_supp[0];
            unsigned long long keepbits = 0ull;
            for (int i = 0; i < cn; ++i) {
                const unsigned long long src = (i < 32) ? r0 : r1;
                const unsigned long long row = __shfl_sync(0xFFFFFFFFu, src, i & 31);
                if (!((removed >> i) & 1ull)) { keepbits |= 1ull << i; removed |= row; }
            }
            // (4) append survivors
            for (int i = tid; i < cn; i += 32)
                if ((keepbits >> i) & 1ull) {
                    const int q = nk + __popcll(keepbits & ((1ull << i) - 1ull));
                    if (kept_s) kept_s[q] = (unsigned short)(c0 + i); else kept_g[q] = (unsigned)(c0 + i);
                }
            if (tid == 0) *sh_nk = nk + __popcll(keepbits);
        }
        __syncthreads();
    }
    return *sh_nk;
}

// Persistent CTAs walk the list of segments the small tier passed on.
template <bool DIOU>
__global__ void __launch_bounds__(NMS_THREADS)
k_segment_nms_big(uint4 *__restrict__ cand, const unsigned *__restrict__ seg_count, unsigned *__restrict__ kept_count,
                  int C, int cap_seg, float thr, const unsigned *__restrict__ big_count, const unsigned *__restrict__ big_list,
                  unsigned *__restrict__ kept_scratch /* [B*C*cap_seg] u32, only when cap_seg > SMEM_R; else null */)
{
    __shared__ unsigned long long sh_key[SMEM_R];
    __shared__ unsigned short sh_idx[SMEM_R];
    __shared__ float4 sh_ubox[SMEM_R];
    __shared__ uint2 sh_uco[SMEM_R];
    __shared__ unsigned short sh_kept[SMEM_R];
    __shared__ unsigned long long sh_rows[CHUNK];
    __shared__ unsigned sh_supp[2];
    __shared__ int sh_nk;

    pdl_trigger();
    pdl_wait();                                                 // the queue filled by k_segment_nms_bins
    const unsigned nbig = *big_count;
    for (unsigned it = blockIdx.x; it < nbig; it += gridDim.x) {
        const int seg = (int)big_list[it];
        const int n = (int)seg_count[seg];
        uint4 *rec = cand + (size_t)seg * cap_seg * 2;
        float *rows = reinterpret_cast<float *>(rec);
        const float fc = (float)(seg % C);
        const int tid = threadIdx.x;
        const bool pos = thr > 0.0f;

        if (n <= SMEM_R) {
            for (int i = tid; i < n; i += NMS_THREADS) {
                const uint4 a = rec[2 * i];
                sh_key[i] = ((unsigned long long)score_desc_bits(a.x) << 32) | (unsigned)(~a.y);
                sh_idx[i] = (unsigned short)i;
                sh_uco[i] = make_uint2(a.z, a.w);
                sh_ubox[i] = as_float4(rec[2 * i + 1]);
            }
            __syncthreads();
            SmemStore s{sh_key, sh_idx, sh_ubox, pos};
            bitonic_sort(s, n);
            const int nk = pos ? greedy_nms<true, DIOU>(s, n, thr, sh_kept, nullptr, sh_supp, sh_rows, &sh_nk)
                               : greedy_nms<false, DIOU>(s, n, thr, sh_kept, nullptr, sh_supp, sh_rows, &sh_nk);
            for (int q = tid; q < nk; q += NMS_THREADS) {
                const int e = sh_idx[sh_kept[q]];
                const uint2 co = sh_uco[e];
                store_row(rows + (size_t)q * 7, sh_ubox[e], co.x, co.y, fc);
            }
            if (tid == 0) kept_count[seg] = (unsigned)nk;
        } else {
            // oversized segment: same algorithm in place in global memory (slow path, correctness only)
            for (int i = tid; i < n; i += NMS_THREADS) {
                const uint4 a = rec[2 * i];
                rec[2 * i] = make_uint4(score_desc_bits(a.x), ~a.y, a.z, a.w);
            }
            __syncthreads();
            GlobalStore s{rec, pos};
            bitonic_sort(s, n);
            unsigned *kept_g = kept_scratch + (size_t)seg * cap_seg;
            const int nk = pos ? greedy_nms<true, DIOU>(s, n, thr, nullptr, kept_g, sh_supp, sh_rows, &sh_nk)
                               : greedy_nms<false, DIOU>(s, n, thr, nullptr, kept_g, sh_supp, sh_rows, &sh_nk);
            // rows replace records in place: kept_g[q] >= q and a row (28 B) is shorter than a record (32 B), so the
            // rows of a chunk never reach a record a later chunk still has to read; go through registers chunk by chunk
            for (int q0 = 0; q0 < nk; q0 += NMS_THREADS) {
                const int q = q0 + tid;
                uint4 a = make_uint4(0u, 0u, 0u, 0u), bb = make_uint4(0u, 0u, 0u, 0u);
                if (q < nk) { a = rec[2 * (size_t)kept_g[q]]; bb = rec[2 * (size_t)kept_g[q] + 1]; }
                __syncthreads();
                if (q < nk) store_row(rows + (size_t)q * 7, as_float4(bb), a.z, a.w, fc);
                __syncthreads();
            }
            if (tid == 0) kept_count[seg] = (unsigned)nk;
        }
        __syncthreads();
    }
}

constexpr int GATHER_THREADS = 128;

// The kept rows of a segment are finished and contiguous at the front of the segment: concatenation is a copy.
__global__ void __launch_bounds__(GATHER_THREADS)
k_gather_rows(const uint4 *__restrict__ cand, const unsigned *__restrict__ seg_count, const unsigned *__restrict__ kept_count,
              int C, int cap_seg, int B, float *__restrict__ out_rows, long cap_out, int *__restrict__ meta, int seg_first)
{
    __shared__ unsigned sh_red[3][GATHER_THREADS / 32];
    pdl_wait();                                                 // kept counts and finished rows of both NMS tiers
    const int seg = seg_first + blockIdx.x;
    const int b = seg / C, c = seg - b * C;
    const int tid = threadIdx.x;
    // the first 2 x 128 float4s of the segment's finished rows (4 KB, the typical segment) are requested before the kept
    // counts are known, so the copy's round trip overlaps the prefix's instead of following it
    const float4 *src4 = reinterpret_cast<const float4 *>(cand + (size_t)seg * cap_seg * 2);
    const unsigned lim4 = (unsigned)cap_seg * 2u;
    float4 spec0 = make_float4(0.f, 0.f, 0.f, 0.f), spec1 = spec0;
    if ((unsigned)tid < lim4) spec0 = src4[tid];
    if ((unsigned)tid + GATHER_THREADS < lim4) spec1 = src4[tid + GATHER_THREADS];
    // exclusive prefix of kept counts over lower classes; class 0 also reduces the candidate statistics
    unsigned pre = 0u, mx = 0u, tot = 0u;
    for (int k = tid; k < C; k += GATHER_THREADS) {
        if (k < c) pre += kept_count[b * C + k];
        if (c == 0) { const unsigned s = seg_count[b * C + k]; mx = max(mx, s); tot += s; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        pre += __shfl_xor_sync(0xFFFFFFFFu, pre, o);
        tot += __shfl_xor_sync(0xFFFFFFFFu, tot, o);
        mx = max(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o));
    }
    if ((tid & 31) == 0) { sh_red[0][tid >> 5] = pre; sh_red[1][tid >> 5] = tot; sh_red[2][tid >> 5] = mx; }
    __syncthreads();
    pre = 0u; tot = 0u; mx = 0u;
#pragma unroll
    for (int w = 0; w < GATHER_THREADS / 32; ++w) { pre += sh_red[0][w]; tot += sh_red[1][w]; mx = max(mx, sh_red[2][w]); }
    const unsigned nk = kept_count[seg];
    if (tid == 0) {
        if (c == C - 1) meta[b] = (int)(pre + nk);
        if (c == 0) { meta[B + b] = (int)mx; meta[2 * B + b] = (int)tot; }
    }
    const unsigned nwr = (unsigned)min((long)nk, max(0L, cap_out - (long)pre));      // rows that fit the output capacity
    const float *src = reinterpret_cast<const float *>(cand + (size_t)seg * cap_seg * 2);
    float *dst = out_rows + ((size_t)b * cap_out + pre) * 7;
    // the source run is 16-byte aligned, the destination only 4-byte: 128-bit loads, scalar stores
    const unsigned nf = nwr * 7u, nf4 = nf >> 2;
    for (unsigned i = tid; i < nf4; i += GATHER_THREADS) {
        const float4 v = (i == (unsigned)tid) ? spec0 : ((i == (unsigned)tid + GATHER_THREADS) ? spec1 : src4[i]);
        float *d = dst + 4 * i;
        d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
    }
    if (tid < (nf & 3u)) dst[4 * nf4 + tid] = src[4 * nf4 + tid];
}

// ---- per-image detection cap (max_det) -----------------------------------------------------------------------
// The kept rows of an image are the first max_det of a stable descending sort of its class-ordered rows by
// s = fl(obj * cls_conf).  Inside a segment the rows are already in that order (score desc, ties by row desc), so the
// kept set is a prefix of every segment: k_select_topk only lowers kept_count and k_gather_rows copies the prefixes.
//   1. T = the max_det-th largest score key of the image: MSB-first radix select, SEL_PASSES histogram passes over the
//      keys (staged in shared memory when the image has at most SEL_SMEM_KEYS rows, otherwise re-read from the rows in
//      global memory on every pass: the degenerate all-ties images, correctness only);
//   2. per class, binary searches on the sorted segment give gt_c (keys > T) and eq_c (keys == T); the ties are admitted
//      in class order: take_c = gt_c + min(eq_c, max(0, need - sum_{c' < c} eq_c')).
constexpr int SEL_THREADS = 512;
constexpr int SEL_SMEM_KEYS = 16384;                         // 64 KB of keys: an image at 608 / conf 1e-4 keeps ~11.5k rows
constexpr int SEL_PASSES = 3;                                // digits of 11, 11 and 10 bits
constexpr int SEL_BINS = 1 << 11;
constexpr size_t SEL_SMEM_BYTES = sizeof(unsigned) * SEL_SMEM_KEYS;

// Order-preserving key of the nms score of a finished row; -0 and +0 get the same key.
__device__ __forceinline__ unsigned row_score_key(const float *row)
{
    const float s = __fadd_rn(__fmul_rn(row[4], row[5]), 0.0f);  // the filter kernels' score expression
    const unsigned u = __float_as_uint(s) == 0x80000000u ? 0u : __float_as_uint(s);
    return u ^ ((u >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}

__global__ void __launch_bounds__(SEL_THREADS)
k_select_topk(const uint4 *__restrict__ cand, unsigned *__restrict__ kept_count, int C, int cap_seg, int max_det,
              int *__restrict__ uncapped, int img_first)
{
    extern __shared__ unsigned sh_keys[];                     // [SEL_SMEM_KEYS], used when the image's rows fit
    __shared__ unsigned sh_hist[SEL_BINS];
    __shared__ unsigned sh_pre[YL_MAX_CLASSES + 1];           // exclusive prefix of kept_count over the classes
    __shared__ unsigned sh_eq[YL_MAX_CLASSES];
    __shared__ unsigned sh_warp[SEL_THREADS / 32];
    __shared__ unsigned sh_digit, sh_above;
    pdl_trigger();
    pdl_wait();                                                 // kept counts and finished rows of both NMS tiers
    const int b = img_first + blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float *seg_rows0 = reinterpret_cast<const float *>(cand + (size_t)b * C * cap_seg * 2);
    const size_t seg_stride = (size_t)cap_seg * 8;             // floats per segment (two uint4 per record)
    {
        // exclusive prefix over the classes (C <= 128: the first four warps, one class per lane)
        const unsigned v = tid < C ? kept_count[b * C + tid] : 0u;
        unsigned incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned u = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += u;
        }
        if (lane == 31) sh_warp[warp] = incl;
        __syncthreads();
        unsigned off = 0u;
        for (int w = 0; w < warp && w < YL_MAX_CLASSES / 32; ++w) off += sh_warp[w];
        if (tid < C) sh_pre[tid] = off + incl - v;
        if (tid == C - 1) sh_pre[C] = off + incl;
        __syncthreads();
    }
    const unsigned n = sh_pre[C];
    if (tid == 0 && uncapped) uncapped[b] = (int)n;
    if (n <= (unsigned)max_det) return;                         // CTA-uniform

    // key of the image's i-th row in class order
    auto global_key = [&](unsigned i) -> unsigned {
        int lo = 0, hi = C;                                     // largest c with sh_pre[c] <= i
        while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (sh_pre[mid] <= i) lo = mid; else hi = mid; }
        return row_score_key(seg_rows0 + (size_t)lo * seg_stride + (size_t)(i - sh_pre[lo]) * 7);
    };
    const bool staged = n <= (unsigned)SEL_SMEM_KEYS;
    if (staged) {
        for (unsigned i = tid; i < n; i += SEL_THREADS) sh_keys[i] = global_key(i);
    }

    // ---- 1. radix select: prefix / mask describe the digits of T fixed so far, need = rows still to take at >= prefix ----
    unsigned prefix = 0u, mask = 0u, need = (unsigned)max_det;
    int shift = 32;
#pragma unroll 1
    for (int p = 0; p < SEL_PASSES; ++p) {
        const int bits = p < 2 ? 11 : 10;
        shift -= bits;
        const unsigned dmask = (1u << bits) - 1u;
        for (int i = tid; i < SEL_BINS; i += SEL_THREADS) sh_hist[i] = 0u;
        __syncthreads();
        for (unsigned i = tid; i < n; i += SEL_THREADS) {
            const unsigned k = staged ? sh_keys[i] : global_key(i);
            if ((k & mask) == prefix) atomicAdd(&sh_hist[(k >> shift) & dmask], 1u);
        }
        __syncthreads();
        // the digit d where the count of keys with a larger digit is < need <= the count at >= d: a suffix sum over the bins,
        // each thread owning a run of SEL_BINS / SEL_THREADS bins from the top
        constexpr int RUN = SEL_BINS / SEL_THREADS;
        const int top = (int)dmask - RUN * tid;                 // this thread's bins: top, top-1, .., top-RUN+1
        unsigned run = 0u;
#pragma unroll
        for (int k = 0; k < RUN; ++k) if (top - k >= 0) run += sh_hist[top - k];
        unsigned incl = run;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) sh_warp[warp] = incl;
        __syncthreads();
        unsigned above = 0u;                                    // keys in the bins above this thread's run
        for (int w = 0; w < warp; ++w) above += sh_warp[w];
        above += incl - run;
        if (above < need && above + run >= need) {              // exactly one thread
            unsigned a = above;
            for (int k = 0; k < RUN; ++k) {
                const unsigned h = sh_hist[top - k];
                if (a + h >= need) { sh_digit = (unsigned)(top - k); sh_above = a; break; }
                a += h;
            }
        }
        __syncthreads();
        prefix |= sh_digit << shift;
        mask |= dmask << shift;
        need -= sh_above;
        __syncthreads();                                        // sh_digit / sh_above / sh_hist are rewritten next pass
    }
    const unsigned T = prefix;                                  // need (>= 1) of the keys equal to T are taken

    // ---- 2. per class: gt_c, eq_c by binary search on the descending keys of the segment's kept rows ----
    unsigned gt = 0u, eq = 0u;
    const int c = tid;
    if (c < C) {
        const unsigned base = sh_pre[c], cnt = sh_pre[c + 1] - base;
        auto key_at = [&](unsigned j) -> unsigned {
            return staged ? sh_keys[base + j] : row_score_key(seg_rows0 + (size_t)c * seg_stride + (size_t)j * 7);
        };
        unsigned lo = 0u, hi = cnt;                             // first j with key <= T
        while (lo < hi) { const unsigned mid = (lo + hi) >> 1; if (key_at(mid) > T) lo = mid + 1u; else hi = mid; }
        gt = lo;
        hi = cnt;                                               // first j with key < T
        while (lo < hi) { const unsigned mid = (lo + hi) >> 1; if (key_at(mid) >= T) lo = mid + 1u; else hi = mid; }
        eq = lo - gt;
        sh_eq[c] = eq;
    }
    __syncthreads();
    if (c < C) {
        unsigned before = 0u;
        for (int k = 0; k < c; ++k) before += sh_eq[k];
        const unsigned ties = need > before ? min(eq, need - before) : 0u;
        kept_count[b * C + c] = gt + ties;
    }
}

// ---- class-agnostic NMS ----------------------------------------------------------------------------------------------
// One greedy NMS per image over all its (box, class) candidates, in the image-wide order s desc, class asc, box row desc
// (the stable descending sort by s of the class-ascending concatenation of the per-class orders); a candidate is dropped when
// IoU >= thr with any earlier kept candidate, whatever either class is.  Only the FIRST copy of a box (its earliest candidate
// in that order) can matter when the literal self-IoU of the box is >= thr: a kept first copy suppresses the later copies,
// and a kept box that suppresses the first copy suppresses every later copy with the same bits.  So the image is reduced to
// first copies, plus every copy of a box whose self-IoU is below thr (NaN, empty or overflowing boxes, thr > 1), before the
// greedy pass.  k_segment_nms_agnostic (one CTA per image) replaces k_segment_nms_bins + k_segment_nms_big and leaves the
// workspace as they do: each class's kept rows at the front of its segment, kept_count written for every class.
//   1. first copies: a per-box table indexed by box row, in the image's slices of the obj / flag tables (dead once the emit or
//      dense filter kernel has run): tab_key[row] = min score key (atomicMin), then tab_cls[row] = lowest class at that key;
//   2. survivors are staged in shared memory (<= AGN_CAP) as (64-bit image-wide key, box, cls_conf / obj_conf), bitonic
//      sorted and suppressed with the chunked greedy_nms; each kept survivor's row goes to its rank within its class;
//   3. more survivors than AGN_CAP (conf <= 0, very large inputs): the same algorithm in global memory.  Every segment is
//      sorted in place, a survivor's image-wide rank is found by binary searches in the other segments, greedy_nms runs
//      over that order (order / kept lists in the agnostic scratch of yl_post_workspace_bytes_ex), and each segment's kept
//      records are compacted in place into rows (a row is shorter than a record and lands at or before its record).
constexpr int AGN_THREADS = 512;
constexpr int AGN_CAP = 4096;                                 // survivors staged in shared memory
constexpr int AGN_ROW_BITS = 25;                              // box rows < 2^25; the class takes the 7 bits above them
constexpr size_t AGN_SMEM_BYTES = (size_t)AGN_CAP * (sizeof(unsigned long long) + sizeof(float4) + sizeof(uint2) + 2 * sizeof(unsigned short));
static_assert(YL_MAX_CLASSES <= (1 << (32 - AGN_ROW_BITS)), "the class must fit above the row in the low key word");

// Image-wide ascending key: (score desc, class asc, row desc).
__device__ __forceinline__ unsigned long long agn_key(unsigned score_bits, int c, unsigned row)
{
    return ((unsigned long long)score_desc_bits(score_bits) << 32) | ((unsigned)c << AGN_ROW_BITS) |
           (~row & ((1u << AGN_ROW_BITS) - 1u));
}

// Survivors in global memory, in image-wide order: order[i] = c * cap_seg + e, the record's offset in the image's segments.
struct MergedStore {
    const uint4 *img;          // the image's first segment
    const unsigned *order;
    bool pos;
    __device__ __forceinline__ float4 get_box(int i) const
    {
        const float4 b = as_float4(img[2 * (size_t)order[i] + 1]);
        return pos ? sanitise(b) : b;
    }
    __device__ __forceinline__ float get_area(int i) const { return box_area(as_float4(img[2 * (size_t)order[i] + 1])); }
};

// Exclusive prefix of one flag per thread over the CTA; *total receives the sum.  Ends with a barrier.
__device__ __forceinline__ unsigned agn_block_scan(bool f, unsigned *sh_w /*[AGN_THREADS / 32]*/, unsigned &total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned m = __ballot_sync(0xFFFFFFFFu, f);
    if (lane == 0) sh_w[warp] = __popc(m);
    __syncthreads();
    unsigned before = 0u;
    total = 0u;
#pragma unroll
    for (int w = 0; w < AGN_THREADS / 32; ++w) { const unsigned v = sh_w[w]; before += w < warp ? v : 0u; total += v; }
    __syncthreads();
    return before + __popc(m & ((1u << lane) - 1u));
}

// DIOU: the DIoU decision, in the greedy pass and in the self test of the first-copy reduction.  The reduction stays exact:
// copies of a box have the same bits, so a decision against one copy is the decision against every copy.
template <bool DIOU>
__global__ void __launch_bounds__(AGN_THREADS, 1)
k_segment_nms_agnostic(uint4 *__restrict__ cand, const unsigned *__restrict__ seg_count, unsigned *__restrict__ kept_count,
                       int C, int cap_seg, float thr, unsigned *__restrict__ tab_key_all, unsigned *__restrict__ tab_cls_all,
                       long M4, unsigned *__restrict__ scratch, int img_first)
{
    extern __shared__ __align__(16) unsigned char agn_smem[];
    unsigned long long *sh_key = reinterpret_cast<unsigned long long *>(agn_smem);       // [AGN_CAP] staging order
    float4 *sh_box = reinterpret_cast<float4 *>(sh_key + AGN_CAP);                       // [AGN_CAP] staging order
    uint2 *sh_co = reinterpret_cast<uint2 *>(sh_box + AGN_CAP);                           // [AGN_CAP] {cls_conf, obj_conf} bits
    unsigned short *sh_idx = reinterpret_cast<unsigned short *>(sh_co + AGN_CAP);         // sorted position -> staging index
    unsigned short *sh_kept = sh_idx + AGN_CAP;                                           // kept survivors, sorted positions
    __shared__ unsigned sh_pre[YL_MAX_CLASSES + 1];           // exclusive prefix of seg_count over the classes
    __shared__ unsigned sh_cnt[AGN_THREADS / 32][YL_MAX_CLASSES];
    __shared__ unsigned sh_w[AGN_THREADS / 32];
    __shared__ unsigned long long sh_rows[CHUNK];
    __shared__ unsigned sh_supp[2];
    __shared__ int sh_nk;
    __shared__ unsigned sh_ns;

    pdl_trigger();
    pdl_wait();                                                 // segment counts and records of the filter kernel
    const int b = img_first + blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned FULL = 0xFFFFFFFFu;
    uint4 *img = cand + (size_t)b * C * cap_seg * 2;
    unsigned *tab_key = tab_key_all + (size_t)b * M4, *tab_cls = tab_cls_all + (size_t)b * M4;
    bool over = false;
    {
        // exclusive prefix over the classes (C <= 128: the first four warps, one class per lane)
        const unsigned v = tid < C ? seg_count[b * C + tid] : 0u;
        over = v > (unsigned)cap_seg;
        unsigned incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned u = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += u;
        }
        if (lane == 31) sh_w[warp] = incl;
        if (tid == 0) sh_ns = 0u;
        __syncthreads();
        unsigned off = 0u;
        for (int w = 0; w < warp && w < YL_MAX_CLASSES / 32; ++w) off += sh_w[w];
        if (tid < C) sh_pre[tid] = off + incl - v;
        if (tid == C - 1) sh_pre[C] = off + incl;
    }
    if (__syncthreads_or(over)) {                                // overflow: reported through meta[], caller re-runs
        for (int c = tid; c < C; c += AGN_THREADS) kept_count[b * C + c] = 0u;
        return;
    }
    const unsigned n = sh_pre[C];
    auto locate = [&](unsigned i, int &c) -> uint4 * {         // i-th record of the image in class order
        int lo = 0, hi = C;                                     // largest c with sh_pre[c] <= i
        while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (sh_pre[mid] <= i) lo = mid; else hi = mid; }
        c = lo;
        return img + ((size_t)lo * cap_seg + (i - sh_pre[lo])) * 2;
    };
    // ---- 1. first copies: the dense filter never writes the tables, so the entries in use are set here ----
    for (unsigned i = tid; i < n; i += AGN_THREADS) {
        int c;
        const unsigned row = locate(i, c)[0].y;
        tab_key[row] = FULL;
        tab_cls[row] = FULL;
    }
    __syncthreads();
    for (unsigned i = tid; i < n; i += AGN_THREADS) {
        int c;
        const uint4 a = locate(i, c)[0];
        atomicMin(&tab_key[a.y], score_desc_bits(a.x));
    }
    __syncthreads();
    for (unsigned i = tid; i < n; i += AGN_THREADS) {
        int c;
        const uint4 a = locate(i, c)[0];
        if (score_desc_bits(a.x) == __ldcg(&tab_key[a.y])) atomicMin(&tab_cls[a.y], (unsigned)c);
    }
    __syncthreads();
    // a copy survives when it is the box's first copy or when its box does not suppress itself (the literal self decision)
    auto survives = [&](const uint4 &a, const float4 &bx, int c) -> bool {
        if (score_desc_bits(a.x) == __ldcg(&tab_key[a.y]) && (unsigned)c == __ldcg(&tab_cls[a.y])) return true;
        const float ar = box_area(bx);
        return !suppresses_any<DIOU>(bx, ar, bx, ar, thr);
    };
    for (unsigned i = tid; i < n; i += AGN_THREADS) {
        int c;
        const uint4 *r = locate(i, c);
        const uint4 a = r[0];
        const float4 bx = as_float4(r[1]);
        if (survives(a, bx, c)) {
            const unsigned slot = atomicAdd(&sh_ns, 1u);
            if (slot < (unsigned)AGN_CAP) {
                sh_key[slot] = agn_key(a.x, c, a.y);
                sh_box[slot] = bx;
                sh_co[slot] = make_uint2(a.z, a.w);
                sh_idx[slot] = (unsigned short)slot;
            }
        }
    }
    __syncthreads();
    const unsigned ns = sh_ns;
    const bool pos = thr > 0.0f;

    if (ns <= (unsigned)AGN_CAP) {
        // ---- 2. shared-memory path.  Every read of the image's records is done: rows may overwrite them from here ----
        SmemStore s{sh_key, sh_idx, sh_box, pos};
        bitonic_sort<SmemStore, AGN_THREADS>(s, (int)ns);
        const int nk = pos ? greedy_nms<true, DIOU, SmemStore, AGN_THREADS>(s, (int)ns, thr, sh_kept, nullptr, sh_supp, sh_rows, &sh_nk)
                           : greedy_nms<false, DIOU, SmemStore, AGN_THREADS>(s, (int)ns, thr, sh_kept, nullptr, sh_supp, sh_rows, &sh_nk);
        // rank within the class: each warp takes a contiguous slice of the kept list; per-class counts per warp, a prefix over
        // the warps, then ranks inside the slice from peer masks
        const int q0 = (int)(((long)nk * warp) / (AGN_THREADS / 32)), q1 = (int)(((long)nk * (warp + 1)) / (AGN_THREADS / 32));
        for (int c = lane; c < C; c += 32) sh_cnt[warp][c] = 0u;
        __syncwarp();
        for (int q = q0 + lane; q < q1; q += 32)
            atomicAdd(&sh_cnt[warp][(int)(sh_key[sh_kept[q]] >> AGN_ROW_BITS) & (YL_MAX_CLASSES - 1)], 1u);
        __syncthreads();
        if (tid < C) {
            unsigned run = 0u;
            for (int w = 0; w < AGN_THREADS / 32; ++w) { const unsigned t = sh_cnt[w][tid]; sh_cnt[w][tid] = run; run += t; }
            kept_count[b * C + tid] = run;
        }
        __syncthreads();
        for (int qb = q0; qb < q1; qb += 32) {                  // warp-uniform trip count
            const int q = qb + lane;
            const bool act = q < q1;
            const unsigned am = __ballot_sync(FULL, act);
            if (act) {
                const int p = sh_kept[q];
                const int c = (int)(sh_key[p] >> AGN_ROW_BITS) & (YL_MAX_CLASSES - 1);
                const unsigned peers = __match_any_sync(am, c);
                const unsigned rank = sh_cnt[warp][c] + __popc(peers & ((1u << lane) - 1u));
                const int e = sh_idx[p];
                const uint2 co = sh_co[e];
                store_row(reinterpret_cast<float *>(img + (size_t)c * cap_seg * 2) + (size_t)rank * 7, sh_box[e], co.x, co.y, (float)c);
                __syncwarp(am);
                if (lane == __ffs(peers) - 1) sh_cnt[warp][c] += __popc(peers);
            }
            __syncwarp();
        }
        return;
    }

    // ---- 3. global-memory path (correctness only) ----
    unsigned *order = scratch + (size_t)b * C * cap_seg * 2, *kept_g = order + (size_t)C * cap_seg;
    unsigned *sh_spre = sh_cnt[1];                              // exclusive prefix of the survivors per class
    for (int c = tid; c < C; c += AGN_THREADS) sh_cnt[0][c] = 0u;
    __syncthreads();
    // records -> sort keys in place: survivors {score desc, ~row}, the others {~0, ~0} (sorted behind every survivor)
    for (unsigned i = tid; i < n; i += AGN_THREADS) {
        int c;
        uint4 *r = locate(i, c);
        const uint4 a = r[0];
        const bool sv = survives(a, as_float4(r[1]), c);
        r[0] = sv ? make_uint4(score_desc_bits(a.x), ~a.y, a.z, a.w) : make_uint4(FULL, FULL, a.z, a.w);
        if (sv) atomicAdd(&sh_cnt[0][c], 1u);
    }
    __syncthreads();
    for (int c = 0; c < C; ++c) {
        GlobalStore g{img + (size_t)c * cap_seg * 2, false};
        bitonic_sort<GlobalStore, AGN_THREADS>(g, (int)(sh_pre[c + 1] - sh_pre[c]));
    }
    if (tid == 0) {
        unsigned run = 0u;
        for (int c = 0; c < C; ++c) { sh_spre[c] = run; run += sh_cnt[0][c]; }
        sh_spre[C] = run;
    }
    __syncthreads();
    // image-wide rank of survivor (c, e): e, plus the survivors of lower classes with a score key <= its own, plus those of
    // higher classes with a key < its own (binary searches on the sorted segments)
    for (unsigned i = tid; i < ns; i += AGN_THREADS) {
        int lo = 0, hi = C;
        while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (sh_spre[mid] <= i) lo = mid; else hi = mid; }
        const int c = lo;
        const unsigned e = i - sh_spre[c];
        const unsigned k = img[((size_t)c * cap_seg + e) * 2].x;
        unsigned rank = e;
        for (int c2 = 0; c2 < C; ++c2) {
            if (c2 == c) continue;
            const uint4 *seg = img + (size_t)c2 * cap_seg * 2;
            unsigned l = 0u, h = sh_cnt[0][c2];                // first position whose key is > k (c2 < c) or >= k (c2 > c)
            while (l < h) {
                const unsigned mid = (l + h) >> 1;
                const unsigned km = seg[2 * (size_t)mid].x;
                if (c2 < c ? km <= k : km < k) l = mid + 1u; else h = mid;
            }
            rank += l;
        }
        order[rank] = (unsigned)c * (unsigned)cap_seg + e;
    }
    __syncthreads();
    MergedStore ms{img, order, pos};
    const int nk = pos ? greedy_nms<true, DIOU, MergedStore, AGN_THREADS>(ms, (int)ns, thr, nullptr, kept_g, sh_supp, sh_rows, &sh_nk)
                       : greedy_nms<false, DIOU, MergedStore, AGN_THREADS>(ms, (int)ns, thr, nullptr, kept_g, sh_supp, sh_rows, &sh_nk);
    // mark the kept records (the key word is free now), then compact every segment in place
    for (unsigned i = tid; i < ns; i += AGN_THREADS) img[2 * (size_t)order[i]].x = 0u;
    __syncthreads();
    for (int q = tid; q < nk; q += AGN_THREADS) img[2 * (size_t)order[kept_g[q]]].x = 1u;
    __syncthreads();
    for (int c = 0; c < C; ++c) {
        uint4 *seg = img + (size_t)c * cap_seg * 2;
        float *rows = reinterpret_cast<float *>(seg);
        const unsigned nsc = sh_cnt[0][c];
        unsigned done = 0u;
        for (unsigned e0 = 0; e0 < nsc; e0 += AGN_THREADS) {
            const unsigned e = e0 + tid;
            uint4 a = make_uint4(0u, 0u, 0u, 0u), bb = a;
            if (e < nsc) { a = seg[2 * (size_t)e]; bb = seg[2 * (size_t)e + 1]; }
            const bool kf = e < nsc && a.x == 1u;
            unsigned tot;
            const unsigned q = done + agn_block_scan(kf, sh_w, tot);     // barrier inside: every read of the chunk is done
            if (kf) store_row(rows + (size_t)q * 7, as_float4(bb), a.z, a.w, (float)c);
            __syncthreads();
            done += tot;
        }
        if (tid == 0) kept_count[b * C + c] = done;
    }
}

// Smallest K such that two positive areas whose bins (float bits >> 21: four per octave) differ by at least K have a
// ratio above 1/(0.999 thr) * (1 + 1e-3): then IoU <= amin/amax < thr with a margin far above fp32 rounding, which is
// the condition under which suppresses_pos returns false on the area test alone.
static int area_bin_gap(float thr)
{
    if (!(thr > 0.0f)) return NBIN + 1;
    const double need = 1.0 / (0.999 * (double)thr) * 1.001;
    for (int K = 1; K <= NBIN; ++K) {
        double worst = 1e300;
        for (int p = 0; p < 4; ++p) {
            // bins p+1 .. : lower edge of bin (p + K) over upper edge of bin p (= lower edge of bin p + 1)
            const int hi = p + K, lo = p + 1;
            const double Lh = ldexp(1.0 + (hi & 3) * 0.25, hi >> 2), Ll = ldexp(1.0 + (lo & 3) * 0.25, lo >> 2);
            worst = fmin(worst, Lh / Ll);
        }
        if (worst >= need) return K;
    }
    return NBIN + 1;
}

}  // namespace yl

using namespace yl;

// Scratch of the agnostic global-memory path, behind the standard workspace: u32 [B][2][C*cap_seg] (order, kept list).
static size_t agn_scratch_bytes(int B, int C, int cap_seg)
{
    return align_up(sizeof(unsigned) * 2 * (size_t)B * C * cap_seg, 256);
}

extern "C" size_t yl_post_workspace_bytes_ex(int B, long M, int C, int cap_seg, int agnostic)
{
    if (agnostic != 0 && agnostic != 1) return 0;
    const size_t base = yl_post_workspace_bytes(B, M, C, cap_seg);
    return (base == 0 || !agnostic) ? base : base + agn_scratch_bytes(B, C, cap_seg);
}

extern "C" int yl_nms_ex2(void *ws, size_t ws_bytes, int B, long M, int C, int cap_seg, float nms_thre, int max_det, int agnostic,
                          int diou, float *out_rows, long cap_out, int *meta, int *uncapped, int img_first, int img_count,
                          yl_stream_t stream)
{
    if (agnostic != 0 && agnostic != 1) return YL_ERR_ARG;
    if (diou != 0 && diou != 1) return YL_ERR_ARG;
    if (!ws || !out_rows || !meta || B <= 0 || M <= 0 || C <= 0 || cap_seg <= 0 || cap_out <= 0) return YL_ERR_ARG;
    if (img_first < 0 || img_count < 0 || img_first + img_count > B) return YL_ERR_ARG;
    if (max_det < 0 || max_det > cap_out) return YL_ERR_ARG;
    if (C > YL_MAX_CLASSES) return YL_ERR_CLASSES;
    // agnostic keys hold the box row in AGN_ROW_BITS bits; the global path addresses an image's records with 32 bits
    if (agnostic && (M >= (1L << AGN_ROW_BITS) || (unsigned long long)C * (unsigned long long)cap_seg > 0xFFFFFFFFull)) return YL_ERR_ARG;
    const PostLayout L = post_layout(B, M, C, cap_seg);
    if (ws_bytes < L.total + (agnostic ? agn_scratch_bytes(B, C, cap_seg) : 0)) return YL_ERR_WORKSPACE;
    if (img_count == 0) return YL_OK;
    char *w = (char *)ws;
    uint4 *cand = (uint4 *)(w + L.off_cand);
    unsigned *seg_count = (unsigned *)(w + L.off_seg_count);
    unsigned *kept_count = (unsigned *)(w + L.off_kept_count);
    unsigned *kept_scratch = (cap_seg > SMEM_R) ? (unsigned *)(w + L.off_kept_scratch) : nullptr;
    const int nseg = img_count * C, seg_first = img_first * C;
    unsigned *big_count = (unsigned *)(w + L.off_big_count) + img_first;
    unsigned *big_list = (unsigned *)(w + L.off_big_list) + seg_first;
    cudaStream_t st = (cudaStream_t)stream;
    // each kernel may become resident while its predecessor drains (PDL); it waits before reading the predecessor's output.
    // The first one follows the emit / dense filter kernel of yl_filter_* on the same stream.
    const bool pdl = pdl_enabled();
    // the same launches with either pair decision: only the instantiation differs
    if (agnostic) {
        const auto k_agn = diou ? k_segment_nms_agnostic<true> : k_segment_nms_agnostic<false>;
        // per device, so set on every call (a host-side attribute: allowed during stream capture)
        YL_CUDA_TRY(cudaFuncSetAttribute(k_agn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AGN_SMEM_BYTES));
        YL_CUDA_TRY(launch_after(k_agn, dim3(img_count), dim3(AGN_THREADS), AGN_SMEM_BYTES, st, pdl, cand,
                                 (const unsigned *)seg_count, kept_count, C, cap_seg, nms_thre, (unsigned *)(w + L.off_obj),
                                 (unsigned *)(w + L.off_flags), L.M4, (unsigned *)(w + L.total), img_first));
    } else {
        const auto k_bins = diou ? k_segment_nms_bins<true> : k_segment_nms_bins<false>;
        const auto k_big = diou ? k_segment_nms_big<true> : k_segment_nms_big<false>;
        YL_CUDA_TRY(launch_after(k_bins, dim3(nseg), dim3(SMALL_THREADS), 0, st, pdl, cand, seg_count, kept_count, C, cap_seg,
                                 nms_thre, area_bin_gap(nms_thre), seg_first, big_count, big_list));
        const int grid_big = nseg < 148 * 2 ? nseg : 148 * 2;
        YL_CUDA_TRY(launch_after(k_big, dim3(grid_big), dim3(NMS_THREADS), 0, st, pdl, cand, (const unsigned *)seg_count, kept_count,
                                 C, cap_seg, nms_thre, (const unsigned *)big_count, (const unsigned *)big_list, kept_scratch));
    }
    if (max_det > 0) {
        YL_CUDA_TRY(cudaFuncSetAttribute(k_select_topk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SEL_SMEM_BYTES));
        YL_CUDA_TRY(launch_after(k_select_topk, dim3(img_count), dim3(SEL_THREADS), SEL_SMEM_BYTES, st, pdl, (const uint4 *)cand,
                                 kept_count, C, cap_seg, max_det, uncapped, img_first));
    }
    YL_CUDA_TRY(launch_after(k_gather_rows, dim3(nseg), dim3(GATHER_THREADS), 0, st, pdl, (const uint4 *)cand, (const unsigned *)seg_count,
                             (const unsigned *)kept_count, C, cap_seg, B, out_rows, cap_out, meta, seg_first));
    return YL_OK;
}

extern "C" int yl_nms_ex(void *ws, size_t ws_bytes, int B, long M, int C, int cap_seg, float nms_thre, int max_det, int agnostic,
                         float *out_rows, long cap_out, int *meta, int *uncapped, int img_first, int img_count, yl_stream_t stream)
{
    return yl_nms_ex2(ws, ws_bytes, B, M, C, cap_seg, nms_thre, max_det, agnostic, 0, out_rows, cap_out, meta, uncapped, img_first,
                      img_count, stream);
}

extern "C" int yl_nms_topk(void *ws, size_t ws_bytes, int B, long M, int C, int cap_seg, float nms_thre, int max_det,
                           float *out_rows, long cap_out, int *meta, int *uncapped, int img_first, int img_count, yl_stream_t stream)
{
    return yl_nms_ex(ws, ws_bytes, B, M, C, cap_seg, nms_thre, max_det, 0, out_rows, cap_out, meta, uncapped, img_first, img_count,
                     stream);
}

extern "C" int yl_nms(void *ws, size_t ws_bytes, int B, long M, int C, int cap_seg, float nms_thre,
                      float *out_rows, long cap_out, int *meta, int img_first, int img_count, yl_stream_t stream)
{
    return yl_nms_topk(ws, ws_bytes, B, M, C, cap_seg, nms_thre, 0, out_rows, cap_out, meta, nullptr, img_first, img_count, stream);
}

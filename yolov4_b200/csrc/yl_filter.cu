// yl_filter.cu -- front ends of the postprocess pipeline: confidence filter -> candidate segments.
//
//   yl_filter_raw    fused YOLOLayer eval decode (yololayer.py:88-166) + xywh->xyxy (utils.py:117-126) + conf filter
//                    with multi-label expansion (utils.py:139-184) straight from the raw head tensors, in two kernels:
//                    a streaming flag pass (k_flag_tma, or k_flag_raw) and an exact pass over the flagged pairs
//                    (k_emit_flagged).
//   yl_filter_dense  the same filter over an already decoded [B,M,5+C] tensor (the literal postprocess() input):
//                    k_filter_dense_rows, or k_filter_dense_unaligned for a base that is not 16-byte aligned.
//
// Both append one self-contained 32-byte record per surviving (box,class) pair to the (image,class) segment
// cand[((b*C+c)*cap_seg + slot)*2 + {0,1}] = {score bits, box row, cls_conf bits, obj_conf bits}, {x1, y1, x2, y2}.
// Slot order inside a segment is arbitrary (atomics); the NMS stage sorts by the unique key (score, row), so final
// results are deterministic.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "yl_common.cuh"
#include "../../include/yolo_head.h"

namespace yl {

constexpr int K1_THREADS = 128;

// Conservative logit-domain bound: every class logit t with fl(obj * sigmoid(t)) >= thr satisfies t >= bound, so
// the streaming loop needs one compare per element and the exact spec-math test runs only on ~1% of them.
//   pass  =>  sigmoid_spec(t) >= (thr/obj)(1 - 2^-23)  =>  sigmoid(t) >= q' := (thr/obj)(1 - 1e-5)   (spec error < 4e-7)
//         =>  t >= logit(min(q', 0.9));  0.01 + 1e-3|L| absorbs the error of the fast __logf / division.
__device__ __forceinline__ float class_logit_bound(float obj, float thr)
{
    if (!(obj >= thr)) return kInf;            // sigmoid <= 1, so fl(obj*cls) <= obj < thr: no class can pass (also NaN obj)
    if (thr <= 0.0f) return -kInf;             // everything non-NaN passes
    float q = fminf((thr / obj) * (1.0f - 1e-5f), 0.9f);
    const float L = __logf(q / (1.0f - q));
    return L - 0.01f - 1e-3f * fabsf(L);
}

// bits |= bit unless t < lth (NaN logits set the bit too): FSETP + predicated LOP3, the whole per-logit cost of phase 1.
__device__ __forceinline__ void flag_or(unsigned &bits, float t, float lth, unsigned bit)
{
    asm("{\n\t.reg .pred p;\n\tsetp.lt.f32 p, %1, %2;\n\t@!p or.b32 %0, %0, %3;\n\t}" : "+r"(bits) : "f"(t), "f"(lth), "r"(bit));
}

// The same test for a packed pair of 16-bit logits (boxes 2j, 2j+1 of one class plane) against the pair's bounds rounded down to
// the element type once per box: one HSETP2 for two logits.  Still conservative (t >= lth implies t >= rd(lth)); a NaN half sets
// its bit, as in flag_or.
__device__ __forceinline__ void flag_or2(unsigned &b0, unsigned &b1, unsigned t2, unsigned l2, unsigned bit, __half)
{
    asm("{\n\t.reg .pred p, q;\n\tsetp.lt.f16x2 p|q, %2, %3;\n\t@!p or.b32 %0, %0, %4;\n\t@!q or.b32 %1, %1, %4;\n\t}"
        : "+r"(b0), "+r"(b1) : "r"(t2), "r"(l2), "r"(bit));
}
__device__ __forceinline__ void flag_or2(unsigned &b0, unsigned &b1, unsigned t2, unsigned l2, unsigned bit, __nv_bfloat16)
{
    asm("{\n\t.reg .pred p, q;\n\tsetp.lt.bf16x2 p|q, %2, %3;\n\t@!p or.b32 %0, %0, %4;\n\t@!q or.b32 %1, %1, %4;\n\t}"
        : "+r"(b0), "+r"(b1) : "r"(t2), "r"(l2), "r"(bit));
}
__device__ __forceinline__ unsigned short round_down_bits(float x, __half) { return __half_as_ushort(__float2half_rd(x)); }
__device__ __forceinline__ unsigned short round_down_bits(float x, __nv_bfloat16) { return __bfloat16_as_ushort(__float2bfloat16_rd(x)); }

// Flags one class plane's VEC logits of a lane into word w of bits.  fp32 and scalar 16-bit elements: flag_or on the (widened)
// value; 16-bit pairs: flag_or2 against the packed rounded-down bounds lpk.
template <typename T, int VEC, int NW>
__device__ __forceinline__ void flag_plane(unsigned (&bits)[VEC][NW], int w, const PlaneVec<T, VEC> &t, const float (&lth)[VEC],
                                           const unsigned (&lpk)[(VEC + 1) / 2], unsigned bit)
{
    if constexpr (sizeof(T) == 4 || VEC == 1) {
#pragma unroll
        for (int v = 0; v < VEC; ++v) flag_or(bits[v][w], t.at(v), lth[v], bit);
    } else {
#pragma unroll
        for (int j = 0; j < VEC / 2; ++j) flag_or2(bits[2 * j][w], bits[2 * j + 1][w], t.w[j], lpk[j], bit, T());
    }
}

// One scale of the head as the kernel sees it.
struct RawLayer {
    const void *raw;       // [B, 3, 5+C, F, F] of the element type the kernel is instantiated for
    int Fw, F2;
    int row_off;           // rows of the lower scales in the concatenated [M] axis (yolov4.py:324)
    int tiles;             // CTAs along x for this scale
    int vec;               // 4 = 128-bit loads (64-bit for 16-bit elements), 1 = scalar loads (planes not aligned, e.g. 19x19)
    int tma;               // streamed with TMA by k_flag_tma (else register-staged loads)
    int tile_boxes;        // boxes per tile (k_flag_tma: 128 TMA, 32 scalar; grid kernels: K1_THREADS * vec)
    float stride;
    float aw[3], ah[3];    // masked anchors in grid units (yololayer.py:73-76)
};
struct RawParams {
    RawLayer layer[3];
    int n_layers, C, cap_seg, img_first;
    int sparse;            // high thresholds: look at the objectness plane first and skip the class planes of dead vectors
    unsigned *reset;       // stages bit 2: the counters of the workspace, zeroed by the flag kernel itself (no memset node)
    int reset_words;
    long M;
    float thr;
    uint4 *cand;
    unsigned *seg_count;
    float *objtab;         // split filter: sigmoid(objectness) of every box, flag kernel -> emit kernel
    unsigned *flags;       // split filter: [NW][B*M4] flag words (see PostLayout)
    long M4;               // row pitch of flags / objtab in split mode (M rounded up to 4)
    long BM4;              // B * M4
};

constexpr int K1_WARPS = K1_THREADS / 32;
constexpr int K1_QCAP = 256;           // flagged (box,class) pairs a warp resolves per batch (a box has at most 128)

// Per-warp scratch of the exact pass.
struct EmitWarp {
    unsigned short ent[K1_QCAP];       // bit15 pass | box slot (7b) << 8 | class (7b)
    unsigned cls[K1_QCAP];             // sigmoid(class logit) bits of passing entries
    unsigned any[4], nan[4];           // per box slot: has a surviving pair / has a NaN class logit
    unsigned flg[4];                   // per box slot: belongs to the batch being resolved (speculative box fetch)
    float4 box[128];                   // decoded corners of the box slots that have a surviving pair
};

// Per-scale grid-sensitivity decode (scale_x_y, DESIGN.md section 1): centre = fl(fl(fl(sigmoid(t) * s) + beta) + cell), beta =
// -(s - 1) / 2.  A kernel parameter of its own after RawParams, so that the flag kernels and RawParams keep their layout.
struct ScaleXY { float s[3], beta[3]; };

// Grid-unit centre of one box: sigmoid(t) + cell, or with SXY the scaled form above.
template <bool SXY>
__device__ __forceinline__ float centre(float sg, int cell, float sxy, float beta)
{
    if constexpr (SXY) return __fadd_rn(__fadd_rn(__fmul_rn(sg, sxy), beta), (float)cell);
    else return __fadd_rn(sg, (float)cell);
}

template <bool SXY>
__device__ __forceinline__ float4 decode_box_v(float tx, float ty, float tw, float th, int Fw, int p, float aw, float ah, float stride,
                                               float sxy, float beta)
{
    const int gy = p / Fw, gx = p - gy * Fw;
    const float bx = __fmul_rn(centre<SXY>(spec_sigmoidf(tx), gx, sxy, beta), stride);
    const float by = __fmul_rn(centre<SXY>(spec_sigmoidf(ty), gy, sxy, beta), stride);
    const float bw = __fmul_rn(__fmul_rn(spec_expf(tw), aw), stride);
    const float bh = __fmul_rn(__fmul_rn(spec_expf(th), ah), stride);
    const float hw = __fmul_rn(bw, 0.5f), hh = __fmul_rn(bh, 0.5f);
    return make_float4(__fsub_rn(bx, hw), __fsub_rn(by, hh), __fadd_rn(bx, hw), __fadd_rn(by, hh));
}

// Decode one box (yololayer.py:150-162) and convert to corners (utils.py:117-126).
template <typename T, bool SXY>
__device__ __forceinline__ float4 decode_box(const T *bp, int F2, int Fw, int p, float aw, float ah, float stride, float sxy, float beta)
{
    const float tx = widen(bp[0]), ty = widen(bp[(size_t)F2]), tw = widen(bp[2 * (size_t)F2]), th = widen(bp[3 * (size_t)F2]);
    return decode_box_v<SXY>(tx, ty, tw, th, Fw, p, aw, ah, stride, sxy, beta);
}

// Exact pass over one batch of `total` queued (box slot, class) pairs of a warp tile.  All lanes take part:
//   1. the box planes of the batch's boxes are requested speculatively (lane i takes the i-th flagged box slot; the
//      conservative flag is tight, >95 % of flagged boxes survive) together with
//   2. the flagged logits (all loads of a 128-entry round in flight), then the exact spec-math test;
//   3. boxes with a surviving pair and no NaN class logit are decoded once, from the registers of step 1;
//   4. one 32-byte record per surviving pair is appended to its (image, class) segment: the slot atomics of four
//      entries per lane are issued before the first record is stored, so their round trips overlap.
// sobj[slot] = sigmoid(objectness) of the warp tile's boxes; wbase = plane 0 of the (image, anchor) at the tile's first box;
// E.flg = box slots of this batch.
__device__ __forceinline__ int nth_slot(const unsigned (&w)[4], const int (&c)[4], int i)
{
    int j = 0;
#pragma unroll
    for (int q = 1; q < 4; ++q) j = (i >= c[q]) ? q : j;
    const unsigned wsel = (j == 0) ? w[0] : ((j == 1) ? w[1] : ((j == 2) ? w[2] : w[3]));
    const int cs = (j == 0) ? c[0] : ((j == 1) ? c[1] : ((j == 2) ? c[2] : c[3]));
    return 32 * j + (int)__fns(wsel, 0, i - cs + 1);
}

template <typename T, int VEC, bool SXY>
__device__ __forceinline__ void emit_batch(const RawParams &P, const RawLayer &Ly, EmitWarp &E, const float *sobj,
                                           const T *wbase, int b, int a, int wp0, int total, float sxy, float beta)
{
    const int lane = threadIdx.x & 31;
    const int C = P.C, F2 = Ly.F2;
    const float thr = P.thr;
    const T *wcp = wbase + 5 * (size_t)F2;
    const int row_base = Ly.row_off + a * F2;                        // + p = row inside the image
    __syncwarp();                                                    // queue entries and flg/any/nan masks are visible
    unsigned fw[4];
    int fc[4], nflag = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        fw[j] = (j < VEC) ? E.flg[j] : 0u;
        fc[j] = nflag;
        nflag += __popc(fw[j]);
    }
    int sbs = -1;
    float tx = 0.f, ty = 0.f, tw = 0.f, th = 0.f;
    if (lane < nflag) {
        sbs = nth_slot(fw, fc, lane);
        const T *bp = wbase + sbs;
        tx = widen(bp[0]); ty = widen(bp[(size_t)F2]); tw = widen(bp[2 * (size_t)F2]); th = widen(bp[3 * (size_t)F2]);
    }
    for (int e0 = 0; e0 < total; e0 += 128) {
        float t[4];
        unsigned en[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int q = e0 + 32 * u + lane;
            en[u] = (q < total) ? E.ent[q] : 0u;
            t[u] = (q < total) ? widen(wcp[(size_t)(en[u] & 0x7F) * F2 + (en[u] >> 8)]) : 0.0f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int q = e0 + 32 * u + lane;
            if (q < total) {
                const int bs = en[u] >> 8;
                // a NaN class logit makes torch.max (utils.py:139) NaN and drops the whole row (:145)
                if (t[u] != t[u]) atomicOr(&E.nan[bs >> 5], 1u << (bs & 31));
                const float cls = spec_sigmoidf(t[u]);
                if (__fmul_rn(sobj[bs], cls) >= thr) {
                    atomicOr(&E.any[bs >> 5], 1u << (bs & 31));
                    E.cls[q] = __float_as_uint(cls);
                    E.ent[q] = (unsigned short)(en[u] | 0x8000u);
                }
            }
        }
    }
    __syncwarp();
    if (sbs >= 0 && (((E.any[sbs >> 5] & ~E.nan[sbs >> 5]) >> (sbs & 31)) & 1u))
        E.box[sbs] = decode_box_v<SXY>(tx, ty, tw, th, Ly.Fw, wp0 + sbs, Ly.aw[a], Ly.ah[a], Ly.stride, sxy, beta);
    for (int i = lane + 32; i < nflag; i += 32) {                    // more than 32 flagged boxes in the batch (dense inputs)
        const int bs = nth_slot(fw, fc, i);
        if (((E.any[bs >> 5] & ~E.nan[bs >> 5]) >> (bs & 31)) & 1u)
            E.box[bs] = decode_box<T, SXY>(wbase + bs, F2, Ly.Fw, wp0 + bs, Ly.aw[a], Ly.ah[a], Ly.stride, sxy, beta);
    }
    __syncwarp();
    for (int q0 = 0; q0 < total; q0 += 128) {
        unsigned slot[4], en[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int q = q0 + 32 * u + lane;
            en[u] = 0u;
            slot[u] = 0xFFFFFFFFu;
            if (q < total) {
                en[u] = E.ent[q];
                const int bs = (en[u] >> 8) & 0x7F;
                if ((en[u] & 0x8000u) && !((E.nan[bs >> 5] >> (bs & 31)) & 1u))
                    slot[u] = atomicAdd(&P.seg_count[(unsigned)(b * C + (int)(en[u] & 0x7F))], 1u);
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (slot[u] < (unsigned)P.cap_seg) {
                const int q = q0 + 32 * u + lane;
                const int bs = (en[u] >> 8) & 0x7F;
                const float cls = __uint_as_float(E.cls[q]);
                const float so = sobj[bs];
                const float s = __fadd_rn(__fmul_rn(so, cls), 0.0f);       // +0 canonicalises -0
                const unsigned seg = (unsigned)(b * C + (int)(en[u] & 0x7F));
                uint4 *r = P.cand + ((size_t)seg * P.cap_seg + slot[u]) * 2;
                const float4 bx = E.box[bs];
                r[0] = make_uint4(__float_as_uint(s), (unsigned)(row_base + wp0 + bs), __float_as_uint(cls), __float_as_uint(so));
                r[1] = make_uint4(__float_as_uint(bx.x), __float_as_uint(bx.y), __float_as_uint(bx.z), __float_as_uint(bx.w));
            }
        }
    }
    __syncwarp();
    if (lane < 4) { E.any[lane] = 0u; E.nan[lane] = 0u; E.flg[lane] = 0u; }
}

// Per-lane flagged-pair count and the warp's exclusive prefix (queue order: lane-major, then box, then class ascending).
template <int VEC, int NW>
__device__ __forceinline__ int pair_prefix(const float (&lth)[VEC], const unsigned (&bits)[VEC][NW], unsigned (&anyv)[VEC],
                                           int &first)
{
    const int lane = threadIdx.x & 31;
    int cntl = 0;
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
        unsigned any = 0u;
        int c = 0;
#pragma unroll
        for (int w = 0; w < NW; ++w) { any |= bits[v][w]; c += __popc(bits[v][w]); }
        if (lth[v] == kInf) { any = 0u; c = 0; }
        anyv[v] = any;
        cntl += c;
    }
    int incl = cntl;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += t;
    }
    first = incl - cntl;
    return __shfl_sync(0xFFFFFFFFu, incl, 31);
}

// Every lane writes its own pairs into the queue at the position the prefix sum gives it; flg gets the flagged box slots.
template <int VEC, int NW>
__device__ __forceinline__ void queue_pairs(const unsigned (&bits)[VEC][NW], const unsigned (&anyv)[VEC], int first,
                                            unsigned short *ent, unsigned *flg)
{
    const int lane = threadIdx.x & 31;
    int q = first;
#pragma unroll
    for (int v = 0; v < VEC; ++v)
        if (anyv[v]) {
            const int bs = lane * VEC + v;
            atomicOr(&flg[bs >> 5], 1u << (bs & 31));
            const unsigned hdr = (unsigned)bs << 8;
#pragma unroll
            for (int w = 0; w < NW; ++w) {
                unsigned m = bits[v][w];
                while (m) {
                    const int k = __ffs(m) - 1;
                    m &= m - 1u;
                    ent[q++] = (unsigned short)(hdr | (unsigned)(32 * w + k));
                }
            }
        }
}

// Phase 2 of a warp tile (32*VEC consecutive boxes, lane L owns boxes L*VEC .. L*VEC+VEC-1, bits[v][w] = flagged classes).
// Common case (at most K1_QCAP flagged pairs in the tile): every lane writes its own pairs into the queue at the
// position a warp prefix sum gives it, and the queue is resolved as one batch.  Dense tiles fall back to expanding the
// flag words box by box and resolving the queue in batches of whole boxes.  sobj must already hold
// sigmoid(objectness) per box slot.
template <typename T, int VEC, int NW, bool SXY>
__device__ __forceinline__ void emit_pairs(const RawParams &P, const RawLayer &Ly, int ba, int wp0,
                                           const float (&lth)[VEC], unsigned (&bits)[VEC][NW], EmitWarp &E, const float *sobj,
                                           float sxy, float beta)
{
    const unsigned FULL = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31;
    const int b = ba / 3, a = ba - 3 * b;
    unsigned anyv[VEC];
    int first;
    const int total = pair_prefix<VEC, NW>(lth, bits, anyv, first);
    if (total == 0) return;                                          // warp-uniform
    const T *wbase = (const T *)Ly.raw + ((size_t)ba * (5 + P.C)) * Ly.F2 + wp0;
    if (lane < 4) { E.any[lane] = 0u; E.nan[lane] = 0u; E.flg[lane] = 0u; }
    __syncwarp();
    if (total <= K1_QCAP) {
        queue_pairs<VEC, NW>(bits, anyv, first, E.ent, E.flg);
        emit_batch<T, VEC, SXY>(P, Ly, E, sobj, wbase, b, a, wp0, total, sxy, beta);
        return;
    }
    unsigned flagged[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) flagged[v] = __ballot_sync(FULL, anyv[v] != 0u);
    int qb = 0;
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
        unsigned lanes = flagged[v];
        while (lanes) {                                              // warp-uniform loop over the flagged boxes
            const int L = __ffs(lanes) - 1;
            lanes &= lanes - 1;
            unsigned m[NW];
            int n = 0;
#pragma unroll
            for (int w = 0; w < NW; ++w) { m[w] = __shfl_sync(FULL, bits[v][w], L); n += __popc(m[w]); }
            if (qb + n > K1_QCAP) { emit_batch<T, VEC, SXY>(P, Ly, E, sobj, wbase, b, a, wp0, qb, sxy, beta); qb = 0; __syncwarp(); }
            const int bs = L * VEC + v;
            if (lane == 0) E.flg[bs >> 5] |= 1u << (bs & 31);
            const unsigned hdr = (unsigned)bs << 8;
#pragma unroll
            for (int w = 0; w < NW; ++w) {
                if ((m[w] >> lane) & 1u) E.ent[qb + __popc(m[w] & ((1u << lane) - 1u))] = (unsigned short)(hdr | (32 * w + lane));
                qb += __popc(m[w]);
            }
        }
    }
    if (qb) emit_batch<T, VEC, SXY>(P, Ly, E, sobj, wbase, b, a, wp0, qb, sxy, beta);
}

// One tile = K1_THREADS*VEC consecutive boxes of one (image, anchor).  Phase 1 (the flag kernels) streams the class
// planes with one compare per logit; phase 2 (k_emit_flagged, whose shared memory this is) resolves the ~1% flagged
// pairs warp-cooperatively (all lanes, all loads in flight together) instead of serially in the lane that owns the box.
struct LdgSmem {
    EmitWarp e[K1_WARPS];
    float sobj[K1_WARPS][128];
};

// Register-staged phase 1 for one lane: VEC consecutive boxes starting at p0 of (image, anchor) ba.  KB class planes are
// requested per batch: eight for fp32, sixteen for 16-bit elements, so a lane keeps as many bytes in flight as the fp32 form of
// its vector shape (16-bit vectors are 64-bit loads: a 128-bit form with 8 boxes per lane would need twice the flag-word
// registers and spills at 80 classes).
template <typename T, int VEC, int NW>
__device__ __forceinline__ void ldg_stream(const RawParams &P, const RawLayer &Ly, int ba, int p0, bool inb,
                                           float (&obj)[VEC], float (&lth)[VEC], unsigned (&bits)[VEC][NW])
{
    constexpr int KB = sizeof(T) == 4 ? 8 : 16;
    const int C = P.C, F2 = Ly.F2;
    const float thr = P.thr;
    const int nch = 5 + C;
    const T *base = (const T *)Ly.raw + ((size_t)ba * nch) * F2 + (inb ? p0 : 0);
    const T *cp = base + 5 * (size_t)F2;
    // The objectness plane and the first KB class planes are requested together: the bound needs sigmoid(obj),
    // but the class loads do not, so no load latency is spent with nothing else in flight.
    // (With a high threshold -- detect setting, conf 0.2 -- almost every box is dead on objectness alone; then the
    // objectness plane is read first and the class planes of dead vectors are never requested.)
    PlaneVec<T, VEC> tob, t0[KB];
    const int kn0 = min(KB, C);
    bool any_alive = false;
    if (P.sparse) {
        if (inb) tob.load(base + 4 * (size_t)F2);
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            obj[v] = inb ? spec_sigmoidf(tob.at(v)) : 0.0f;
            lth[v] = inb ? class_logit_bound(obj[v], thr) : kInf;
            any_alive |= (lth[v] != kInf);
        }
        if (any_alive) {
#pragma unroll
            for (int u = 0; u < KB; ++u)
                if (u < kn0) t0[u].load(cp + (size_t)u * F2);
        }
    } else {
        if (inb) {
            tob.load(base + 4 * (size_t)F2);
#pragma unroll
            for (int u = 0; u < KB; ++u)
                if (u < kn0) t0[u].load(cp + (size_t)u * F2);
        }
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            obj[v] = inb ? spec_sigmoidf(tob.at(v)) : 0.0f;
            lth[v] = inb ? class_logit_bound(obj[v], thr) : kInf;
            any_alive |= (lth[v] != kInf);
        }
    }
    unsigned lpk[(VEC + 1) / 2];                                     // 16-bit pairs: the bounds rounded down, packed
#pragma unroll
    for (int j = 0; j < (VEC + 1) / 2; ++j) {
        if constexpr (sizeof(T) == 2 && VEC > 1)
            lpk[j] = (unsigned)round_down_bits(lth[2 * j], T()) | ((unsigned)round_down_bits(lth[2 * j + 1], T()) << 16);
        else
            lpk[j] = 0u;
    }
#pragma unroll
    for (int v = 0; v < VEC; ++v)
#pragma unroll
        for (int w = 0; w < NW; ++w) bits[v][w] = 0u;
    if (any_alive) {
#pragma unroll
        for (int u = 0; u < KB; ++u)
            if (u < kn0) flag_plane<T, VEC, NW>(bits, 0, t0[u], lth, lpk, 1u << u);
#pragma unroll
        for (int w = 0; w < NW; ++w) {
            const int kn = min(32, C - 32 * w);
#pragma unroll
            for (int kk = (w == 0 ? KB : 0); kk < 32; kk += KB) {    // fully unrolled: every bit mask is an immediate
                if (kk < kn) {
                    PlaneVec<T, VEC> t[KB];
#pragma unroll
                    for (int u = 0; u < KB; ++u)
                        if (kk + u < kn) t[u].load(cp + (size_t)(32 * w + kk + u) * F2);
#pragma unroll
                    for (int u = 0; u < KB; ++u)
                        if (kk + u < kn) flag_plane<T, VEC, NW>(bits, w, t[u], lth, lpk, 1u << (kk + u));
                }
            }
        }
    }
#pragma unroll
    for (int v = 0; v < VEC; ++v)
        if (lth[v] == kInf) {
#pragma unroll
            for (int w = 0; w < NW; ++w) bits[v][w] = 0u;
        }
}

// ---------------------------------------------------------------------------------------------------------------
// The streaming kernel does nothing but load, compare and store 16 bytes per box (flag words + sigmoid(objectness)),
// so it runs at the memory system's pace; k_emit_flagged then resolves the flagged pairs.
// ---------------------------------------------------------------------------------------------------------------
template <typename T, int VEC, int NW>
__device__ __forceinline__ void flag_tile(const RawParams &P, const RawLayer &Ly, int tile, int ba)
{
    const int p0 = (tile * K1_THREADS + threadIdx.x) * VEC;
    if (p0 >= Ly.F2) return;                                         // F2 % VEC == 0: a vector is all in or all out
    float obj[VEC], lth[VEC];
    unsigned bits[VEC][NW];
    ldg_stream<T, VEC, NW>(P, Ly, ba, p0, true, obj, lth, bits);
    const int b = ba / 3, a = ba - 3 * b;
    const size_t r = (size_t)b * P.M4 + (Ly.row_off + a * Ly.F2 + p0);
    // the emit kernel reads these 16 B per box right after this kernel: keep them in L2 while the raw stream passes through
    if (VEC == 4) {
        stg_keep4(P.objtab + r, make_uint4(__float_as_uint(obj[0]), __float_as_uint(obj[1 % VEC]), __float_as_uint(obj[2 % VEC]),
                                           __float_as_uint(obj[3 % VEC])));
#pragma unroll
        for (int w = 0; w < NW; ++w)
            stg_keep4(P.flags + (size_t)w * P.BM4 + r, make_uint4(bits[0][w], bits[1 % VEC][w], bits[2 % VEC][w], bits[3 % VEC][w]));
    } else {
        stg_keep1(P.objtab + r, __float_as_uint(obj[0]));
#pragma unroll
        for (int w = 0; w < NW; ++w) stg_keep1(P.flags + (size_t)w * P.BM4 + r, bits[0][w]);
    }
}

#ifndef YL_FLAG_MINB
#define YL_FLAG_MINB 8
#endif
template <typename T, int NW>
__global__ void __launch_bounds__(K1_THREADS, YL_FLAG_MINB)
k_flag_raw(const __grid_constant__ RawParams P)
{
    pdl_trigger();
    if (P.reset_words > 0 && blockIdx.y == 0) {
        // yl_post_reset folded into this kernel: nothing reads the counters before the emit kernel, which waits for this
        // grid to complete
        for (int i = blockIdx.x * K1_THREADS + threadIdx.x; i < P.reset_words; i += gridDim.x * K1_THREADS) P.reset[i] = 0u;
    }
    const int ba = P.img_first * 3 + blockIdx.y;
    int tile = blockIdx.x;
    int l = 0;
    while (l < P.n_layers - 1 && tile >= P.layer[l].tiles) { tile -= P.layer[l].tiles; ++l; }
    if (P.layer[l].vec == 4) flag_tile<T, 4, NW>(P, P.layer[l], tile, ba);
    else flag_tile<T, 1, NW>(P, P.layer[l], tile, ba);
}

template <typename T, int VEC, int NW, bool SXY>
__device__ __forceinline__ void emit_tile(const RawParams &P, const RawLayer &Ly, int tile, int ba, LdgSmem &sm, float sxy, float beta)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int p0 = (tile * K1_THREADS + threadIdx.x) * VEC;
    const bool inb = p0 < Ly.F2;
    const int b = ba / 3, a = ba - 3 * b;
    const size_t r = (size_t)b * P.M4 + (Ly.row_off + a * Ly.F2 + (inb ? p0 : 0));
    float lth[VEC];
    unsigned bits[VEC][NW];
#pragma unroll
    for (int v = 0; v < VEC; ++v) lth[v] = 0.0f;
    if (VEC == 4) {
#pragma unroll
        for (int w = 0; w < NW; ++w) {
            const uint4 m = inb ? *reinterpret_cast<const uint4 *>(P.flags + (size_t)w * P.BM4 + r) : make_uint4(0u, 0u, 0u, 0u);
            bits[0][w] = m.x; bits[1 % VEC][w] = m.y; bits[2 % VEC][w] = m.z; bits[3 % VEC][w] = m.w;
        }
    } else {
#pragma unroll
        for (int w = 0; w < NW; ++w) bits[0][w] = inb ? P.flags[(size_t)w * P.BM4 + r] : 0u;
    }
    // sigmoid(objectness) is requested together with the flag words (one round trip, not two)
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
    if (inb) {
        if (VEC == 4) o = *reinterpret_cast<const float4 *>(P.objtab + r);
        else o.x = P.objtab[r];
    }
    unsigned any = 0u;
#pragma unroll
    for (int v = 0; v < VEC; ++v)
#pragma unroll
        for (int w = 0; w < NW; ++w) any |= bits[v][w];
    if (!__any_sync(0xFFFFFFFFu, any != 0u)) return;                 // warp-uniform: nothing flagged in these 32*VEC boxes
    if (VEC == 4) *reinterpret_cast<float4 *>(&sm.sobj[warp][lane * 4]) = o;
    else sm.sobj[warp][lane] = o.x;
    emit_pairs<T, VEC, NW, SXY>(P, Ly, ba, (tile * K1_THREADS + warp * 32) * VEC, lth, bits, sm.e[warp], sm.sobj[warp], sxy, beta);
}

#ifndef YL_EMIT_MINB
#define YL_EMIT_MINB 8
#endif
template <typename T, int NW, bool SXY>
__device__ __forceinline__ void emit_flagged(const RawParams &P, const ScaleXY &S)
{
    __shared__ LdgSmem sm;
    pdl_trigger();
    pdl_wait();                                                      // the flag words / sigmoid(obj) of k_flag_raw
    // Reverse order of k_flag_raw: the planes that kernel streamed last are still in L2 (126 MB of the 495 MB), so the
    // flagged logits / box planes of the first tiles handled here are re-read from L2 instead of DRAM.
    const int ba = P.img_first * 3 + ((int)gridDim.y - 1 - (int)blockIdx.y);
    int tile = (int)gridDim.x - 1 - (int)blockIdx.x;
    int l = 0;
    while (l < P.n_layers - 1 && tile >= P.layer[l].tiles) { tile -= P.layer[l].tiles; ++l; }
    if (P.layer[l].vec == 4) emit_tile<T, 4, NW, SXY>(P, P.layer[l], tile, ba, sm, S.s[l], S.beta[l]);
    else emit_tile<T, 1, NW, SXY>(P, P.layer[l], tile, ba, sm, S.s[l], S.beta[l]);
}

// Two overloads of one kernel: the plain decode, and the grid-sensitivity decode with the per-scale scale_x_y of S.
template <typename T, int NW>
__global__ void __launch_bounds__(K1_THREADS, YL_EMIT_MINB)
k_emit_flagged(const __grid_constant__ RawParams P)
{
    emit_flagged<T, NW, false>(P, ScaleXY{});
}

template <typename T, int NW>
__global__ void __launch_bounds__(K1_THREADS, YL_EMIT_MINB)
k_emit_flagged(const __grid_constant__ RawParams P, const __grid_constant__ ScaleXY S)
{
    emit_flagged<T, NW, true>(P, S);
}

// ---------------------------------------------------------------------------------------------------------------
// Bulk and tensor-map (TMA) copies into shared memory, each completing on a transaction mbarrier the consumer waits on:
// the class-plane rings of k_flag_tma and the row batches of k_filter_dense_rows.
// ---------------------------------------------------------------------------------------------------------------
#ifndef YL_WT_KC
#define YL_WT_KC 8
#endif
constexpr int WT_KC = YL_WT_KC;            // class planes per TMA box (one ring stage of k_flag_tma)
constexpr int WT_BOX = 128;                // boxes per warp tile (32 lanes x float4)

__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity)
{
    unsigned ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// 2-D tiled TMA load (SASS UTMALDG): box [WT_KC planes x WT_BOX boxes] at (column x, plane row y) of a scale's
// [B*3*(5+C) planes, F*F] view.  Out-of-range columns/rows are zero-filled and still count as transferred bytes.
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, int x, int y, unsigned long long *bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(smem_u32(dst)), "l"(map), "r"(x), "r"(y), "r"(smem_u32(bar)) : "memory");
}

struct TmaMaps { CUtensorMap m[3]; };

struct WtTile {
    const float *src;      // plane 0 of this (image, anchor) at the tile's first box
    int layer, ba, p0, np; // np = boxes in the tile (<= 128, multiple of 4); np == 0: no tile
    int row0;              // plane row of class 0 in the scale's 2-D view: ba*(5+C) + 5
    int tma;
};

// ---------------------------------------------------------------------------------------------------------------
// TMA form of the streaming FLAG pass (YL_FLAG=tma): the same output as k_flag_raw (flag words + sigmoid(objectness), 16 B per
// box, for k_emit_flagged), produced by ONE persistent CTA per SM that needs a quarter of the register file:
//   * streaming warps   private TMA rings ([WT_KC class planes x 128 boxes] per stage, UTMALDG.2D + transaction mbarriers,
//                       objectness plane by a 1-D bulk copy): the bytes in flight live in shared memory, not in registers
//                       (k_flag_raw keeps 8 CTAs x 128 threads x 64 registers busy to have 128 KB in flight per SM);
//   * scalar warps      the scales whose planes are not 16-byte aligned (19x19: 4.8 % of the bytes), register-staged loads.
// What it buys is not its own speed but ROOM: with 640 threads x <= 64 registers and 107 KB of shared memory resident, the emit /
// NMS / gather CTAs of the previous steps fit next to it, so with several steps in flight (bench.py keeps three, each a CUDA graph
// on its own stream) the chain's latency-bound kernels run UNDER the next step's stream instead of after their own:
// 184 -> 160 us per step.  Splitting ONE step into image groups does not pay at B=64 (profiles/r2_summary.md).
// ---------------------------------------------------------------------------------------------------------------
#ifndef YL_FT_STREAM
#define YL_FT_STREAM 8
#endif
#ifndef YL_FT_SCALAR
#define YL_FT_SCALAR 12                        // a scalar warp has 8 loads in flight: it takes a dozen of them per SM to hide the 19x19 scale
#endif
#ifndef YL_FT_STAGES
#define YL_FT_STAGES 3
#endif
#ifndef YL_FT_MAXREG
#define YL_FT_MAXREG 64
#endif
constexpr int FT_STREAM = YL_FT_STREAM;        // streaming warps per CTA
constexpr int FT_SCALAR = YL_FT_SCALAR;        // scalar warps per CTA
constexpr int FT_STAGES = YL_FT_STAGES;        // ring stages per streaming warp (4 KB each)
constexpr int FT_THREADS = 32 * (FT_STREAM + FT_SCALAR);

struct alignas(128) FtStream {
    float stage[FT_STAGES][WT_KC][WT_BOX];
    float objp[2][WT_BOX];                     // objectness plane of the current / the next tile
    unsigned long long full[FT_STAGES], obj_full[2];
};
struct FtSmem {
    FtStream s[FT_STREAM];
};
static_assert(sizeof(FtSmem) <= 200 * 1024, "the flag CTA must leave shared memory for co-resident emit / NMS CTAs");

// t-th tile among the scales with layer.tma == tma (layer[l].tiles = warp tiles per (image, anchor)); np == 0: no such tile.
__device__ __forceinline__ WtTile ft_tile(const RawParams &P, int t, int nba, int tma)
{
    WtTile T;
    T.np = 0; T.src = nullptr; T.layer = 0; T.ba = 0; T.p0 = 0; T.row0 = 0; T.tma = tma;
    for (int l = 0; l < P.n_layers; ++l) {
        if (P.layer[l].tma != tma) continue;
        const int tp = P.layer[l].tiles, cnt = tp * nba;
        if (t < cnt) {
            const int bal = t / tp, tx = t - bal * tp;
            T.layer = l;
            T.ba = P.img_first * 3 + bal;
            T.p0 = tx * P.layer[l].tile_boxes;
            T.np = min(P.layer[l].tile_boxes, P.layer[l].F2 - T.p0);
            T.src = (const float *)P.layer[l].raw + ((size_t)T.ba * (5 + P.C)) * P.layer[l].F2 + T.p0;
            T.row0 = T.ba * (5 + P.C) + 5;
            return T;
        }
        t -= cnt;
    }
    return T;
}

template <int NW>
__global__ void __maxnreg__(YL_FT_MAXREG)
k_flag_tma(const __grid_constant__ RawParams P, const __grid_constant__ TmaMaps maps, int nba,
           unsigned *__restrict__ tile_counter, unsigned *__restrict__ scalar_counter)
{
    extern __shared__ __align__(128) unsigned char ft_smem_raw[];
    FtSmem &S = *reinterpret_cast<FtSmem *>(ft_smem_raw);
    const unsigned FULL = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int C = P.C;

    if (threadIdx.x == 0) {
        for (int w = 0; w < FT_STREAM; ++w) {
            for (int s = 0; s < FT_STAGES; ++s) mbar_init(&S.s[w].full[s], 1);
            mbar_init(&S.s[w].obj_full[0], 1);
            mbar_init(&S.s[w].obj_full[1], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    pdl_trigger();
    if (P.reset_words > 0) {
        // yl_post_reset folded into this kernel (nothing reads the counters before the emit kernel, which waits for this grid);
        // the two tile counters this kernel itself draws from are NOT among the words it zeroes (see the host code)
        for (int i = blockIdx.x * FT_THREADS + threadIdx.x; i < P.reset_words; i += gridDim.x * FT_THREADS) P.reset[i] = 0u;
    }

    if (warp < FT_STREAM) {
        // ---------------- streaming warp ----------------
        FtStream &W = S.s[warp];
        const int n_cc = (C + WT_KC - 1) / WT_KC;                    // class chunks per tile (>= FT_STAGES, host-checked)
        auto issue_chunk = [&](const WtTile &T, int c, int s) {
            mbar_expect_tx(&W.full[s], WT_KC * WT_BOX * 4u);         // full box, zero fill included
            tma_load_2d(&W.stage[s][0][0], &maps.m[T.layer], T.p0, T.row0 + c * WT_KC, &W.full[s]);
        };
        auto issue_obj = [&](const WtTile &T, int slot) {
            const unsigned bytes = (unsigned)T.np * 4u;
            mbar_expect_tx(&W.obj_full[slot], bytes);
            bulk_g2s(&W.objp[slot][0], T.src + 4 * (size_t)P.layer[T.layer].F2, bytes, &W.obj_full[slot]);
        };
        // the tile counter's round trip is taken one tile ahead: `ahead` is the ticket of the tile after `nxt`
        auto draw = [&]() { int t = 0; if (lane == 0) t = (int)atomicAdd(tile_counter, 1u); return t; };
        auto resolve = [&](int t) { return ft_tile(P, __shfl_sync(FULL, t, 0), nba, 1); };
        WtTile cur = resolve(draw());
        WtTile nxt = cur;
        if (cur.np != 0) nxt = resolve(draw());
        if (lane == 0 && cur.np != 0) {
            issue_obj(cur, 0);
            for (int c = 0; c < FT_STAGES; ++c) issue_chunk(cur, c, c);
        }
        int s = 0;                       // ring stage of the next chunk to consume
        unsigned ph = 0u;                // phase bit per ring stage
        unsigned it = 0u;                // tiles processed (objectness slot = it & 1, its phase = (it >> 1) & 1)
        while (cur.np != 0) {
            const int ahead = (nxt.np != 0) ? draw() : 0;
            if (lane == 0 && nxt.np != 0) issue_obj(nxt, (it + 1) & 1);
            const bool inb = lane * 4 < cur.np;
            float obj[4], lth[4];
            {
                mbar_wait(&W.obj_full[it & 1], (it >> 1) & 1u);
                const float4 to = *reinterpret_cast<const float4 *>(&W.objp[it & 1][lane * 4]);
                const float tv[4] = {to.x, to.y, to.z, to.w};
#pragma unroll
                for (int v = 0; v < 4; ++v) {
                    obj[v] = inb ? spec_sigmoidf(tv[v]) : 0.0f;
                    lth[v] = inb ? class_logit_bound(obj[v], P.thr) : kInf;
                }
            }
            const RawLayer &Ly = P.layer[cur.layer];
            const int b = cur.ba / 3, a = cur.ba - 3 * b;
            const size_t r = (size_t)b * P.M4 + (Ly.row_off + a * Ly.F2 + cur.p0 + lane * 4);
            if (inb) stg_keep4(P.objtab + r, make_uint4(__float_as_uint(obj[0]), __float_as_uint(obj[1]), __float_as_uint(obj[2]),
                                                        __float_as_uint(obj[3])));
            constexpr int CPW = 32 / WT_KC;                              // chunks per flag word
            unsigned m0 = 0u, m1 = 0u, m2 = 0u, m3 = 0u;
#pragma unroll 1
            for (int c = 0; c < n_cc; ++c) {
                mbar_wait(&W.full[s], (ph >> s) & 1u);
                const int kn = min(WT_KC, C - c * WT_KC);
                const float *sp = &W.stage[s][0][lane * 4];
                unsigned a0 = 0u, a1 = 0u, a2 = 0u, a3 = 0u;
                if (kn == WT_KC) {
                    // full chunk (every chunk when C is a multiple of WT_KC): all LDS.128 issued before the first compare
                    float4 tv[WT_KC];
#pragma unroll
                    for (int k = 0; k < WT_KC; ++k) tv[k] = *reinterpret_cast<const float4 *>(sp + k * WT_BOX);
#pragma unroll
                    for (int k = 0; k < WT_KC; ++k) {
                        flag_or(a0, tv[k].x, lth[0], 1u << k);
                        flag_or(a1, tv[k].y, lth[1], 1u << k);
                        flag_or(a2, tv[k].z, lth[2], 1u << k);
                        flag_or(a3, tv[k].w, lth[3], 1u << k);
                    }
                } else {
#pragma unroll 1
                    for (int k = 0; k < kn; ++k) {
                        const float4 tv = *reinterpret_cast<const float4 *>(sp + k * WT_BOX);
                        flag_or(a0, tv.x, lth[0], 1u << k);
                        flag_or(a1, tv.y, lth[1], 1u << k);
                        flag_or(a2, tv.z, lth[2], 1u << k);
                        flag_or(a3, tv.w, lth[3], 1u << k);
                    }
                }
                const int sh = (c % CPW) * WT_KC;
                m0 |= a0 << sh; m1 |= a1 << sh; m2 |= a2 << sh; m3 |= a3 << sh;
                __syncwarp();                                            // every lane has read the stage
                if (lane == 0) {
                    const int cn = c + FT_STAGES;                        // the chunk that takes this stage next
                    if (cn < n_cc) issue_chunk(cur, cn, s);
                    else if (nxt.np != 0) issue_chunk(nxt, cn - n_cc, s);
                }
                ph ^= 1u << s;
                s = (s + 1 == FT_STAGES) ? 0 : s + 1;
                if ((c + 1) % CPW == 0 || c + 1 == n_cc) {
                    // a dead box (objectness below the threshold) flags nothing, whatever its logits are (NaN / +inf set bits)
                    if (lth[0] == kInf) m0 = 0u;
                    if (lth[1] == kInf) m1 = 0u;
                    if (lth[2] == kInf) m2 = 0u;
                    if (lth[3] == kInf) m3 = 0u;
                    if (inb) stg_keep4(P.flags + (size_t)(c / CPW) * P.BM4 + r, make_uint4(m0, m1, m2, m3));
                    m0 = m1 = m2 = m3 = 0u;
                }
            }
            cur = nxt;
            if (nxt.np != 0) nxt = resolve(ahead);
            ++it;
        }
    } else {
        // ---------------- scalar warp: 32 boxes per tile, register-staged loads ----------------
        for (;;) {
            int t = 0;
            if (lane == 0) t = (int)atomicAdd(scalar_counter, 1u);
            const WtTile T = ft_tile(P, __shfl_sync(FULL, t, 0), nba, 0);
            if (T.np == 0) break;
            const RawLayer &Ly = P.layer[T.layer];
            float obj1[1], lth1[1];
            unsigned bits1[1][NW];
            const bool inb = lane < T.np;
            ldg_stream<float, 1, NW>(P, Ly, T.ba, T.p0 + lane, inb, obj1, lth1, bits1);
            if (inb) {
                const int b = T.ba / 3, a = T.ba - 3 * b;
                const size_t r = (size_t)b * P.M4 + (Ly.row_off + a * Ly.F2 + T.p0 + lane);
                stg_keep1(P.objtab + r, __float_as_uint(obj1[0]));
#pragma unroll
                for (int w = 0; w < NW; ++w) stg_keep1(P.flags + (size_t)w * P.BM4 + r, bits1[0][w]);
            }
        }
    }
}

// Dense front end: rows of 5+C contiguous floats (cx, cy, w, h, obj, classes): NaN-propagating row pre-filter, per-class
// test, one record per surviving pair.
constexpr int KD_THREADS = 256;
constexpr int KD_MAXJ = (5 + YL_MAX_CLASSES + 31) / 32;

// One decoded row held one element per lane and slot: e[j] = row[32 j + lane].
template <int NJ>
__device__ __forceinline__ void dense_row(const float (&e)[NJ], int nch, int C, int num_classes, float thr,
                                          int cap_seg, long r, long M, uint4 *__restrict__ cand, unsigned *__restrict__ seg_count)
{
    const int lane = threadIdx.x & 31;
    const float obj = __shfl_sync(0xFFFFFFFFu, e[0], 4);
    bool pass[NJ];
    bool any = false, anyn = false, has_nan = false;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
        const int idx = 32 * j + lane;
        pass[j] = (idx >= 5 && idx < nch) && (__fmul_rn(e[j], obj) >= thr);    // utils.py:170
        any |= pass[j];
        anyn |= pass[j] && idx < 5 + num_classes;
        has_nan |= (idx >= 5 && idx < 5 + num_classes) && (e[j] != e[j]);
    }
    if (obj > 0.0f && obj < kInf) {
        // Row pre-filter obj * max_{c < num_classes} cls >= thr (utils.py:139-148).  For a finite obj > 0, fl(obj*x) is monotone
        // in x and never NaN for a non-NaN x, so without NaNs the row passes exactly when one of its first num_classes classes
        // passes the per-class test: no max reduction for the ~99 % of rows that produce nothing.  (+-0 and +inf are not:
        // 0 * inf and inf * 0 are NaN, so the max can fail where a smaller class passes.)
        if (!__any_sync(0xFFFFFFFFu, anyn)) return;
        if (__any_sync(0xFFFFFFFFu, has_nan)) return;                 // torch.max propagates NaN: NaN >= thr is False
    } else {
        // +-0, +inf, negative or NaN objectness (not a finite sigmoid output): literal form, max with torch.max NaN propagation
        float mx = -kInf;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const int idx = 32 * j + lane;
            if (idx >= 5 && idx < 5 + num_classes) mx = fmaxf(mx, e[j]);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o));
        if (__any_sync(0xFFFFFFFFu, has_nan) || !(__fmul_rn(obj, mx) >= thr)) return;
        if (!__any_sync(0xFFFFFFFFu, any)) return;
    }
    // image / row of the few rows that get here (the 64-bit division costs more than the rest of the row test)
    int b;
    unsigned row;
    if (r < 0x7FFFFFFFL && M < 0x7FFFFFFFL) { b = (int)((unsigned)r / (unsigned)M); row = (unsigned)r - (unsigned)b * (unsigned)M; }
    else { b = (int)(r / M); row = (unsigned)(r - (long)b * M); }
    const float cx = __shfl_sync(0xFFFFFFFFu, e[0], 0), cy = __shfl_sync(0xFFFFFFFFu, e[0], 1);
    const float w = __shfl_sync(0xFFFFFFFFu, e[0], 2), h = __shfl_sync(0xFFFFFFFFu, e[0], 3);
    const float hw = __fmul_rn(w, 0.5f), hh = __fmul_rn(h, 0.5f);          // utils.py:117-126
    const uint4 corners = make_uint4(__float_as_uint(__fsub_rn(cx, hw)), __float_as_uint(__fsub_rn(cy, hh)),
                                     __float_as_uint(__fadd_rn(cx, hw)), __float_as_uint(__fadd_rn(cy, hh)));
#pragma unroll
    for (int j = 0; j < NJ; ++j)
        if (pass[j]) {
            const int k = 32 * j + lane - 5;
            const float s = __fadd_rn(__fmul_rn(obj, e[j]), 0.0f);        // nms score = obj*cls (utils.py:209)
            const unsigned seg = (unsigned)(b * C + k);
            const unsigned slot = atomicAdd(&seg_count[seg], 1u);
            if (slot < (unsigned)cap_seg) {
                uint4 *r = cand + ((size_t)seg * cap_seg + slot) * 2;
                r[0] = make_uint4(__float_as_uint(s), row, __float_as_uint(e[j]), __float_as_uint(obj));
                r[1] = corners;
            }
        }
}

// Row-per-lane form of the dense front end (16-byte aligned base).  A warp takes 32 consecutive rows -- 32 * (5+C) * 4 contiguous
// bytes, 16-byte aligned when the first row index is a multiple of four -- as ONE bulk copy into its private shared-memory buffer
// (UBLKCP, transaction mbarrier; the next batch is in flight while this one is walked), and every lane then walks ITS OWN row: the
// reference's row filter is literally `obj * max_c cls >= conf` (utils.py:139-148), i.e. one NaN-propagating max chain
// (FMNMX3.NAN, a class pitch of 5+C = 85 words is conflict-free) and one multiply-compare per row and lane, a quarter of the
// instructions of a warp-per-row walk, which spends a vote per row.  The ~8 % of rows that pass are emitted with all lanes.
constexpr int KR_ROWS = 32;

__device__ __forceinline__ float max_nan(float a, float b)
{
    float d;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
    return d;
}

template <int NJ>
__global__ void __launch_bounds__(320, 1)
k_filter_dense_rows(const float *__restrict__ pred, long M, int C, int num_classes, float thr, int cap_seg,
                    long row_first, long row_end, long rows_total, uint4 *__restrict__ cand, unsigned *__restrict__ seg_count)
{
    extern __shared__ __align__(128) unsigned char kr_smem[];
    const unsigned FULL = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const int nch = 5 + C;
    const int buf_floats = KR_ROWS * nch;                                      // a multiple of four floats
    float *buf0 = reinterpret_cast<float *>(kr_smem) + (size_t)warp * 2 * buf_floats;
    unsigned long long *bar = reinterpret_cast<unsigned long long *>(reinterpret_cast<float *>(kr_smem) + (size_t)n_warps * 2 * buf_floats) + 2 * warp;
    if (lane == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    const long g_first = row_first / KR_ROWS, g_end = (row_end + KR_ROWS - 1) / KR_ROWS;
    const long wid = (long)blockIdx.x * n_warps + warp, nw = (long)gridDim.x * n_warps;
    // batch g = rows [32 g, 32 g + 32) of the tensor; the part of it inside the tensor arrives as one bulk copy (whole 16-byte
    // units) plus at most three trailing floats by plain loads (tensor sizes that are not a multiple of four rows)
    auto issue = [&](long g, int slot) {
        const long r0 = g * KR_ROWS;
        const long n_rows = min((long)KR_ROWS, rows_total - r0);
        const unsigned bytes = (unsigned)(n_rows * nch * 4);
        const unsigned bulk = bytes & ~15u;
        float *dst = buf0 + (size_t)slot * buf_floats;
        const float *src = pred + (size_t)r0 * nch;
        if (lane == 0) {
            mbar_expect_tx(&bar[slot], bulk);                                   // bulk == 0: the arrival alone completes the phase
            if (bulk) bulk_g2s(dst, src, bulk, &bar[slot]);
        }
        const unsigned tail = (bytes - bulk) >> 2;
        if ((unsigned)lane < tail) dst[(bulk >> 2) + lane] = src[(bulk >> 2) + lane];
    };
    long g = g_first + wid;
    if (g < g_end) issue(g, 0);
    unsigned it = 0;
    while (g < g_end) {
        const long gn = g + nw;
        if (gn < g_end) issue(gn, (it + 1) & 1);                                // that buffer was walked in the previous iteration
        mbar_wait(&bar[it & 1], (it >> 1) & 1u);
        __syncwarp();                                                           // the tail floats of the plain loads
        const float *buf = buf0 + (size_t)(it & 1) * buf_floats;
        const long r0 = g * KR_ROWS;
        const long row = r0 + lane;
        const bool valid = row >= row_first && row < row_end;
        bool pass = false;
        if (valid) {
            const float *rp = buf + lane * nch;
            const float obj = rp[4];
            float m0 = -kInf, m1 = -kInf, m2 = -kInf, m3 = -kInf;                // four chains: the max is associative
            int k = 0;
            for (; k + 4 <= num_classes; k += 4) {
                m0 = max_nan(m0, rp[5 + k]); m1 = max_nan(m1, rp[6 + k]);
                m2 = max_nan(m2, rp[7 + k]); m3 = max_nan(m3, rp[8 + k]);
            }
            for (; k < num_classes; ++k) m0 = max_nan(m0, rp[5 + k]);
            const float m = max_nan(max_nan(m0, m1), max_nan(m2, m3));           // torch.max: NaN propagates (utils.py:139-141)
            pass = __fmul_rn(obj, m) >= thr;                                     // :145  (NaN >= thr is False)
        }
        unsigned mask = __ballot_sync(FULL, pass);
        while (mask) {
            // The rows that passed the row filter (no NaN among their first num_classes classes, obj * max >= conf), four at a
            // time so that the slot atomics of four rows are in flight together: one record per class column with
            // obj * cls >= conf (utils.py:170 looks at every column >= 5), all lanes, lane = column mod 32.
            int rrs[4];
            int nq = 0;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                rrs[q] = 0;
                if (mask) { rrs[q] = __ffs(mask) - 1; mask &= mask - 1u; nq = q + 1; }
            }
            float e[4][NJ], obj[4];
            unsigned slot[4][NJ], segb[4], rowi[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float *rp = buf + rrs[q] * nch;
                obj[q] = rp[4];
                const long r = r0 + rrs[q];
                const unsigned b = (unsigned)(r / M);
                rowi[q] = (unsigned)(r - (long)b * M);
                segb[q] = b * (unsigned)C;
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    const int idx = 32 * j + lane;
                    e[q][j] = (q < nq && idx >= 5 && idx < nch) ? rp[idx] : __int_as_float(0x7FC00000);   // NaN never passes
                    slot[q][j] = 0xFFFFFFFFu;
                    if (__fmul_rn(e[q][j], obj[q]) >= thr) slot[q][j] = atomicAdd(&seg_count[segb[q] + (unsigned)(idx - 5)], 1u);
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (q >= nq) break;
                const float *rp = buf + rrs[q] * nch;
                const float cx = rp[0], cy = rp[1], hw = __fmul_rn(rp[2], 0.5f), hh = __fmul_rn(rp[3], 0.5f);   // utils.py:117-126
                const uint4 corners = make_uint4(__float_as_uint(__fsub_rn(cx, hw)), __float_as_uint(__fsub_rn(cy, hh)),
                                                 __float_as_uint(__fadd_rn(cx, hw)), __float_as_uint(__fadd_rn(cy, hh)));
#pragma unroll
                for (int j = 0; j < NJ; ++j)
                    if (slot[q][j] < (unsigned)cap_seg) {
                        const int k = 32 * j + lane - 5;
                        const float sc = __fadd_rn(__fmul_rn(obj[q], e[q][j]), 0.0f);       // nms score = obj*cls (utils.py:209)
                        uint4 *rec = cand + ((size_t)(segb[q] + (unsigned)k) * cap_seg + slot[q][j]) * 2;
                        rec[0] = make_uint4(__float_as_uint(sc), rowi[q], __float_as_uint(e[q][j]), __float_as_uint(obj[q]));
                        rec[1] = corners;
                    }
            }
        }
        __syncwarp();                                                           // every lane has read the buffer
        g = gn;
        ++it;
    }
}

// Fallback for a tensor whose base is not 16-byte aligned: one warp per row, scalar loads.
__global__ void __launch_bounds__(KD_THREADS)
k_filter_dense_unaligned(const float *__restrict__ pred, long M, int C, int num_classes, float thr, int cap_seg,
                         long row_first, long row_end, uint4 *__restrict__ cand, unsigned *__restrict__ seg_count)
{
    const int lane = threadIdx.x & 31;
    const long wid = ((long)blockIdx.x * KD_THREADS + threadIdx.x) >> 5;
    const long nwarps = ((long)gridDim.x * KD_THREADS) >> 5;
    const int nch = 5 + C;
    const int nj = (nch + 31) >> 5;
    for (long r = row_first + wid; r < row_end; r += nwarps) {
        const float *p = pred + (size_t)r * nch;
        float e[KD_MAXJ];
#pragma unroll
        for (int j = 0; j < KD_MAXJ; ++j) {
            const int idx = 32 * j + lane;
            e[j] = (j < nj && idx < nch) ? ldg_stream1(p + idx) : 0.0f;
        }
        dense_row<KD_MAXJ>(e, nch, C, num_classes, thr, cap_seg, r, M, cand, seg_count);
    }
}

}  // namespace yl

using namespace yl;

typedef CUresult (*PFN_encodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                    const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// YL_FLAG selects the streaming flag kernel: "tma" (default; k_flag_tma: one persistent CTA per SM, TMA rings in shared
// memory, 40 % of the register file and 107 KB of shared memory -- the form that lets the emit / NMS / gather CTAs of the PREVIOUS
// steps run next to it when several steps are in flight) or "ldg" (k_flag_raw: register-staged loads, a few per cent faster alone
// -- 81 us against 86 -- but it fills the register file, so nothing overlaps it).
static const bool g_flag_tma = getenv("YL_FLAG") ? strcmp(getenv("YL_FLAG"), "tma") == 0 : true;
// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda).
static int encode_plane_map(CUtensorMap *map, const float *raw, int F2, long rows, int box_rows = WT_KC)
{
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p) return YL_ERR_CUDA_BASE + (int)cudaErrorNotSupported;
        fn = (PFN_encodeTiled)p;
    }
    const cuuint64_t gdim[2] = {(cuuint64_t)F2, (cuuint64_t)rows};
    const cuuint64_t gstr[1] = {(cuuint64_t)F2 * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)WT_BOX, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void *)raw, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? YL_OK : YL_ERR_CUDA_BASE + (int)cudaErrorInvalidValue;
}

static int g_num_sms()
{
    static int n = 0;
    if (!n) { int dev = 0; cudaGetDevice(&dev); if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148; }
    return n;
}

extern "C" size_t yl_post_workspace_bytes(int B, long M, int C, int cap_seg)
{
    if (B <= 0 || M <= 0 || C <= 0 || cap_seg <= 0) return 0;
    return post_layout(B, M, C, cap_seg).total;
}

extern "C" int yl_post_reset(void *ws, size_t ws_bytes, int B, long M, int C, int cap_seg, yl_stream_t stream)
{
    if (!ws || B <= 0 || M <= 0 || C <= 0 || cap_seg <= 0) return YL_ERR_ARG;
    const PostLayout L = post_layout(B, M, C, cap_seg);
    if (ws_bytes < L.total) return YL_ERR_WORKSPACE;
    YL_CUDA_TRY(cudaMemsetAsync(ws, 0, L.counters_bytes, (cudaStream_t)stream));
    return YL_OK;
}

// gridDim.y (image, anchor) of k_flag_raw / k_emit_flagged is at most 65535.
constexpr int kSliceImages = 65535 / 3;

// The register-staged flag kernel (unless the caller has already streamed the scales with k_flag_tma) and the emit kernel for
// element type T over images [P.img_first, P.img_first + img_count), tiles CTAs along x.  A batch of more than kSliceImages
// images goes out in slices of that many, one launch per kernel and slice, each told its first image; up to that size each
// kernel is one launch with the same grid.  Only the first flag slice zeroes the counters (P.reset_words), and every emit
// slice follows the last flag slice on the stream.  pdl: the first emit launch may overlap its predecessor's tail, which is
// allowed only when that predecessor is the flag launch whose tables it reads (so not after a sliced flag pass).
// sxy: the per-scale scale_x_y of the emit kernel, or nullptr for the unscaled decode.
template <typename T>
static int launch_flag_emit(const RawParams &P, const ScaleXY *sxy, int tiles, int img_count, bool flag, bool emit, bool pdl, int NW,
                            cudaStream_t st)
{
    for (int i0 = 0; flag && i0 < img_count; i0 += kSliceImages) {
        RawParams Q = P;
        Q.img_first += i0;
        if (i0 > 0) Q.reset_words = 0;
        const dim3 grid(tiles, 3 * min(kSliceImages, img_count - i0));
        switch (NW) {
        case 1: k_flag_raw<T, 1><<<grid, K1_THREADS, 0, st>>>(Q); break;
        case 2: k_flag_raw<T, 2><<<grid, K1_THREADS, 0, st>>>(Q); break;
        case 3: k_flag_raw<T, 3><<<grid, K1_THREADS, 0, st>>>(Q); break;
        default: k_flag_raw<T, 4><<<grid, K1_THREADS, 0, st>>>(Q); break;
        }
        YL_LAUNCH_CHECK();
    }
    if (flag && img_count > kSliceImages) pdl = false;
    for (int i0 = 0; emit && i0 < img_count; i0 += kSliceImages) {
        RawParams Q = P;
        Q.img_first += i0;
        const dim3 grid(tiles, 3 * min(kSliceImages, img_count - i0));
        const bool pdl_i = pdl && i0 == 0;
        cudaError_t le;
        void (*plain)(RawParams);
        void (*scaled)(RawParams, ScaleXY);
#define YL_EMIT_CASE(NW_)                                                                                                    \
        plain = k_emit_flagged<T, NW_>;                                                                                      \
        scaled = k_emit_flagged<T, NW_>;                                                                                     \
        le = sxy ? launch_after(scaled, grid, dim3(K1_THREADS), 0, st, pdl_i, Q, *sxy)                                       \
                 : launch_after(plain, grid, dim3(K1_THREADS), 0, st, pdl_i, Q);
        switch (NW) {
        case 1: YL_EMIT_CASE(1) break;
        case 2: YL_EMIT_CASE(2) break;
        case 3: YL_EMIT_CASE(3) break;
        default: YL_EMIT_CASE(4) break;
        }
#undef YL_EMIT_CASE
        if (le != cudaSuccess) return YL_ERR_CUDA_BASE + (int)le;
    }
    return YL_OK;
}

static int filter_raw_impl(const void *const *raw, int dtype, const int *F, int n_layers, int B, int C,
                           const float *anchors_px, const int *anchor_mask, float conf_thre, const float *scale_x_y,
                           void *ws, size_t ws_bytes, long M, int cap_seg, int img_first, int img_count,
                           yl_stream_t stream, int stages)
{
    if (dtype != YL_DTYPE_F32 && dtype != YL_DTYPE_F16 && dtype != YL_DTYPE_BF16) return YL_ERR_ARG;
    if (!raw || !F || !anchors_px || !anchor_mask || !ws) return YL_ERR_ARG;
    if (n_layers < 1 || n_layers > 3 || B <= 0 || C <= 0 || cap_seg <= 0) return YL_ERR_ARG;
    // scale_x_y: NULL or every scale exactly 1 is the unscaled emit kernel (the same launches and bytes as without it)
    ScaleXY sxy;
    bool scaled = false;
    for (int l = 0; l < 3; ++l) {
        const float s = (scale_x_y && l < n_layers) ? scale_x_y[l] : 1.0f;
        if (!scale_xy_valid(s)) return YL_ERR_ARG;
        sxy.s[l] = s;
        sxy.beta[l] = scale_xy_beta(s);
        scaled |= s != 1.0f;
    }
    if (img_first < 0 || img_count < 0 || img_first + img_count > B) return YL_ERR_ARG;
    if (C > YL_MAX_CLASSES) return YL_ERR_CLASSES;
    long m_sum = 0;
    for (int l = 0; l < n_layers; ++l) { if (F[l] <= 0 || !raw[l]) return YL_ERR_ARG; m_sum += 3L * F[l] * F[l]; }
    if (m_sum != M) return YL_ERR_ARG;
    const PostLayout L = post_layout(B, M, C, cap_seg);
    if (ws_bytes < L.total) return YL_ERR_WORKSPACE;
    if (img_count == 0) return YL_OK;
    const int NW = (C + 31) / 32;
    if (NW < 1 || NW > 4) return YL_ERR_CLASSES;
    char *w = (char *)ws;
    cudaStream_t st = (cudaStream_t)stream;
    RawParams base;
    base.C = C; base.cap_seg = cap_seg; base.img_first = img_first; base.M = M; base.thr = conf_thre;
    base.sparse = conf_thre >= 0.02f ? 1 : 0;     // sigmoid(obj) >= 0.02 is rare for background cells (obj logit >= -3.9)
    base.cand = (uint4 *)(w + L.off_cand); base.seg_count = (unsigned *)(w + L.off_seg_count);
    base.objtab = (float *)(w + L.off_obj); base.n_layers = 0;
    base.flags = (unsigned *)(w + L.off_flags); base.M4 = L.M4; base.BM4 = (long)B * L.M4;
    base.reset = (unsigned *)w; base.reset_words = 0;

    // ---- the scales as the kernels see them ----
    RawLayer lay[3];
    int row_off = 0, n_tma = 0;
    const int n_cc = (C + WT_KC - 1) / WT_KC;
    // the TMA flag kernel streams every plane of every box; with a high threshold the register-staged kernel's objectness-first
    // mode skips most class planes instead.  It has an fp32 form only.
    const bool f32 = dtype == YL_DTYPE_F32;
    const bool flag_tma = g_flag_tma && !base.sparse && f32;
    for (int l = 0; l < n_layers; ++l) {
        RawLayer &Ly = lay[l];
        Ly.raw = raw[l]; Ly.Fw = F[l]; Ly.F2 = F[l] * F[l]; Ly.row_off = row_off;
        Ly.stride = (float)(8 << l);                                        // yololayer.py:54
        for (int a = 0; a < 3; ++a) {                                       // yololayer.py:73-76 (doubles, then fp32)
            const int q = anchor_mask[3 * l + a];
            if (q < 0 || q > 8) return YL_ERR_ARG;
            Ly.aw[a] = (float)((double)anchors_px[2 * q] / (double)Ly.stride);
            Ly.ah[a] = (float)((double)anchors_px[2 * q + 1] / (double)Ly.stride);
        }
        // 128-bit loads / bulk copies need 16-byte aligned planes: F^2 % 4 == 0 and an aligned base (19x19, 13x13 fall back).
        // 16-bit planes are read with 64-bit loads where F^2 % 4 == 0 and the base is 8-byte aligned.  Either way the flag and
        // objectness tables of a vector scale are stored and loaded as uint4 / float4 at row b*M4 + row_off + a*F^2 + p, so the
        // scale's rows must start 16-byte aligned as well: a lower scale with an odd grid (e.g. 75x75 below 38x38) makes row_off
        // odd, and the scale then takes the scalar path.
        if (f32) Ly.vec = ((Ly.F2 % 4 == 0) && (((uintptr_t)raw[l]) % 16 == 0) && row_off % 4 == 0) ? 4 : 1;
        else Ly.vec = ((Ly.F2 % 4 == 0) && (((uintptr_t)raw[l]) % 8 == 0) && row_off % 4 == 0) ? 4 : 1;
        Ly.tma = (Ly.vec == 4 && n_cc >= FT_STAGES) ? 1 : 0;              // k_flag_tma's ring needs FT_STAGES class chunks
        Ly.tile_boxes = 0; Ly.tiles = 0;
        n_tma += Ly.tma;
        row_off += 3 * Ly.F2;
    }
    // Pt: k_flag_tma (warp tiles of 128 boxes, 32 for the scalar scales; TMA scales first).  Pl: k_flag_raw / k_emit_flagged
    // (CTA tiles of K1_THREADS * vec boxes).
    const bool persistent = flag_tma && n_tma > 0;
    RawParams Pt = base, Pl = base;
    if (persistent)
        for (int tma = 1; tma >= 0; --tma)
            for (int l = 0; l < n_layers; ++l) {
                if (lay[l].tma != tma) continue;
                RawLayer Ly = lay[l];
                Ly.tile_boxes = tma ? WT_BOX : 32;
                Ly.tiles = (Ly.F2 + Ly.tile_boxes - 1) / Ly.tile_boxes;
                Pt.layer[Pt.n_layers++] = Ly;
            }
    int tiles_ldg = 0;
    for (int l = 0; l < n_layers; ++l) {
        RawLayer Ly = lay[l];
        Ly.tma = 0;
        Ly.tile_boxes = K1_THREADS * Ly.vec;
        Ly.tiles = (Ly.F2 / Ly.vec + K1_THREADS - 1) / K1_THREADS;
        tiles_ldg += Ly.tiles;
        Pl.layer[Pl.n_layers++] = Ly;
    }
    for (int l = Pt.n_layers; l < 3; ++l) { Pt.layer[l] = lay[0]; Pt.layer[l].tiles = 0; Pt.layer[l].tma = -1; }
    for (int l = Pl.n_layers; l < 3; ++l) { Pl.layer[l] = lay[0]; Pl.layer[l].tiles = 0; }

    // ---- counters (stages bit 2: the caller skipped yl_post_reset) ----
    if (stages & 4) {
        if ((stages & 1) && persistent) {
            // the TMA flag kernel zeroes the segment counters itself, but not the two tile counters it draws from
            Pt.reset_words = (int)(L.off_tile_count / sizeof(unsigned));
            YL_CUDA_TRY(cudaMemsetAsync(w + L.off_tile_count, 0, L.counters_bytes - L.off_tile_count, st));
        } else if (stages & 1) {
            Pl.reset_words = (int)(L.counters_bytes / sizeof(unsigned));   // k_flag_raw zeroes the counters (no memset node)
        } else {
            YL_CUDA_TRY(cudaMemsetAsync(ws, 0, L.counters_bytes, st));
        }
    }

    // ---- streaming flag kernel ----
    if ((stages & 1) && persistent) {
        const int nba = img_count * 3;
        unsigned *tile_counter = (unsigned *)(w + L.off_tile_count) + img_first;
        unsigned *scalar_counter = (unsigned *)(w + L.off_tile_count) + B + img_first;
        TmaMaps maps;
        memset(&maps, 0, sizeof(maps));
        int n_tma_tiles = 0;
        for (int l = 0; l < Pt.n_layers; ++l) {
            if (Pt.layer[l].tma != 1) continue;
            n_tma_tiles += Pt.layer[l].tiles * nba;
            const int rc = encode_plane_map(&maps.m[l], (const float *)Pt.layer[l].raw, Pt.layer[l].F2, (long)B * 3 * (5 + C));
            if (rc != YL_OK) return rc;
        }
        const size_t smem = sizeof(FtSmem);
        const int want = (n_tma_tiles + FT_STREAM - 1) / FT_STREAM;
        const int ft_grid = want < g_num_sms() ? (want > 0 ? want : 1) : g_num_sms();
#define YL_FT_CASE(NW_)                                                                                              \
    case NW_: {                                                                                                      \
        static bool attr_done = false;                                                                               \
        if (!attr_done) {                                                                                            \
            YL_CUDA_TRY(cudaFuncSetAttribute(k_flag_tma<NW_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
            attr_done = true;                                                                                        \
        }                                                                                                            \
        k_flag_tma<NW_><<<ft_grid, FT_THREADS, smem, st>>>(Pt, maps, nba, tile_counter, scalar_counter);              \
    } break;
        switch (NW) { YL_FT_CASE(1) YL_FT_CASE(2) YL_FT_CASE(3) YL_FT_CASE(4) }
#undef YL_FT_CASE
        YL_LAUNCH_CHECK();
    }

    // ---- register-staged flag kernel and emit kernel ----
    const bool flag_ldg = (stages & 1) && !persistent;
    const bool pdl = pdl_enabled() && (stages & 1);                         // the emit kernel directly follows the flag kernel
    switch (dtype) {
    case YL_DTYPE_F16: return launch_flag_emit<__half>(Pl, scaled ? &sxy : nullptr, tiles_ldg, img_count, flag_ldg, stages & 2, pdl, NW, st);
    case YL_DTYPE_BF16:
        return launch_flag_emit<__nv_bfloat16>(Pl, scaled ? &sxy : nullptr, tiles_ldg, img_count, flag_ldg, stages & 2, pdl, NW, st);
    default: return launch_flag_emit<float>(Pl, scaled ? &sxy : nullptr, tiles_ldg, img_count, flag_ldg, stages & 2, pdl, NW, st);
    }
}

extern "C" int yl_filter_raw_ex(const void *const *raw, int dtype, const int *F, int n_layers, int B, int C,
                                const float *anchors_px, const int *anchor_mask, float conf_thre, const float *scale_x_y,
                                void *ws, size_t ws_bytes, long M, int cap_seg, int img_first, int img_count,
                                int stages, yl_stream_t stream)
{
    if (stages < 1 || stages > 7 || (stages & 3) == 0) return YL_ERR_ARG;
    return filter_raw_impl(raw, dtype, F, n_layers, B, C, anchors_px, anchor_mask, conf_thre, scale_x_y, ws, ws_bytes, M, cap_seg,
                           img_first, img_count, stream, stages);
}

extern "C" int yl_filter_raw_typed(const void *const *raw, int dtype, const int *F, int n_layers, int B, int C,
                                   const float *anchors_px, const int *anchor_mask, float conf_thre,
                                   void *ws, size_t ws_bytes, long M, int cap_seg, int img_first, int img_count,
                                   int stages, yl_stream_t stream)
{
    return yl_filter_raw_ex(raw, dtype, F, n_layers, B, C, anchors_px, anchor_mask, conf_thre, nullptr, ws, ws_bytes, M, cap_seg,
                            img_first, img_count, stages, stream);
}

extern "C" int yl_filter_raw(const float *const *raw, const int *F, int n_layers, int B, int C,
                             const float *anchors_px, const int *anchor_mask, float conf_thre,
                             void *ws, size_t ws_bytes, long M, int cap_seg, int img_first, int img_count,
                             yl_stream_t stream)
{
    return yl_filter_raw_typed((const void *const *)raw, YL_DTYPE_F32, F, n_layers, B, C, anchors_px, anchor_mask, conf_thre, ws,
                               ws_bytes, M, cap_seg, img_first, img_count, 3, stream);
}

extern "C" int yl_filter_raw_stage(const float *const *raw, const int *F, int n_layers, int B, int C,
                                   const float *anchors_px, const int *anchor_mask, float conf_thre,
                                   void *ws, size_t ws_bytes, long M, int cap_seg, int img_first, int img_count,
                                   int stages, yl_stream_t stream)
{
    return yl_filter_raw_typed((const void *const *)raw, YL_DTYPE_F32, F, n_layers, B, C, anchors_px, anchor_mask, conf_thre, ws,
                               ws_bytes, M, cap_seg, img_first, img_count, stages, stream);
}

extern "C" int yl_filter_dense(const float *pred, int B, long M, int C, int num_classes, float conf_thre,
                               void *ws, size_t ws_bytes, int cap_seg, int img_first, int img_count, yl_stream_t stream)
{
    if (!pred || !ws || B <= 0 || M <= 0 || C <= 0 || cap_seg <= 0) return YL_ERR_ARG;
    if (num_classes < 1 || num_classes > C) return YL_ERR_ARG;
    if (img_first < 0 || img_count < 0 || img_first + img_count > B) return YL_ERR_ARG;
    if (C > YL_MAX_CLASSES) return YL_ERR_CLASSES;
    const PostLayout L = post_layout(B, M, C, cap_seg);
    if (ws_bytes < L.total) return YL_ERR_WORKSPACE;
    if (img_count == 0) return YL_OK;
    char *w = (char *)ws;
    const long row_first = (long)img_first * M, row_end = (long)(img_first + img_count) * M, rows_total = (long)B * M;
    uint4 *cand = (uint4 *)(w + L.off_cand);
    unsigned *seg_count = (unsigned *)(w + L.off_seg_count);
    if (((uintptr_t)pred) % 16 == 0) {
        // row-per-lane form: 2 x 32 rows of shared memory per warp, as many warps per CTA as fit 226 KB (at most 8), one CTA per SM
        static_assert(2 * KR_ROWS * (5 + YL_MAX_CLASSES) * sizeof(float) <= 226 * 1024 - 256,
                      "the two row buffers of one warp must fit the shared-memory budget at YL_MAX_CLASSES");
        const size_t per_warp = (size_t)2 * KR_ROWS * (5 + C) * sizeof(float);
        int warps = (int)((226 * 1024 - 256) / per_warp);
        warps = warps > 8 ? 8 : warps;
        const size_t smem = per_warp * warps + 16 * (size_t)warps;
        const long batches = (row_end + KR_ROWS - 1) / KR_ROWS - row_first / KR_ROWS;
        const long ctas = (batches + warps - 1) / warps;
        const int grid = (int)(ctas < g_num_sms() ? (ctas > 0 ? ctas : 1) : g_num_sms());
        cudaStream_t st = (cudaStream_t)stream;
        switch ((5 + C + 31) / 32) {
#define YL_KR_CASE(NJ_)                                                                                               \
    case NJ_: {                                                                                                       \
        static size_t attr_smem = 0;                                                                                  \
        if (smem > attr_smem) {                                                                                       \
            YL_CUDA_TRY(cudaFuncSetAttribute(k_filter_dense_rows<NJ_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
            attr_smem = smem;                                                                                         \
        }                                                                                                             \
        k_filter_dense_rows<NJ_><<<grid, 32 * warps, smem, st>>>(pred, M, C, num_classes, conf_thre, cap_seg, row_first, row_end, \
                                                                 rows_total, cand, seg_count);                        \
    } break;
            YL_KR_CASE(1) YL_KR_CASE(2) YL_KR_CASE(3) YL_KR_CASE(4)
        default: YL_KR_CASE(KD_MAXJ)
#undef YL_KR_CASE
        }
    } else {
        const long blocks_needed = ((row_end - row_first) * 32 + KD_THREADS - 1) / KD_THREADS;
        const int grid = (int)(blocks_needed < 148L * 64 ? blocks_needed : 148L * 64);
        k_filter_dense_unaligned<<<grid, KD_THREADS, 0, (cudaStream_t)stream>>>(pred, M, C, num_classes, conf_thre, cap_seg, row_first,
                                                                               row_end, cand, seg_count);
    }
    YL_LAUNCH_CHECK();
    return YL_OK;
}

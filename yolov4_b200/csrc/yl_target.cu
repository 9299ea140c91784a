// yl_target.cu -- YOLOLoss.build_target (yolo/model/yololoss.py:118-371) and the bboxes_iou it calls (:16-91).
//
//   k_target_objmask   per cell: obj_mask = !(max_n IoU(pred, GT_n) > ignore_thresh)          (:276-294)
//   k_target_scatter   per image: GT <-> 9-anchor IoU argmax (:249-265) and the assignment of
//                      obj_mask / tgt_mask / tgt_scale / target at the matched cells (:304-369),
//                      resolving same-cell collisions the way the reference's sequential loop does:
//                      scalar fields last-writer-wins, class one-hots accumulate (SURVEY.md 7-9).  A class id writes
//                      channel 5 + cls with Python's negative-index wrap (class_channel): a negative id lands on another
//                      class or on the box targets 0..3 / objectness 4.
// The dense zero background of target / tgt_mask / tgt_scale (:156-167, 99.9 % of the 16 MB/image this path writes) is
// stored by k_target_objmask itself, 128 bits at a time, before it computes its cells' IoUs: the pass runs at the pace
// of the HBM writes and the IoU arithmetic hides underneath instead of following three memsets.
#include "yl_target.cuh"
#include "../../include/yolo_head.h"

namespace yl {

// The CTA zeroes n floats at p (4-byte aligned): scalar head up to a 16-byte boundary, float4 body, scalar tail.
__device__ __forceinline__ void cta_zero(float *p, int n)
{
    int head = (int)(((16u - (unsigned)((uintptr_t)p & 15u)) & 15u) >> 2);
    if (head > n) head = n;
    if ((int)threadIdx.x < head) p[threadIdx.x] = 0.0f;
    float4 *p4 = reinterpret_cast<float4 *>(p + head);
    const int n4 = (n - head) >> 2;
#pragma unroll 4
    for (int i = threadIdx.x; i < n4; i += TG_THREADS) p4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    const int tail = head + 4 * n4 + (int)threadIdx.x;
    if (tail < n) p[tail] = 0.0f;
}

// One scale of the head as the kernels see it; up to three scales share one launch (yl_build_target3), so the latency-bound
// small grids (38x38: 17 CTAs per image, 19x19: 5) fill the machine next to the 76x76 one instead of following it.
struct TargetLayer {
    const float *pred;                 // [B,3,F,F,4] with element strides s0..s4
    long s0, s1, s2, s3, s4;
    int F, blocks;                     // blocks: CTAs along x of this scale
    float stride;
    AnchorSet an;
    float *target, *obj_mask, *tgt_mask, *tgt_scale;
};
struct TargetParams {
    TargetLayer layer[3];
    int n_layers, K, C;
    const float *labels;
    float ignore_thre;
    int *status;
};

__global__ void __launch_bounds__(TG_THREADS)
k_target_objmask(const __grid_constant__ TargetParams P)
{
    __shared__ __align__(16) float tb[TG_MAXK][4];
    __shared__ __align__(16) float tc[TG_MAXK][4];       // GT corners (x1, y1, x2, y2) for the overlap pre-test
    __shared__ float tcls[TG_MAXK];
    __shared__ float tarea[TG_MAXK];
    __shared__ unsigned char tns[TG_MAXK];
    __shared__ float tkey[TG_MAXK];
    __shared__ int sh_n, sh_ns;
    int l = 0, blk = blockIdx.x;
    while (l < P.n_layers - 1 && blk >= P.layer[l].blocks) { blk -= P.layer[l].blocks; ++l; }
    const TargetLayer &Ly = P.layer[l];
    const int F = Ly.F, C = P.C;
    const int b = blockIdx.y;
    const int cells = 3 * F * F;
    pdl_trigger();                                                    // k_target_scatter may load / match its labels meanwhile
    {
        // zero background of this CTA's cells (contiguous runs in all three tensors); k_target_scatter follows in stream order
        const int c0 = blk * TG_THREADS;
        const int nc = min(TG_THREADS, cells - c0);
        const size_t g0 = (size_t)b * cells + c0;
        cta_zero(Ly.target + g0 * (5 + C), nc * (5 + C));
        cta_zero(Ly.tgt_mask + g0 * (4 + C), nc * (4 + C));
        cta_zero(Ly.tgt_scale + g0 * 2, nc * 2);
    }
    const int n = load_truth(P.labels, b, P.K, Ly.stride, tb, tcls, &sh_n);
    const int cell = blk * TG_THREADS + threadIdx.x;
    if (n == 0) {                                                     // :225-227 obj_mask stays 1
        if (cell < cells) Ly.obj_mask[(size_t)b * cells + cell] = 1.0f;
        return;
    }
    prep_truth(n, tb, tc, tarea, tns, tkey, &sh_ns);
    if (cell >= cells) return;
    const int a = cell / (F * F);
    const int r = cell - a * F * F;
    const int j = r / F, i = r - j * F;
    const float *pp = Ly.pred + (size_t)b * Ly.s0 + (size_t)a * Ly.s1 + (size_t)j * Ly.s2 + (size_t)i * Ly.s3;
    const float ax = pp[0], ay = pp[Ly.s4], aw = pp[2 * Ly.s4], ah = pp[3 * Ly.s4];
    const bool best_above = iou_max_above(ax, ay, aw, ah, n, tb, tc, tarea, tns, sh_ns, P.ignore_thre);
    Ly.obj_mask[(size_t)b * cells + cell] = best_above ? 0.0f : 1.0f;          // :286-294
}


constexpr int TS_SLICES = 4;

__global__ void __launch_bounds__(TG_THREADS)
k_target_scatter(const __grid_constant__ TargetParams P)
{
    __shared__ float tb[TG_MAXK][4];
    __shared__ float tcls[TG_MAXK];
    __shared__ int tcell[TG_MAXK];       // matched cell index within the image, or -1
    __shared__ int tanc[TG_MAXK];        // anchor slot a = best_n % 3
    __shared__ int sh_n;
    // grid (B, TS_SLICES, scales): every CTA matches all GTs of its image (the collision test needs them), slice y writes the
    // cells of GTs t = y*8 + warp, + 8*TS_SLICES, ... so that an image's ~50 assignments are not one CTA's serial chain
    const TargetLayer &Ly = P.layer[blockIdx.z];
    const AnchorSet &an = Ly.an;
    const int F = Ly.F, C = P.C;
    float *target = Ly.target, *obj_mask = Ly.obj_mask, *tgt_mask = Ly.tgt_mask, *tgt_scale = Ly.tgt_scale;
    int *status = P.status;
    const int b = blockIdx.x;
    const int n = load_truth(P.labels, b, P.K, Ly.stride, tb, tcls, &sh_n);
    if (n == 0) return;
    const int nch = 5 + C;
    const int cells = 3 * F * F;
    for (int t = threadIdx.x; t < n; t += TG_THREADS) {
        int anc;
        const int cell = match_truth(tb[t], F, an, &anc, blockIdx.y == 0 ? status : nullptr);
        tcell[t] = cell;
        tanc[t] = anc;
    }
    __syncthreads();
    pdl_wait();                                                       // zero background and ignore mask of k_target_objmask
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int t = (int)blockIdx.y * (TG_THREADS / 32) + warp; t < n; t += (TG_THREADS / 32) * (int)gridDim.y) {
        const int cell = tcell[t];
        if (cell < 0) continue;
        const size_t gc = (size_t)b * cells + cell;
        bool overridden = false;                                       // a later matched GT lands on the same cell
        for (int u = t + 1 + lane; u < n; u += 32) overridden |= (tcell[u] == cell);
        overridden = __any_sync(0xFFFFFFFFu, overridden);
        for (int k = lane; k < 4 + C; k += 32) tgt_mask[gc * (4 + C) + k] = 1.0f;             // :333
        if (lane == 0) {
            obj_mask[gc] = 1.0f;                                                              // :330
            float *tg = target + gc * nch;
            if (!overridden) {
                const float tw = tb[t][2], th = tb[t][3];
                const float sc = __fsqrt_rn(__fsub_rn(2.0f, __fdiv_rn(__fdiv_rn(__fmul_rn(tw, th), (float)F), (float)F)));   // :337
                tgt_scale[gc * 2] = sc; tgt_scale[gc * 2 + 1] = sc;
                tg[0] = __fsub_rn(tb[t][0], (float)(short)(int)tb[t][0]);                     // :346
                tg[1] = __fsub_rn(tb[t][1], (float)(short)(int)tb[t][1]);                     // :349
                const int a = tanc[t];
                tg[2] = spec_logf(__fadd_rn(__fdiv_rn(tw, an.w[an.mask[a]]), 1e-16f));        // :362
                tg[3] = spec_logf(__fadd_rn(__fdiv_rn(th, an.h[an.mask[a]]), 1e-16f));        // :365
            }
            tg[4] = 1.0f;                                                                     // :367
            const int kc = class_channel(tcls[t], nch);                                       // :369
            // An overridden GT's write to channels 0..4 is a no-op or overwritten by the cell's last GT in the reference's
            // order; skipping it keeps it from racing with that GT's writes (another warp, possibly another CTA).
            if (kc < 0 || kc >= nch) { if (status) atomicExch(status, 1); }
            else if (!overridden || kc >= 5) tg[kc] = 1.0f;
        }
    }
}

static int fill_target_layer(TargetLayer &Ly, const float *pred, const long *ps, int F, int layer_no, const float *anchors_px,
                             const int *anchor_mask3, float *target, float *obj_mask, float *tgt_mask, float *tgt_scale)
{
    if (!pred || !ps || !anchors_px || !anchor_mask3 || !target || !obj_mask || !tgt_mask || !tgt_scale) return YL_ERR_ARG;
    if (F <= 0 || layer_no < 0 || layer_no > 2) return YL_ERR_ARG;
    Ly.pred = pred; Ly.s0 = ps[0]; Ly.s1 = ps[1]; Ly.s2 = ps[2]; Ly.s3 = ps[3]; Ly.s4 = ps[4];
    Ly.F = F; Ly.blocks = (3 * F * F + TG_THREADS - 1) / TG_THREADS;
    Ly.stride = (float)(8 << layer_no);                                                       // yololoss.py:99,136
    for (int q = 0; q < 9; ++q) {                                                             // :139-150
        Ly.an.w[q] = (float)((double)anchors_px[2 * q] / (double)Ly.stride);
        Ly.an.h[q] = (float)((double)anchors_px[2 * q + 1] / (double)Ly.stride);
    }
    for (int a = 0; a < 3; ++a) {
        if (anchor_mask3[a] < 0 || anchor_mask3[a] > 8) return YL_ERR_ARG;
        Ly.an.mask[a] = anchor_mask3[a];
    }
    Ly.target = target; Ly.obj_mask = obj_mask; Ly.tgt_mask = tgt_mask; Ly.tgt_scale = tgt_scale;
    return YL_OK;
}

static int launch_targets(TargetParams &P, int B, cudaStream_t st)
{
    if (P.status) YL_CUDA_TRY(cudaMemsetAsync(P.status, 0, sizeof(int), st));
    int blocks = 0;
    for (int l = 0; l < P.n_layers; ++l) blocks += P.layer[l].blocks;
    for (int l = P.n_layers; l < 3; ++l) { P.layer[l] = P.layer[0]; P.layer[l].blocks = 0; }
    k_target_objmask<<<dim3(blocks, B), TG_THREADS, 0, st>>>(P);
    YL_LAUNCH_CHECK();
    YL_CUDA_TRY(launch_after(k_target_scatter, dim3(B, TS_SLICES, P.n_layers), dim3(TG_THREADS), 0, st, pdl_enabled(), P));
    return YL_OK;
}

}  // namespace yl

using namespace yl;

extern "C" int yl_build_target(const float *pred, const long *ps, const float *labels, int B, int F, int K,
                               int C, int layer_no, const float *anchors_px, const int *anchor_mask3, float ignore_thre,
                               float *target, float *obj_mask, float *tgt_mask, float *tgt_scale, int *status,
                               yl_stream_t stream)
{
    if (!labels || B <= 0 || K <= 0 || K > TG_MAXK || C <= 0) return YL_ERR_ARG;
    TargetParams P;
    P.n_layers = 1; P.K = K; P.C = C; P.labels = labels; P.ignore_thre = ignore_thre; P.status = status;
    const int rc = fill_target_layer(P.layer[0], pred, ps, F, layer_no, anchors_px, anchor_mask3, target, obj_mask, tgt_mask, tgt_scale);
    if (rc != YL_OK) return rc;
    return launch_targets(P, B, (cudaStream_t)stream);
}

extern "C" int yl_build_target3(const float *const *pred, const long *ps15, const float *labels, int B, const int *F, int K,
                                int C, int n_layers, const int *layer_no, const float *anchors_px, const int *anchor_mask,
                                float ignore_thre, float *const *target, float *const *obj_mask, float *const *tgt_mask,
                                float *const *tgt_scale, int *status, yl_stream_t stream)
{
    if (!pred || !ps15 || !labels || !F || !layer_no || !anchor_mask || !target || !obj_mask || !tgt_mask || !tgt_scale) return YL_ERR_ARG;
    if (B <= 0 || K <= 0 || K > TG_MAXK || C <= 0 || n_layers < 1 || n_layers > 3) return YL_ERR_ARG;
    TargetParams P;
    P.n_layers = n_layers; P.K = K; P.C = C; P.labels = labels; P.ignore_thre = ignore_thre; P.status = status;
    for (int l = 0; l < n_layers; ++l) {
        if (layer_no[l] < 0 || layer_no[l] > 2) return YL_ERR_ARG;
        const int rc = fill_target_layer(P.layer[l], pred[l], ps15 + 5 * l, F[l], layer_no[l], anchors_px, anchor_mask + 3 * layer_no[l],
                                         target[l], obj_mask[l], tgt_mask[l], tgt_scale[l]);
        if (rc != YL_OK) return rc;
    }
    return launch_targets(P, B, (cudaStream_t)stream);
}

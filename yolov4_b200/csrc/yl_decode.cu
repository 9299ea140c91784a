// yl_decode.cu -- the contract-literal YOLOLayer.forward outputs.
//
//   k_decode_dense        eval branch (yololayer.py:146-166): planar raw [B,3,5+C,F,F] -> AoS rows [.., 5+C], written
//                         directly at the layer's row offset of the concatenated [B, M, 5+C] tensor (yolov4.py:324).
//                         Coalesced 256-byte plane reads, shared-memory transpose, linear coalesced row writes.
//   k_decode_train        train branch (yololayer.py:122-145): planar `output` (sigmoid on xy/obj/cls) + planar `pred`.
//   k_decode_train_bwd    d(output)/d(raw) for the autograd wrapper.
#include "yl_common.cuh"
#include "../../include/yolo_head.h"

namespace yl {

constexpr int DD_TP = 64;          // boxes per tile
constexpr int DD_THREADS = 256;    // 4 channel rows x 64 boxes per pass

// SXY: the centres take the grid-sensitivity decode fl(fl(fl(sigmoid(t) * sxy) + beta) + cell) (scale_x_y, DESIGN.md section 1);
// otherwise sxy / beta are not read.
template <bool SXY>
__global__ void __launch_bounds__(DD_THREADS)
k_decode_dense(const float *__restrict__ raw, int Fw, int F2, int C, float stride,
               float aw0, float ah0, float aw1, float ah1, float aw2, float ah2,
               float *__restrict__ out, long rows_per_image, long row_offset, int ba0, float sxy, float beta)
{
    extern __shared__ __align__(16) float tile[];   // [DD_TP][nch]: the output layout itself (odd nch, e.g. 85: conflict-free stores)
    const int nch = 5 + C;
    const int nchp = nch;
    const int ba = ba0 + (int)blockIdx.y;
    const int b = ba / 3, a = ba - 3 * b;
    const int p0 = blockIdx.x * DD_TP;
    const int np = min(DD_TP, F2 - p0);
    const int pl = threadIdx.x & (DD_TP - 1);
    const int kr = threadIdx.x / DD_TP;
    const float aw = (a == 0) ? aw0 : ((a == 1) ? aw1 : aw2);
    const float ah = (a == 0) ? ah0 : ((a == 1) ? ah1 : ah2);
    if (pl < np) {
        const int p = p0 + pl;
        const int gy = p / Fw, gx = p - gy * Fw;
        constexpr int KR = DD_THREADS / DD_TP;                       // channel rows per pass
        // this thread's channels are kr, kr+KR, ...: one pointer walks them, eight loads per batch at constant plane strides;
        // only the last batch of a row can be partial, so the full batches carry no per-load predicates or index arithmetic
        const size_t rs = (size_t)KR * F2;
        const float *q = raw + ((size_t)ba * nch + kr) * F2 + p;
        float *tp = tile + pl * nchp + kr;
        // first batch: slot 0 is one of tx, ty, tw, th; the others are obj / classes
        {
            float t[8];
            if (kr + KR * 7 < nch) {
#pragma unroll
                for (int u = 0; u < 8; ++u) t[u] = ldg_stream1(q + u * rs);
            } else {
#pragma unroll
                for (int u = 0; u < 8; ++u) t[u] = (kr + KR * u < nch) ? ldg_stream1(q + u * rs) : 0.0f;
            }
            float sg[8];
            spec_sigmoid_batch<8>(t, sg);                              // one range test for the batch
            if (kr >= 2) sg[0] = spec_expf(t[0]);                       // tw / th
            float v0;
            if constexpr (SXY) {
                if (kr < 2) sg[0] = __fadd_rn(__fmul_rn(sg[0], sxy), beta);
            }
            if (kr == 0) v0 = __fmul_rn(__fadd_rn(sg[0], (float)gx), stride);
            else if (kr == 1) v0 = __fmul_rn(__fadd_rn(sg[0], (float)gy), stride);
            else if (kr == 2) v0 = __fmul_rn(__fmul_rn(sg[0], aw), stride);
            else v0 = __fmul_rn(__fmul_rn(sg[0], ah), stride);
            tp[0] = v0;
#pragma unroll
            for (int u = 1; u < 8; ++u)
                if (kr + KR * u < nch) tp[KR * u] = sg[u];
        }
        // the remaining batches are class channels only
        int k0 = kr + KR * 8;
        q += 8 * rs;
        tp += KR * 8;
        for (; k0 + KR * 7 < nch; k0 += KR * 8, q += 8 * rs, tp += KR * 8) {
            float t[8], sg[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) t[u] = ldg_stream1(q + u * rs);
            spec_sigmoid_batch<8>(t, sg);
#pragma unroll
            for (int u = 0; u < 8; ++u) tp[KR * u] = sg[u];
        }
        if (k0 < nch) {
            float t[8], sg[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) t[u] = (k0 + KR * u < nch) ? ldg_stream1(q + u * rs) : 0.0f;
            spec_sigmoid_batch<8>(t, sg);
#pragma unroll
            for (int u = 0; u < 8; ++u)
                if (k0 + KR * u < nch) tp[KR * u] = sg[u];
        }
    }
    __syncthreads();
    // the tile is a contiguous run of np*nch floats in the output: straight copy, 128-bit where the run is aligned
    float *dst = out + ((size_t)b * rows_per_image + row_offset + (size_t)a * F2 + p0) * nch;
    const int n = np * nch;
    if ((((uintptr_t)dst) & 15) == 0) {
        const int n4 = n >> 2;
        for (int e = threadIdx.x; e < n4; e += DD_THREADS)
            reinterpret_cast<float4 *>(dst)[e] = reinterpret_cast<const float4 *>(tile)[e];
        for (int e = (n4 << 2) + threadIdx.x; e < n; e += DD_THREADS) dst[e] = tile[e];
    } else {
        for (int e = threadIdx.x; e < n; e += DD_THREADS) dst[e] = tile[e];
    }
}

constexpr int DT_THREADS = 256;

// One CTA per plane (image, anchor, channel): the channel's case analysis is CTA-uniform and no thread divides a 64-bit
// element index by F*F / (5+C) (the grid-stride form spent more instructions on that than on the spec math).
template <int VEC>
__global__ void __launch_bounds__(DT_THREADS)
k_decode_train(const float *__restrict__ raw, int Fw, int F2, int C,
               float aw0, float ah0, float aw1, float ah1, float aw2, float ah2,
               float *__restrict__ output_planar, float *__restrict__ pred_planar)
{
    const int nch = 5 + C;
    const unsigned plane = blockIdx.x;
    const int ba = (int)(plane / (unsigned)nch);
    const int k = (int)(plane - (unsigned)ba * (unsigned)nch);
    const int a = ba % 3;
    const size_t base = (size_t)plane * F2;
    const bool sig = (k != 2 && k != 3);                                      // yololayer.py:105
    const float anc = (k == 2) ? ((a == 0) ? aw0 : ((a == 1) ? aw1 : aw2)) : ((a == 0) ? ah0 : ((a == 1) ? ah1 : ah2));
    float *pdst = pred_planar + ((size_t)ba * 4 + (k < 4 ? k : 0)) * F2;
    for (int p = threadIdx.x * VEC; p < F2; p += DT_THREADS * VEC) {
        Vec<VEC> t;
        t.load(raw + base + p);
        float o[VEC];
        if (VEC == 4 && sig) {                                                // two values per packed op, one range test
            const float tt[4] = {t.v[0], t.v[1 % VEC], t.v[2 % VEC], t.v[3 % VEC]};
            float ss[4];
            spec_sigmoid_batch<4>(tt, ss);
            o[0] = ss[0]; o[1 % VEC] = ss[1]; o[2 % VEC] = ss[2]; o[3 % VEC] = ss[3];
        } else {
#pragma unroll
            for (int v = 0; v < VEC; ++v) o[v] = sig ? spec_sigmoidf(t.v[v]) : t.v[v];
        }
        if (VEC == 4) *reinterpret_cast<float4 *>(output_planar + base + p) = make_float4(o[0], o[1 % VEC], o[2 % VEC], o[3 % VEC]);
        else output_planar[base + p] = o[0];
        if (k < 4) {
            float pv[VEC], ex[VEC];
            if (k >= 2) {
                if (VEC == 4) { spec_exp2(t.v[0], t.v[1 % VEC], ex[0], ex[1 % VEC]); spec_exp2(t.v[2 % VEC], t.v[3 % VEC], ex[2 % VEC], ex[3 % VEC]); }
                else ex[0] = spec_expf(t.v[0]);
            }
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                const int pp = p + v;
                if (k == 0) pv[v] = __fadd_rn(o[v], (float)(pp % Fw));                   // :126
                else if (k == 1) pv[v] = __fadd_rn(o[v], (float)(pp / Fw));              // :129
                else pv[v] = __fmul_rn(ex[v], anc);                                      // :132, :134
            }
            if (VEC == 4) *reinterpret_cast<float4 *>(pdst + p) = make_float4(pv[0], pv[1 % VEC], pv[2 % VEC], pv[3 % VEC]);
            else pdst[p] = pv[0];
        }
    }
}

// FROM_RAW: `src` is the raw head tensor and sigmoid(raw) is recomputed with the spec sequence (the bits of the forward pass),
// so the autograd node does not have to keep the tensor it returned: the reference's YOLOLoss.forward multiplies `output` by its
// masks IN PLACE (yololoss.py:402-408), which would invalidate a saved `output`.  Otherwise `src` is the forward's output_planar.
template <int VEC, bool FROM_RAW>
__global__ void __launch_bounds__(DT_THREADS)
k_decode_train_bwd(const float *__restrict__ src, const float *__restrict__ grad_out, int F2, int C,
                   float *__restrict__ grad_raw)
{
    const int nch = 5 + C;
    const unsigned plane = blockIdx.x;
    const int k = (int)(plane % (unsigned)nch);
    const size_t base = (size_t)plane * F2;
    const bool sig = (k != 2 && k != 3);
    for (int p = threadIdx.x * VEC; p < F2; p += DT_THREADS * VEC) {
        Vec<VEC> g, o;
        g.load(grad_out + base + p);
        if (sig) {
            o.load(src + base + p);
            if (FROM_RAW) {
                if (VEC == 4) {
                    const float tt[4] = {o.v[0], o.v[1 % VEC], o.v[2 % VEC], o.v[3 % VEC]};
                    float ss[4];
                    spec_sigmoid_batch<4>(tt, ss);
                    o.v[0] = ss[0]; o.v[1 % VEC] = ss[1]; o.v[2 % VEC] = ss[2]; o.v[3 % VEC] = ss[3];
                } else {
                    o.v[0] = spec_sigmoidf(o.v[0]);
                }
            }
        }
        float r[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) r[v] = sig ? (g.v[v] * (1.0f - o.v[v])) * o.v[v] : g.v[v];     // ATen sigmoid_backward order
        if (VEC == 4) *reinterpret_cast<float4 *>(grad_raw + base + p) = make_float4(r[0], r[1 % VEC], r[2 % VEC], r[3 % VEC]);
        else grad_raw[base + p] = r[0];
    }
}

}  // namespace yl

using namespace yl;

extern "C" int yl_decode_dense_ex(const float *raw, int B, int F, int C, const float *ag, float stride, float scale_x_y,
                                  float *out, long rows_per_image, long row_offset, yl_stream_t stream)
{
    if (!raw || !ag || !out || B <= 0 || F <= 0 || C <= 0 || rows_per_image < 3L * F * F + row_offset || row_offset < 0)
        return YL_ERR_ARG;
    if (3L * B > 0x7FFFFFFFL || !scale_xy_valid(scale_x_y)) return YL_ERR_ARG;
    const int F2 = F * F;
    const size_t smem = sizeof(float) * DD_TP * (5 + C);
    // a scale of exactly 1 is the unscaled kernel (the same launch and bytes as yl_decode_dense)
    const bool scaled = scale_x_y != 1.0f;
    const float beta = scale_xy_beta(scale_x_y);
    auto kernel = scaled ? k_decode_dense<true> : k_decode_dense<false>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return YL_ERR_CUDA_BASE + (int)e;
    }
    // gridDim.y is at most 65535: larger batches go out in slices of (image, anchor) pairs, one launch when B*3 fits
    constexpr int kMaxGridY = 65535;
    const long pairs = 3L * B;
    for (long ba0 = 0; ba0 < pairs; ba0 += kMaxGridY) {
        dim3 grid((F2 + DD_TP - 1) / DD_TP, (unsigned)min((long)kMaxGridY, pairs - ba0));
        kernel<<<grid, DD_THREADS, smem, (cudaStream_t)stream>>>(raw, F, F2, C, stride, ag[0], ag[1], ag[2], ag[3], ag[4], ag[5], out,
                                                                 rows_per_image, row_offset, (int)ba0, scale_x_y, beta);
        YL_LAUNCH_CHECK();
    }
    return YL_OK;
}

extern "C" int yl_decode_dense(const float *raw, int B, int F, int C, const float *ag, float stride,
                               float *out, long rows_per_image, long row_offset, yl_stream_t stream)
{
    return yl_decode_dense_ex(raw, B, F, C, ag, stride, 1.0f, out, rows_per_image, row_offset, stream);
}

extern "C" int yl_decode_train(const float *raw, int B, int F, int C, const float *ag,
                               float *output_planar, float *pred_planar, yl_stream_t stream)
{
    if (!raw || !ag || !output_planar || !pred_planar || B <= 0 || F <= 0 || C <= 0) return YL_ERR_ARG;
    const int F2 = F * F;
    const long planes = (long)B * 3 * (5 + C);
    if (planes > 0x7FFFFFFFL) return YL_ERR_ARG;
    // planes are 16-byte aligned when F*F is a multiple of 4 and the bases are: then four elements per thread
    const bool vec4 = (F2 % 4 == 0) && (((uintptr_t)raw | (uintptr_t)output_planar | (uintptr_t)pred_planar) % 16 == 0);
    if (vec4)
        k_decode_train<4><<<(unsigned)planes, DT_THREADS, 0, (cudaStream_t)stream>>>(raw, F, F2, C, ag[0], ag[1], ag[2], ag[3], ag[4],
                                                                                   ag[5], output_planar, pred_planar);
    else
        k_decode_train<1><<<(unsigned)planes, DT_THREADS, 0, (cudaStream_t)stream>>>(raw, F, F2, C, ag[0], ag[1], ag[2], ag[3], ag[4],
                                                                                   ag[5], output_planar, pred_planar);
    YL_LAUNCH_CHECK();
    return YL_OK;
}

static int decode_train_backward_impl(const float *src, const float *grad_out_planar, int B, int F, int C, float *grad_raw,
                                      yl_stream_t stream, bool from_raw)
{
    if (!src || !grad_out_planar || !grad_raw || B <= 0 || F <= 0 || C <= 0) return YL_ERR_ARG;
    const int F2 = F * F;
    const long planes = (long)B * 3 * (5 + C);
    if (planes > 0x7FFFFFFFL) return YL_ERR_ARG;
    const bool vec4 = (F2 % 4 == 0) && (((uintptr_t)src | (uintptr_t)grad_out_planar | (uintptr_t)grad_raw) % 16 == 0);
    cudaStream_t st = (cudaStream_t)stream;
    if (vec4) {
        if (from_raw) k_decode_train_bwd<4, true><<<(unsigned)planes, DT_THREADS, 0, st>>>(src, grad_out_planar, F2, C, grad_raw);
        else k_decode_train_bwd<4, false><<<(unsigned)planes, DT_THREADS, 0, st>>>(src, grad_out_planar, F2, C, grad_raw);
    } else {
        if (from_raw) k_decode_train_bwd<1, true><<<(unsigned)planes, DT_THREADS, 0, st>>>(src, grad_out_planar, F2, C, grad_raw);
        else k_decode_train_bwd<1, false><<<(unsigned)planes, DT_THREADS, 0, st>>>(src, grad_out_planar, F2, C, grad_raw);
    }
    YL_LAUNCH_CHECK();
    return YL_OK;
}

extern "C" int yl_decode_train_backward(const float *output_planar, const float *grad_out_planar, int B, int F, int C,
                                        float *grad_raw, yl_stream_t stream)
{
    return decode_train_backward_impl(output_planar, grad_out_planar, B, F, C, grad_raw, stream, false);
}

extern "C" int yl_decode_train_backward_raw(const float *raw, const float *grad_out_planar, int B, int F, int C,
                                            float *grad_raw, yl_stream_t stream)
{
    return decode_train_backward_impl(raw, grad_out_planar, B, F, C, grad_raw, stream, true);
}

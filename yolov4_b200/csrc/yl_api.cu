// yl_api.cu -- ABI bookkeeping and the host-buffer entry point (yl_context / yl_detect_host).
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "yl_common.cuh"
#include "../../include/yolo_head.h"

extern "C" int yl_abi_version(void) { return YL_ABI_VERSION; }

#ifndef YL_SOURCE_HASH
#define YL_SOURCE_HASH "unknown"
#endif
extern "C" const char *yl_source_hash(void) { return YL_SOURCE_HASH; }

extern "C" const char *yl_error_string(int code)
{
    static thread_local char buf[160];
    switch (code) {
    case YL_OK: return "ok";
    case YL_ERR_ARG: return "invalid argument (null pointer, non-positive size or unsupported shape)";
    case YL_ERR_CLASSES: return "too many classes for the candidate bitmask (YL_MAX_CLASSES)";
    case YL_ERR_WORKSPACE: return "workspace smaller than yl_post_workspace_bytes()";
    case YL_ERR_CAPACITY: return "a class segment overflowed cap_seg; recreate the context with a larger cap_seg";
    default: break;
    }
    if (code >= YL_ERR_CUDA_BASE) {
        snprintf(buf, sizeof(buf), "CUDA error %d: %s", code - YL_ERR_CUDA_BASE, cudaGetErrorString((cudaError_t)(code - YL_ERR_CUDA_BASE)));
        return buf;
    }
    return "unknown error";
}

// Self-test of the spec math: rcp_rn_bounded(d) against __frcp_rn(d) (= the IEEE quotient 1.0f / d of the oracle) for every
// float d in [1, 2^125]; *bad_dev receives the number of mismatches.
namespace yl {
__global__ void k_selftest_rcp(unsigned long long *bad)
{
    const unsigned lo = 0x3F800000u, hi = 0x7E000000u;              // 1.0f .. 2^125
    unsigned long long n = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x + lo; i <= hi;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const float d = __uint_as_float((unsigned)i);
        n += (__float_as_uint(rcp_rn_bounded(d)) != __float_as_uint(__frcp_rn(d))) ? 1ull : 0ull;
    }
    if (n) atomicAdd(bad, n);
}
}  // namespace yl

extern "C" int yl_selftest_rcp(unsigned long long *bad_dev, yl_stream_t stream)
{
    if (!bad_dev) return YL_ERR_ARG;
    YL_CUDA_TRY(cudaMemsetAsync(bad_dev, 0, sizeof(unsigned long long), (cudaStream_t)stream));
    yl::k_selftest_rcp<<<148 * 16, 256, 0, (cudaStream_t)stream>>>(bad_dev);
    YL_LAUNCH_CHECK();
    return YL_OK;
}

// -------------------------------------------------------------------------------------------------------------
// Host-buffer path.  Images are independent (utils.py:133), so the batch is cut into groups: group g's H2D copy
// runs on the copy stream while group g-1 is filtered and suppressed on the compute stream and the kept rows of
// group g-2 travel back on a third stream (PCIe is full duplex), so only the last group's results trail the uploads.
// -------------------------------------------------------------------------------------------------------------
struct yl_context {
    int device, B, n_layers, C, cap_seg, n_groups, dtype;
    size_t esize;                  // bytes per head tensor element (dtype)
    long cap_out, M;
    int F[3];
    float anchors[18];
    int mask[9];
    void *d_raw[3];
    void *ws;
    size_t ws_bytes;
    float *d_rows;
    int *d_meta;
    int *h_meta;                   // pinned
    cudaStream_t s_copy, s_comp, s_back;
    cudaEvent_t ev_copied[16], ev_meta[16], ev_done;
};

extern "C" int yl_context_destroy(yl_context *c)
{
    if (!c) return YL_OK;
    cudaSetDevice(c->device);
    for (int l = 0; l < 3; ++l) if (c->d_raw[l]) cudaFree(c->d_raw[l]);
    if (c->ws) cudaFree(c->ws);
    if (c->d_rows) cudaFree(c->d_rows);
    if (c->d_meta) cudaFree(c->d_meta);
    if (c->h_meta) cudaFreeHost(c->h_meta);
    for (int g = 0; g < 16; ++g) if (c->ev_copied[g]) cudaEventDestroy(c->ev_copied[g]);
    for (int g = 0; g < 16; ++g) if (c->ev_meta[g]) cudaEventDestroy(c->ev_meta[g]);
    if (c->s_back) cudaStreamDestroy(c->s_back);
    if (c->ev_done) cudaEventDestroy(c->ev_done);
    if (c->s_copy) cudaStreamDestroy(c->s_copy);
    if (c->s_comp) cudaStreamDestroy(c->s_comp);
    free(c);
    return YL_OK;
}

extern "C" int yl_context_create_typed(yl_context **out, int device, int B, const int *F, int n_layers, int C, int dtype,
                                       const float *anchors_px, const int *anchor_mask, int cap_seg, long cap_out)
{
    if (!out || !F || !anchors_px || !anchor_mask || B <= 0 || n_layers < 1 || n_layers > 3 || C <= 0 || cap_seg <= 0 || cap_out <= 0)
        return YL_ERR_ARG;
    if (dtype != YL_DTYPE_F32 && dtype != YL_DTYPE_F16 && dtype != YL_DTYPE_BF16) return YL_ERR_ARG;
    if (C > YL_MAX_CLASSES) return YL_ERR_CLASSES;
    yl_context *c = (yl_context *)calloc(1, sizeof(yl_context));
    if (!c) return YL_ERR_ARG;
    c->device = device; c->B = B; c->n_layers = n_layers; c->C = C; c->cap_seg = cap_seg; c->cap_out = cap_out;
    c->dtype = dtype; c->esize = dtype == YL_DTYPE_F32 ? sizeof(float) : 2;
    c->n_groups = B >= 16 ? 8 : (B >= 2 ? 2 : 1);
    memcpy(c->anchors, anchors_px, sizeof(float) * 18);
    memcpy(c->mask, anchor_mask, sizeof(int) * 9);
    c->M = 0;
    for (int l = 0; l < n_layers; ++l) { c->F[l] = F[l]; c->M += 3L * F[l] * F[l]; }
    int rc = YL_OK;
#define CTX_TRY(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { rc = YL_ERR_CUDA_BASE + (int)e__; goto fail; } } while (0)
    CTX_TRY(cudaSetDevice(device));
    for (int l = 0; l < n_layers; ++l)
        CTX_TRY(cudaMalloc(&c->d_raw[l], c->esize * (size_t)B * 3 * (5 + C) * F[l] * F[l]));
    c->ws_bytes = yl_post_workspace_bytes(B, c->M, C, cap_seg);
    CTX_TRY(cudaMalloc(&c->ws, c->ws_bytes));
    CTX_TRY(cudaMalloc(&c->d_rows, sizeof(float) * 7 * (size_t)B * cap_out));
    CTX_TRY(cudaMalloc(&c->d_meta, sizeof(int) * 3 * (size_t)B));
    CTX_TRY(cudaMallocHost(&c->h_meta, sizeof(int) * 3 * (size_t)B));
    CTX_TRY(cudaStreamCreateWithFlags(&c->s_copy, cudaStreamNonBlocking));
    CTX_TRY(cudaStreamCreateWithFlags(&c->s_comp, cudaStreamNonBlocking));
    CTX_TRY(cudaStreamCreateWithFlags(&c->s_back, cudaStreamNonBlocking));
    for (int g = 0; g < c->n_groups; ++g) CTX_TRY(cudaEventCreateWithFlags(&c->ev_copied[g], cudaEventDisableTiming));
    for (int g = 0; g < c->n_groups; ++g) CTX_TRY(cudaEventCreateWithFlags(&c->ev_meta[g], cudaEventDisableTiming));
    CTX_TRY(cudaEventCreateWithFlags(&c->ev_done, cudaEventDisableTiming));
#undef CTX_TRY
    *out = c;
    return YL_OK;
fail:
    yl_context_destroy(c);
    return rc;
}

extern "C" int yl_context_create(yl_context **out, int device, int B, const int *F, int n_layers, int C,
                                 const float *anchors_px, const int *anchor_mask, int cap_seg, long cap_out)
{
    return yl_context_create_typed(out, device, B, F, n_layers, C, YL_DTYPE_F32, anchors_px, anchor_mask, cap_seg, cap_out);
}

extern "C" int yl_detect_host_ex3(yl_context *c, const float *const *raw_host, float conf_thre, float nms_thre, int max_det,
                                  int agnostic, int diou, const float *scale_x_y, float *out_rows_host, int *counts_host)
{
    if (!c || !raw_host || !out_rows_host || !counts_host) return YL_ERR_ARG;
    if (max_det < 0 || max_det > c->cap_out) return YL_ERR_ARG;
    if (agnostic != 0 && agnostic != 1) return YL_ERR_ARG;
    if (diou != 0 && diou != 1) return YL_ERR_ARG;
    for (int l = 0; scale_x_y && l < c->n_layers; ++l)
        if (!yl::scale_xy_valid(scale_x_y[l])) return YL_ERR_ARG;
    YL_CUDA_TRY(cudaSetDevice(c->device));
    const int B = c->B, C = c->C, G = c->n_groups;
    const size_t need = yl_post_workspace_bytes_ex(B, c->M, C, c->cap_seg, agnostic);
    if (need == 0) return YL_ERR_ARG;
    if (c->ws_bytes < need) {
        // the agnostic scratch is allocated on first use; nothing is in flight here (every call ends synchronised)
        void *ws = nullptr;
        YL_CUDA_TRY(cudaMalloc(&ws, need));
        cudaFree(c->ws);
        c->ws = ws;
        c->ws_bytes = need;
    }
    int rc = yl_post_reset(c->ws, c->ws_bytes, B, c->M, C, c->cap_seg, c->s_comp);
    if (rc != YL_OK) return rc;
    for (int g = 0; g < G; ++g) {
        const int i0 = (int)((long)B * g / G), i1 = (int)((long)B * (g + 1) / G);
        if (i1 == i0) continue;
        for (int l = 0; l < c->n_layers; ++l) {
            const size_t per_img = (size_t)3 * (5 + C) * c->F[l] * c->F[l];
            // raw_host[l] holds elements of the context's dtype, whatever the declared pointer type
            const size_t off = c->esize * per_img * i0;
            YL_CUDA_TRY(cudaMemcpyAsync((char *)c->d_raw[l] + off, (const char *)raw_host[l] + off, c->esize * per_img * (i1 - i0),
                                        cudaMemcpyHostToDevice, c->s_copy));
        }
        YL_CUDA_TRY(cudaEventRecord(c->ev_copied[g], c->s_copy));
        YL_CUDA_TRY(cudaStreamWaitEvent(c->s_comp, c->ev_copied[g], 0));
        rc = yl_filter_raw_ex((const void *const *)c->d_raw, c->dtype, c->F, c->n_layers, B, C, c->anchors, c->mask, conf_thre,
                              scale_x_y, c->ws, c->ws_bytes, c->M, c->cap_seg, i0, i1 - i0, 3, c->s_comp);
        if (rc != YL_OK) return rc;
        rc = yl_nms_ex2(c->ws, c->ws_bytes, B, c->M, C, c->cap_seg, nms_thre, max_det, agnostic, diou, c->d_rows, c->cap_out,
                        c->d_meta, nullptr, i0, i1 - i0, c->s_comp);
        if (rc != YL_OK) return rc;
        // this group's three meta slices (kept rows, largest segment, candidate total) follow the kernels
        for (int k = 0; k < 3; ++k)
            YL_CUDA_TRY(cudaMemcpyAsync(c->h_meta + (size_t)k * B + i0, c->d_meta + (size_t)k * B + i0, sizeof(int) * (size_t)(i1 - i0),
                                        cudaMemcpyDeviceToHost, c->s_comp));
        YL_CUDA_TRY(cudaEventRecord(c->ev_meta[g], c->s_comp));
    }
    // everything above is enqueued; the host now follows the groups and sends each one's kept rows back while the
    // uploads of the later groups are still running
    int status = YL_OK;
    for (int g = 0; g < G; ++g) {
        const int i0 = (int)((long)B * g / G), i1 = (int)((long)B * (g + 1) / G);
        if (i1 == i0) continue;
        YL_CUDA_TRY(cudaEventSynchronize(c->ev_meta[g]));
        for (int b = i0; b < i1; ++b) {
            if (c->h_meta[B + b] > c->cap_seg) status = YL_ERR_CAPACITY;
            counts_host[b] = c->h_meta[b];
            const long k = c->h_meta[b] < c->cap_out ? c->h_meta[b] : c->cap_out;
            if (k > 0 && status == YL_OK)
                YL_CUDA_TRY(cudaMemcpyAsync(out_rows_host + (size_t)b * c->cap_out * 7, c->d_rows + (size_t)b * c->cap_out * 7,
                                            sizeof(float) * 7 * (size_t)k, cudaMemcpyDeviceToHost, c->s_back));
        }
    }
    YL_CUDA_TRY(cudaStreamSynchronize(c->s_back));
    YL_CUDA_TRY(cudaStreamSynchronize(c->s_comp));
    return status;
}

extern "C" int yl_detect_host_ex2(yl_context *c, const float *const *raw_host, float conf_thre, float nms_thre, int max_det,
                                  int agnostic, int diou, float *out_rows_host, int *counts_host)
{
    return yl_detect_host_ex3(c, raw_host, conf_thre, nms_thre, max_det, agnostic, diou, nullptr, out_rows_host, counts_host);
}

extern "C" int yl_detect_host_ex(yl_context *c, const float *const *raw_host, float conf_thre, float nms_thre, int max_det,
                                 int agnostic, float *out_rows_host, int *counts_host)
{
    return yl_detect_host_ex3(c, raw_host, conf_thre, nms_thre, max_det, agnostic, 0, nullptr, out_rows_host, counts_host);
}

extern "C" int yl_detect_host_topk(yl_context *c, const float *const *raw_host, float conf_thre, float nms_thre, int max_det,
                                   float *out_rows_host, int *counts_host)
{
    return yl_detect_host_ex(c, raw_host, conf_thre, nms_thre, max_det, 0, out_rows_host, counts_host);
}

extern "C" int yl_detect_host(yl_context *c, const float *const *raw_host, float conf_thre, float nms_thre,
                              float *out_rows_host, int *counts_host)
{
    return yl_detect_host_topk(c, raw_host, conf_thre, nms_thre, 0, out_rows_host, counts_host);
}

// yl_xchg.cu -- the final exchange of the image-sharded path (SURVEY.md 8(e)): every rank ends up with the detections of
// every image, rank r's images at rows [r*B, (r+1)*B).
//
// One process per GPU.  Each rank owns ONE device allocation (the "window") that its peers map through CUDA IPC:
//     rows   [slots][world*B][cap_out][7] fp32     counts [slots][world*B] i32
//     flag   [slots][world] u32   "source s has delivered epoch e of this slot"      (written by the peers)
//     ack    [slots][world] u32   "reader s has released epoch e of this slot"       (written by the peers)
//     epoch  [slots] u32          completed exchanges of the slot                      (local)
// k_xchg_push_bulk copies the kept rows of the local images (exactly counts[b] rows each) into every window: bulk copies
// through shared memory, then one bulk store per peer over NVLink, or one bulk store to the windows' multicast mapping that
// the switch replicates (fire-and-forget writes, no collective); it then publishes flag = epoch + 1 behind a system-scope
// fence.  k_xchg_wait spins (bounded) until every source's flag reached epoch + 1; k_xchg_release bumps the epoch and tells
// every peer that this rank is done reading the slot, which is what a peer's next push into that slot waits for (credit: a
// slot is never overwritten while somebody still reads it).  Nothing here needs a host synchronisation or a changing kernel
// argument, so push / wait / release are captured into the step's CUDA graph on a side branch and the exchange of step i
// runs under the kernels of step i+1.
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "yl_common.cuh"
#include "../../include/yolo_head.h"

namespace yl {

constexpr int XCHG_MAX_WORLD = 16;

struct XchgWindow {                  // device pointers into ONE rank's window
    float *rows;
    int *counts;
    unsigned *flag, *ack, *epoch;
};
struct XchgPeers {
    XchgWindow w[XCHG_MAX_WORLD];
};

struct XchgLayout {
    size_t off_rows, off_counts, off_flag, off_ack, off_epoch, off_done, off_status, total;
};
static XchgLayout xchg_layout(int world, int B, long cap_out, int slots)
{
    XchgLayout L;
    size_t o = 0;
    L.off_rows = o;   o += align_up(sizeof(float) * 7 * (size_t)slots * world * B * cap_out, 256);
    L.off_counts = o; o += align_up(sizeof(int) * (size_t)slots * world * B, 256);
    L.off_flag = o;   o += align_up(sizeof(unsigned) * (size_t)slots * XCHG_MAX_WORLD, 256);
    L.off_ack = o;    o += align_up(sizeof(unsigned) * (size_t)slots * XCHG_MAX_WORLD, 256);
    L.off_epoch = o;  o += align_up(sizeof(unsigned) * (size_t)slots, 256);
    L.off_done = o;   o += align_up(sizeof(unsigned) * (size_t)slots, 256);
    L.off_status = o; o += 256;
    L.total = o;
    return L;
}

__device__ __forceinline__ unsigned ld_sys(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_sys(unsigned *p, unsigned v)
{
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long now_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// Spin until *p >= want (wrap-safe), at most limit_ns; returns false on time-out (the caller records it instead of hanging).
__device__ __forceinline__ bool spin_ge(const unsigned *p, unsigned want, unsigned long long limit_ns)
{
    const unsigned long long t0 = now_ns();
    while ((int)(ld_sys(p) - want) < 0) {
        __nanosleep(200);
        if (now_ns() - t0 > limit_ns) return false;
    }
    return true;
}

// ---- the push: the rows go global -> shared memory -> every window as cp.async.bulk transfers of XB_BYTES (SASS UBLKCP),
// issued by ONE thread per CTA over a ring of XB_STAGES shared-memory stages.  No register staging, no per-thread 16-byte
// stores: the copy engines of the SM (TMA) produce large NVLink write bursts while the CTA's other warps do not exist at all
// (32 threads per CTA), so the push takes almost nothing from the step's kernels it runs next to.  With a multicast mapping
// (windows in symmetric memory; torch does the CUDA VMM / fabric plumbing) one bulk store reaches every rank's window and the
// switch replicates it: a rank sends 1/world of the bytes of the per-peer stores, and what arrives is unchanged.
__device__ __forceinline__ void mc_st1(unsigned *mc, unsigned v)
{
    asm volatile("multimem.st.relaxed.sys.global.u32 [%0], %1;" ::"l"(mc), "r"(v) : "memory");
}

constexpr unsigned XB_BYTES = 16384;
constexpr int XB_STAGES = 4;
constexpr int XB_DEPTH = 1;                    // bulk loads in flight ahead of the stores (XB_DEPTH < XB_STAGES); deeper look-ahead with
                                               // 4 KB units measured no better (the push is not what bounds the exchange)
constexpr int XB_SMEM = XB_STAGES * (int)XB_BYTES;     // dynamic shared memory of k_xchg_push_bulk

__device__ __forceinline__ unsigned xb_smem(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

struct XbUnit { int b; unsigned lo, len; };

__global__ void __launch_bounds__(32)
k_xchg_push_bulk(const __grid_constant__ XchgPeers P, XchgWindow mc, int rank, int world, int B, long cap_out, int slots, int slot,
                 const float *__restrict__ rows, const int *__restrict__ counts, unsigned *__restrict__ done,
                 int *__restrict__ status, unsigned long long limit_ns)
{
    extern __shared__ __align__(128) unsigned char xb_stage[];         // XB_STAGES x XB_BYTES
    __shared__ __align__(8) unsigned long long bar[XB_STAGES];
    __shared__ int sh_ok;
    const XchgWindow &me = P.w[rank];
    const unsigned epoch = me.epoch[slot];
    if (threadIdx.x == 0) sh_ok = 1;
    __syncwarp();
    // credit: every reader has released the previous use of this slot
    if (threadIdx.x < world && !spin_ge(me.ack + slot * XCHG_MAX_WORLD + threadIdx.x, epoch, limit_ns)) sh_ok = 0;
    __syncwarp();
    if (!sh_ok) {
        if (threadIdx.x == 0) atomicExch(status, 1);
        return;
    }
    const size_t img_bytes = (size_t)cap_out * 28;                     // cap_out % 4 == 0: a multiple of 16
    const int n_chunks = (int)((img_bytes + XB_BYTES - 1) / XB_BYTES);
    if (threadIdx.x == 0) {
        for (int s = 0; s < XB_STAGES; ++s)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(xb_smem(&bar[s])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        // The CTA's units are (image, 4 KB chunk) pairs u = blockIdx.x, + gridDim.x, ... that lie inside the image's kept rows.
        // Two cursors walk that sequence: `up` issues the bulk loads XB_DEPTH units ahead, `uc` stores what has landed.
        const int n_units = B * n_chunks;
        auto next = [&](int &u, XbUnit &U) -> bool {
            for (; u < n_units; u += gridDim.x) {
                const int b = u / n_chunks, c = u - b * n_chunks;
                const int n = min(max(counts[b], 0), (int)cap_out);
                const size_t nbytes = (((size_t)n * 28 + 15) / 16) * 16;   // whole 16-byte units: the padding lies inside the image's capacity
                const size_t lo = (size_t)c * XB_BYTES;
                if (lo < nbytes) {
                    U.b = b; U.lo = (unsigned)lo; U.len = (unsigned)min((size_t)XB_BYTES, nbytes - lo);
                    u += gridDim.x;
                    return true;
                }
            }
            return false;
        };
        auto load = [&](const XbUnit &U, unsigned k) {
            const int s = (int)(k % XB_STAGES);
            // the stage is free once the store group that read it XB_STAGES units ago has read it; groups committed so far: k - XB_DEPTH
            asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(XB_STAGES - XB_DEPTH - 1) : "memory");
            const char *src = reinterpret_cast<const char *>(rows) + (size_t)U.b * img_bytes + U.lo;
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(xb_smem(&bar[s])), "r"(U.len) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(xb_smem(xb_stage + (size_t)s * XB_BYTES)), "l"(src), "r"(U.len), "r"(xb_smem(&bar[s])) : "memory");
        };
        int up = blockIdx.x, uc = blockIdx.x;
        unsigned kp = 0, kc = 0;                                       // units loaded / stored
        XbUnit U;
        for (; kp < (unsigned)XB_DEPTH && next(up, U); ++kp) load(U, kp);
        XbUnit V;
        while (next(uc, V)) {
            if (next(up, U)) { load(U, kp); ++kp; }
            const int s = (int)(kc % XB_STAGES);
            const unsigned parity = (kc / XB_STAGES) & 1u;
            unsigned ok;
            do {
                asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                             : "=r"(ok) : "r"(xb_smem(&bar[s])), "r"(parity) : "memory");
            } while (!ok);
            const unsigned src_s = xb_smem(xb_stage + (size_t)s * XB_BYTES);
            const size_t dst_off = (((size_t)slot * world * B + (size_t)rank * B + V.b)) * img_bytes + V.lo;
            if (mc.rows) {                                             // multicast mapping: one bulk store, the switch replicates
                char *dst = reinterpret_cast<char *>(mc.rows) + dst_off;
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src_s), "r"(V.len) : "memory");
            } else {
                for (int p = 0; p < world; ++p) {
                    char *dst = reinterpret_cast<char *>(P.w[p].rows) + dst_off;
                    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src_s), "r"(V.len) : "memory");
                }
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            ++kc;
        }
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");     // every store of this CTA has been performed
    }
    // counts (a few bytes per image) by plain stores
    for (int b = blockIdx.x * 32 + threadIdx.x; b < B; b += gridDim.x * 32) {
        const int n = min(max(counts[b], 0), (int)cap_out);
        const size_t ci = (size_t)slot * world * B + (size_t)rank * B + b;
        if (mc.rows) mc_st1(reinterpret_cast<unsigned *>(mc.counts) + ci, (unsigned)n);
        else for (int p = 0; p < world; ++p) P.w[p].counts[ci] = n;
    }
    __syncwarp();
    if (threadIdx.x == 0) {
        asm volatile("fence.proxy.async;" ::: "memory");
        __threadfence_system();
        sh_ok = (atomicAdd(done + slot, 1u) == gridDim.x - 1) ? 2 : 1;
    }
    __syncwarp();
    if (sh_ok == 2) {
        if (threadIdx.x == 0) done[slot] = 0u;
        __threadfence_system();
        if (mc.rows) { if (threadIdx.x == 0) mc_st1(mc.flag + slot * XCHG_MAX_WORLD + rank, epoch + 1u); }
        else if (threadIdx.x < world) st_sys(P.w[threadIdx.x].flag + slot * XCHG_MAX_WORLD + rank, epoch + 1u);
    }
}

__global__ void k_xchg_wait(const __grid_constant__ XchgPeers P, int rank, int world, int slot, int *__restrict__ status,
                            unsigned long long limit_ns)
{
    const XchgWindow &me = P.w[rank];
    const unsigned epoch = me.epoch[slot];
    if (threadIdx.x < world && !spin_ge(me.flag + slot * XCHG_MAX_WORLD + threadIdx.x, epoch + 1u, limit_ns)) atomicExch(status, 2);
    __threadfence_system();
}

__global__ void k_xchg_release(const __grid_constant__ XchgPeers P, int rank, int world, int slot)
{
    const XchgWindow &me = P.w[rank];
    __shared__ unsigned sh_epoch;
    if (threadIdx.x == 0) sh_epoch = me.epoch[slot] + 1u;
    __syncthreads();
    if (threadIdx.x < world) st_sys(P.w[threadIdx.x].ack + slot * XCHG_MAX_WORLD + rank, sh_epoch);
    __syncthreads();
    if (threadIdx.x == 0) me.epoch[slot] = sh_epoch;
}

}  // namespace yl

using namespace yl;

struct yl_xchg {
    int device, rank, world, B, slots, push_ctas;
    long cap_out;
    XchgLayout L;
    char *window;                      // this rank's allocation
    char *peer[XCHG_MAX_WORLD];        // mapped windows (peer[rank] == window)
    XchgPeers P;
    unsigned long long limit_ns;
    bool connected, external;          // external: the windows belong to the caller (symmetric memory), not to this object
    char *mc;                          // multicast mapping of the windows, or null
    XchgWindow MC;
};

static XchgWindow window_of(char *base, const XchgLayout &L)
{
    XchgWindow w;
    w.rows = (float *)(base + L.off_rows);
    w.counts = (int *)(base + L.off_counts);
    w.flag = (unsigned *)(base + L.off_flag);
    w.ack = (unsigned *)(base + L.off_ack);
    w.epoch = (unsigned *)(base + L.off_epoch);
    return w;
}

extern "C" int yl_xchg_destroy(yl_xchg *x)
{
    if (!x) return YL_OK;
    cudaSetDevice(x->device);
    if (!x->external) {
        for (int p = 0; p < x->world; ++p)
            if (p != x->rank && x->peer[p]) cudaIpcCloseMemHandle(x->peer[p]);
        if (x->window) cudaFree(x->window);
    }
    free(x);
    return YL_OK;
}

// What both creation paths share on the host: the argument checks, the window layout, the time limit and the push grid.  Returns
// null for arguments they reject and when the allocation fails (both YL_ERR_ARG).  Through the multicast mapping a rank sends
// 1/world of the bytes: 16 single-warp CTAs keep the switch busy (8 GPUs: 267 us per step with 16, 273 us with 64); the stores
// to every peer want 64.
static yl_xchg *xchg_new(int device, int rank, int world, int B, long cap_out, int slots, bool multicast)
{
    if (rank < 0 || world < 1 || world > XCHG_MAX_WORLD || rank >= world || B <= 0 || cap_out <= 0 || cap_out % 4 != 0 || slots < 1 ||
        slots > 8)
        return nullptr;
    yl_xchg *x = (yl_xchg *)calloc(1, sizeof(yl_xchg));
    if (!x) return nullptr;
    x->device = device; x->rank = rank; x->world = world; x->B = B; x->cap_out = cap_out; x->slots = slots;
    x->L = xchg_layout(world, B, cap_out, slots);
    x->limit_ns = 5000000000ull;                                     // 5 s: a missing peer is reported, not waited for forever
    x->push_ctas = multicast ? 16 : 64;
    return x;
}

// What both share on the object's device, once it is current and x->window is set: the push kernel may use XB_SMEM bytes of
// dynamic shared memory (an attribute of each device, so every object sets it on its own device and the push sets nothing),
// and this rank's flags, acks, epochs and counters start at zero (the row area needs no initialisation).
static cudaError_t xchg_init_window(yl_xchg *x)
{
    cudaError_t e = cudaFuncSetAttribute(k_xchg_push_bulk, cudaFuncAttributeMaxDynamicSharedMemorySize, XB_SMEM);
    if (e == cudaSuccess) e = cudaMemset(x->window + x->L.off_counts, 0, x->L.total - x->L.off_counts);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    return e;
}

extern "C" int yl_xchg_create(yl_xchg **out, int device, int rank, int world, int B, long cap_out, int slots)
{
    yl_xchg *x = out ? xchg_new(device, rank, world, B, cap_out, slots, false) : nullptr;
    if (!x) return YL_ERR_ARG;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaMalloc(&x->window, x->L.total);
    if (e == cudaSuccess) e = xchg_init_window(x);
    if (e != cudaSuccess) { yl_xchg_destroy(x); return YL_ERR_CUDA_BASE + (int)e; }
    x->peer[rank] = x->window;
    *out = x;
    return YL_OK;
}

extern "C" size_t yl_xchg_window_bytes(int world, int B, long cap_out, int slots)
{
    if (world < 1 || world > XCHG_MAX_WORLD || B <= 0 || cap_out <= 0 || cap_out % 4 != 0 || slots < 1 || slots > 8) return 0;
    return xchg_layout(world, B, cap_out, slots).total;
}

extern "C" int yl_xchg_create_external(yl_xchg **out, int device, int rank, int world, int B, long cap_out, int slots,
                                       void *const *windows, void *multicast)
{
    yl_xchg *x = (out && windows) ? xchg_new(device, rank, world, B, cap_out, slots, multicast != nullptr) : nullptr;
    if (!x) return YL_ERR_ARG;
    for (int p = 0; p < world; ++p)
        if (!windows[p] || ((uintptr_t)windows[p]) % 256 != 0) { free(x); return YL_ERR_ARG; }
    x->external = true;
    for (int p = 0; p < world; ++p) { x->peer[p] = (char *)windows[p]; x->P.w[p] = window_of(x->peer[p], x->L); }
    x->window = x->peer[rank];
    x->mc = (char *)multicast;
    if (x->mc) x->MC = window_of(x->mc, x->L);
    // only THIS rank's window is zeroed: the caller synchronises the ranks before the first push
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = xchg_init_window(x);
    if (e != cudaSuccess) { free(x); return YL_ERR_CUDA_BASE + (int)e; }
    x->connected = true;
    *out = x;
    return YL_OK;
}

extern "C" size_t yl_xchg_handle_bytes(void) { return sizeof(cudaIpcMemHandle_t); }

extern "C" int yl_xchg_local_handle(yl_xchg *x, void *handle)
{
    if (!x || !handle) return YL_ERR_ARG;
    YL_CUDA_TRY(cudaSetDevice(x->device));
    cudaIpcMemHandle_t h;
    YL_CUDA_TRY(cudaIpcGetMemHandle(&h, x->window));
    memcpy(handle, &h, sizeof(h));
    return YL_OK;
}

extern "C" int yl_xchg_connect(yl_xchg *x, const void *handles)
{
    if (!x || (!handles && x->world > 1)) return YL_ERR_ARG;
    YL_CUDA_TRY(cudaSetDevice(x->device));
    for (int p = 0; p < x->world; ++p) {
        if (p == x->rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char *)handles + (size_t)p * sizeof(h), sizeof(h));
        void *ptr = nullptr;
        YL_CUDA_TRY(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
        x->peer[p] = (char *)ptr;
    }
    for (int p = 0; p < x->world; ++p) x->P.w[p] = window_of(x->peer[p], x->L);
    x->connected = true;
    return YL_OK;
}

extern "C" int yl_xchg_push(yl_xchg *x, const float *rows, const int *counts, int slot, yl_stream_t stream)
{
    if (!x || !rows || !counts || slot < 0 || slot >= x->slots || !x->connected) return YL_ERR_ARG;
    if (((uintptr_t)rows) % 16 != 0) return YL_ERR_ARG;
    // without a multicast mapping x->MC is all null and the kernel stores to every peer's window
    k_xchg_push_bulk<<<x->push_ctas, 32, XB_SMEM, (cudaStream_t)stream>>>(x->P, x->MC, x->rank, x->world, x->B, x->cap_out, x->slots, slot,
                                                                          rows, counts, (unsigned *)(x->window + x->L.off_done),
                                                                          (int *)(x->window + x->L.off_status), x->limit_ns);
    YL_LAUNCH_CHECK();
    return YL_OK;
}

extern "C" int yl_xchg_wait(yl_xchg *x, int slot, yl_stream_t stream)
{
    if (!x || slot < 0 || slot >= x->slots || !x->connected) return YL_ERR_ARG;
    k_xchg_wait<<<1, 32, 0, (cudaStream_t)stream>>>(x->P, x->rank, x->world, slot, (int *)(x->window + x->L.off_status), x->limit_ns);
    YL_LAUNCH_CHECK();
    return YL_OK;
}

extern "C" int yl_xchg_release(yl_xchg *x, int slot, yl_stream_t stream)
{
    if (!x || slot < 0 || slot >= x->slots || !x->connected) return YL_ERR_ARG;
    k_xchg_release<<<1, 32, 0, (cudaStream_t)stream>>>(x->P, x->rank, x->world, slot);
    YL_LAUNCH_CHECK();
    return YL_OK;
}

extern "C" void *yl_xchg_rows(yl_xchg *x, int slot)
{
    if (!x || slot < 0 || slot >= x->slots) return nullptr;
    return x->window + x->L.off_rows + sizeof(float) * 7 * (size_t)slot * x->world * x->B * x->cap_out;
}

extern "C" void *yl_xchg_counts(yl_xchg *x, int slot)
{
    if (!x || slot < 0 || slot >= x->slots) return nullptr;
    return x->window + x->L.off_counts + sizeof(int) * (size_t)slot * x->world * x->B;
}

extern "C" void *yl_xchg_status(yl_xchg *x)
{
    return x ? (void *)(x->window + x->L.off_status) : nullptr;
}

// Shared plumbing for libqck.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/qck.h"

#define QCK_SIDE_STREAMS 8

struct qck_handle {
    int device;
    int sm_count;
    int max_smem_optin;
    int64_t launches;
    char err[512];
    // small device scratch for reductions (per-CTA partials); the last 8 doubles are reserved for the
    // streaming simulator (instance label) and never handed out by qck_ensure_partials
    double* d_partials;
    size_t partials_count;
    // pinned host scratch for scalar read-backs
    double* h_pinned;
    // growable device scratch (contraction weights, split-K partials)
    void* scratch;
    size_t scratch_bytes;
    // side streams for fanning out independent small launches (created lazily)
    cudaStream_t side[QCK_SIDE_STREAMS];
    cudaEvent_t side_done[QCK_SIDE_STREAMS];
    cudaEvent_t fork;
    int side_ready;
    int region;            // a qck_sim_region is open: batch calls fan out and do not join
    unsigned region_used;  // side streams the open region has launched on
    unsigned region_forked;  // side streams that already wait for the CURRENT call's fork point
    unsigned side_next;    // rotating pick of the next side stream
    // workspace of nearest_probability_distribution (npd.cu): state, bins, per-CTA partials
    void* npd_ws;
    // register-resident simulator (sim_warp_kernel.inc): branch stash (grows only) and CTAs per SM per variant
    // (one buffer per call slot: the calls of one qck_sim_region overlap on the device and must not share it)
    void* warp_stash[QCK_SIDE_STREAMS];
    size_t warp_stash_bytes[QCK_SIDE_STREAMS];
    size_t warp_cnt_bytes[QCK_SIDE_STREAMS];  // leading bytes that hold arrival counters (zero between launches)
    unsigned region_calls;                     // batch calls made inside the open region
    int warp_occ[6];
    int tree_occ[6];
    // knit_outer: work counters [1024] + arrival ticket (zeroed once; the last CTA of a launch resets them)
    unsigned long long* knit_ctr;
};

#define QCK_FAIL(h, code, ...)                                    \
    do {                                                          \
        if (h) snprintf((h)->err, sizeof((h)->err), __VA_ARGS__); \
        return (code);                                            \
    } while (0)

#define QCK_CUDA(h, expr)                                                                 \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess)                                                            \
            QCK_FAIL(h, QCK_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                     __FILE__, __LINE__);                                                 \
    } while (0)

#define QCK_CHECK_LAUNCH(h)                                                                   \
    do {                                                                                      \
        cudaError_t _e = cudaGetLastError();                                                  \
        if (_e != cudaSuccess)                                                                \
            QCK_FAIL(h, QCK_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), \
                     __FILE__, __LINE__);                                                     \
        (h)->launches++;                                                                      \
    } while (0)

// Allow a kernel to use all opt-in shared memory that its static allocation leaves free.
template <typename K>
static inline cudaError_t qck_allow_max_smem(K kernel, int optin) {
    cudaFuncAttributes attr;
    cudaError_t e = cudaFuncGetAttributes(&attr, kernel);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)attr.sharedSizeBytes);
}

struct DeviceGuard {
    int prev;
    bool changed;
    explicit DeviceGuard(int dev) : prev(-1), changed(false) {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) {
            cudaSetDevice(dev);
            changed = true;
        }
    }
    ~DeviceGuard() {
        if (changed) cudaSetDevice(prev);
    }
};

// ---- bit helpers -----------------------------------------------------------------------
// insert a zero bit at position q:  ...hhh lll -> ...hhh 0 lll
__host__ __device__ __forceinline__ uint32_t insert_zero(uint32_t p, int q) {
    uint32_t lo = p & ((1u << q) - 1u);
    return ((p >> q) << (q + 1)) | lo;
}
__host__ __device__ __forceinline__ uint64_t insert_zero64(uint64_t p, int q) {
    uint64_t lo = p & ((1ull << q) - 1ull);
    return ((p >> q) << (q + 1)) | lo;
}

// generic software pext / pdep (no hardware instruction on NVIDIA GPUs)
__host__ __device__ __forceinline__ uint64_t soft_pext(uint64_t y, uint64_t mask) {
    uint64_t out = 0;
    int j = 0;
    while (mask) {
        uint64_t low = mask & (~mask + 1);  // lowest set bit
        if (y & low) out |= (1ull << j);
        ++j;
        mask ^= low;
    }
    return out;
}
__host__ __device__ __forceinline__ uint64_t soft_pdep(uint64_t x, uint64_t mask) {
    uint64_t out = 0;
    int j = 0;
    while (mask) {
        uint64_t low = mask & (~mask + 1);
        if ((x >> j) & 1ull) out |= low;
        ++j;
        mask ^= low;
    }
    return out;
}

// ---- block reductions ------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ---- cross-rank exchange of a qck_stats through peer mailboxes (reduce.cu: stats_exchange_kernel; knit.cu: the
// tail of knit_outer).  Every rank writes its four doubles straight into a slot of every peer's mailbox (NVLink
// stores into cudaIpc-mapped memory), publishes a sequence number, waits until its own mailbox holds the current
// sequence number from every rank and adds the slots in rank order (the same bits on every rank).  Slots are
// double buffered by the parity of the sequence number.
struct StatsSlot {
    double sum, min, sum_sqrt, nnz;
    unsigned long long seq;
    unsigned long long pad[3];
};
struct ExchangeParams {
    StatsSlot* box[QCK_MAX_RANKS];  // mailbox of every rank: [2][world] slots
    int rank, world;
};
// one full warp; `stats` holds this rank's values on entry and the combined ones on return (lane 0 writes)
__device__ __forceinline__ void stats_exchange_warp(const ExchangeParams& P, qck_stats* stats, unsigned long long* seq_counter) {
    const int lane = threadIdx.x & 31;
    unsigned long long seq = 0;
    if (lane == 0) seq = *seq_counter + 1ull;
    seq = __shfl_sync(0xffffffffu, seq, 0);
    const int buf = (int)(seq & 1ull);
    if (lane < P.world) {  // my values into slot [rank] of rank `lane`'s mailbox, the sequence number last
        volatile StatsSlot* dst = P.box[lane] + buf * P.world + P.rank;
        dst->sum = stats->sum;
        dst->min = stats->min;
        dst->sum_sqrt = stats->sum_sqrt;
        dst->nnz = stats->nnz;
        __threadfence_system();
        dst->seq = seq;
    }
    double s = 0.0, m = INFINITY, q = 0.0, z = 0.0;
    bool tracked = true;
    if (lane < P.world) {  // wait for rank `lane`'s values in my own mailbox
        volatile StatsSlot* src = P.box[P.rank] + buf * P.world + lane;
        const long long t0 = clock64();
        while (src->seq != seq) {
            if (clock64() - t0 > 8000000000ll) {  // ~4 s: a peer never came
                printf("qck: stats exchange: rank %d waited in vain for rank %d (sequence %llu)\n", P.rank, lane, seq);
                __trap();
            }
        }
        __threadfence_system();
        s = src->sum;
        m = src->min;
        q = src->sum_sqrt;
        z = src->nnz;
        tracked = !(z < 0.0);
    }
    // rank order, one lane after the other: identical bits on every rank
    double ss = 0.0, mm = INFINITY, qq = 0.0, zz = 0.0;
    bool all_tracked = true;
    for (int r = 0; r < P.world; ++r) {
        ss += __shfl_sync(0xffffffffu, s, r);
        mm = fmin(mm, __shfl_sync(0xffffffffu, m, r));
        qq += __shfl_sync(0xffffffffu, q, r);
        zz += __shfl_sync(0xffffffffu, z, r);
        all_tracked = all_tracked && __shfl_sync(0xffffffffu, (int)tracked, r);
    }
    if (lane == 0) {
        stats->sum = ss;
        stats->min = mm;
        stats->sum_sqrt = qq;
        stats->nnz = all_tracked ? zz : -1.0;
        *seq_counter = seq;
    }
}

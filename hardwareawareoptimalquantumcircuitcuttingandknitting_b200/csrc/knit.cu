// Knitting kernels (sm_100a): exact closed form of VirtualCircuit.knit
// (third_party/qvm/qvm/virtual_circuit.py:50-68,150-171,216-228 + virtual_gates.py knit rules).
//
//   knit_outer    K = 0:  out[y] = prod_f T_f[pext(y, mask_f)]             (HBM-write bound)
//   knit_contract K >= 1: out[y] = sum_l w(l) prod_f Q_f[l_f][pext(y, mask_f)]  (FP64 FMA bound)
//
// knit_outer is a pure streaming-store kernel.  The output index is split into a chunk
// (low c = 12 bits, 32 KiB of output) and a chunk number.  Within a chunk the table index
// of every fragment is (row chosen by the high bits) + (offset given by the low bits): the
// offsets are per-thread loop invariants kept in registers, the rows are staged in shared
// memory and reloaded only when they change.  Chunks are enumerated so that the bits of
// fragments with small rows vary fastest, which makes row reloads rare (for syc-32 the
// 18-qubit fragment's row changes every 16384 chunks).  Warp 0 prepares the next chunk's
// descriptor (address, row numbers, scalar factors) while the CTA streams the current one.
#include "qck_common.cuh"

#include <stdlib.h>

#define KO_MAXF 8
#define KO_MAXV 4         // fragments that own bits inside a chunk ("vector" fragments)
#define KO_CHUNK_BITS 12  // 4096 doubles = 32 KiB of output per chunk
#define KO_THREADS 256
#define KO_ITEMS ((1 << KO_CHUNK_BITS) / (4 * KO_THREADS))  // 256-bit stores per thread per chunk
#define KO_BATCH 8        // chunks per work item (one atomic fetch + one barrier per batch)

struct OuterParams {
    int n_frag, n_vec;
    const double* table[KO_MAXF];
    unsigned long long hi_mask[KO_MAXF];  // mask >> c
    unsigned int lo_mask[KO_MAXF];        // mask & (2^c - 1)
    int nlo[KO_MAXF];
    int row_off[KO_MAXF];
    int n_free;
    int order[32];
    unsigned long long y_hi_base;
    unsigned long long n_chunks;
    unsigned long long y_begin;
    double* out;
    double* partials;
    unsigned long long* work_counter;  // [n_rows] counters: zero when the launch starts, reset by its last CTA
    unsigned long long* ticket;        // arrival counter of the CTAs (same protocol)
    qck_stats* stats;                  // the last CTA reduces the partials into it (fixed order) ...
    int exchange;                      // ... and, on a sharded result, exchanges it with the peers (xp, seq_counter)
    ExchangeParams xp;
    unsigned long long* seq_counter;
    int n_fast;                         // low bits of the chunk number that do not change any row
    int n_rows;                         // 2^(n_free - n_fast)
    unsigned long long batches_per_row;
};

struct ChunkDesc {
    unsigned long long y_hi;
    unsigned int hi[KO_MAXV];
    double scal;  // product of the scalar fragments, multiplied in fragment order
};

__device__ __forceinline__ void st_stream4(double* p, double a, double b, double c, double d) {
    asm volatile("st.global.cs.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d)
                 : "memory");
}

// one lane prepares one descriptor
__device__ __forceinline__ void make_desc(const OuterParams& P, unsigned long long g, ChunkDesc* d) {
    unsigned long long y_hi = P.y_hi_base;
    for (int j = 0; j < P.n_free; ++j) y_hi |= ((g >> j) & 1ull) << P.order[j];
    double prod = 1.0;
    for (int f = 0; f < P.n_frag; ++f) {
        const unsigned int hi = (unsigned int)soft_pext(y_hi, P.hi_mask[f]);
        if (f < P.n_vec)
            d->hi[f] = hi;
        else
            prod *= __ldg(P.table[f] + hi);
    }
    d->y_hi = y_hi;
    d->scal = prod;
}

// The LAST CTA of a knit_outer launch finishes the call (round 2: this was a separate one-warp launch, a memset node
// in front of the kernel and, on a sharded result, the exchange launch - three dependent graph nodes of a 0.68 ms
// step at 8 GPUs).  It resets the work counters and the ticket for the next launch, reduces the per-CTA partials
// in the fixed order of finalize_stats_kernel (same bits) and runs the peer exchange.  Not inlined: its registers
// (spin loop, printf) must not weigh on the streaming loop.
__device__ __noinline__ void knit_outer_tail(const OuterParams& P) {
    const int tid = threadIdx.x;
    __shared__ int is_last;
    if (tid == 0) {
        __threadfence();
        const unsigned long long t = atomicAdd(P.ticket, 1ull);
        is_last = t == (unsigned long long)gridDim.x - 1ull;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    for (int i = tid; i < P.n_rows; i += KO_THREADS) P.work_counter[i] = 0ull;
    if (tid == 0) *P.ticket = 0ull;
    if (tid < 32 && P.stats && P.partials) {
        double s = 0.0, m = INFINITY, z = 0.0, zmin = 0.0;
        for (int i = tid; i < (int)gridDim.x; i += 32) {
            s += __ldcg(P.partials + 3 * i + 0);
            m = fmin(m, __ldcg(P.partials + 3 * i + 1));
            z += __ldcg(P.partials + 3 * i + 2);
            zmin = fmin(zmin, __ldcg(P.partials + 3 * i + 2));
        }
        s = warp_sum(s);
        m = warp_min(m);
        z = warp_sum(z);
        zmin = warp_min(zmin);
        if (tid == 0) {
            P.stats->sum = s;
            P.stats->min = m;
            P.stats->sum_sqrt = 0.0;
            P.stats->nnz = zmin < 0.0 ? -1.0 : z;
        }
        __syncwarp();
        if (P.exchange) stats_exchange_warp(P.xp, P.stats, P.seq_counter);
    }
}

// Streaming outer product.  Per chunk and thread the inner loop is 16 multiplies and four
// 256-bit streaming stores - the per-thread products of the vector fragments (pv) are
// loop-invariant registers, recomputed only when a vector fragment's row changes.
template <int FV, bool WRITE>
__global__ void __launch_bounds__(KO_THREADS) knit_outer_kernel(const __grid_constant__ OuterParams P) {
    extern __shared__ __align__(16) double rows[];
    __shared__ ChunkDesc desc[2][KO_BATCH];
    const int tid = threadIdx.x;
    double pv[KO_ITEMS][4];
#pragma unroll
    for (int e = 0; e < KO_ITEMS; ++e)
#pragma unroll
        for (int j = 0; j < 4; ++j) pv[e][j] = 1.0;
    // statistics of this thread's invariant factors: out = pv * sc, and rounding is monotone, so
    // min_i fl(pv_i sc) = fl(min_i(pv_i) sc) for sc >= 0 (max for sc < 0) - exact; the running
    // sum uses fl(sum_i pv_i) * sc, within a few ulp of the sum of the rounded products
    double pv_sum = 4.0 * KO_ITEMS, pv_min = 1.0, pv_max = 1.0;
    unsigned int loaded[FV > 0 ? FV : 1];
#pragma unroll
    for (int f = 0; f < FV; ++f) loaded[f] = 0xffffffffu;

    // Work distribution is DYNAMIC: CTAs pull batches of KO_BATCH consecutive chunk numbers from
    // a global counter.  A static split leaves the kernel waiting for the slowest SMs and caps a
    // pure-store stream at ~6.3 TB/s on B200; pulling work reaches ~7.4 TB/s (tools/write_patterns.cu).
    // The chunk number is (row, column): the row bits select the rows of the vector fragments, the
    // column bits only scalar factors.  Each row has its own counter; a CTA stays on its row (no
    // reload) until it is exhausted, then steals from the following rows.
    // When its row is exhausted warp 0 LOOKS at the counters of the other rows, 32 at a time, and jumps to the first
    // one with work left: trying the rows one by one with the atomic itself is a chain of up to n_rows dependent
    // atomics on contended counters before a CTA can conclude that nothing is left (a 4 GiB slice back to back:
    // 0.619 -> 0.609 ms per launch).  Pulling sub-batches near the end of a row ("guided" pulls) was measured too: no
    // gain on any slice size.
    __shared__ unsigned long long s_batch[2];
    __shared__ int s_my_row;
    const unsigned long long DONE = ~0ull;
    if (tid == 0) s_my_row = (int)(blockIdx.x % (unsigned)P.n_rows);
    __syncwarp();
    auto next_batch = [&]() -> unsigned long long {  // all lanes of warp 0; the same result in every lane
        for (;;) {
            const int my_row = s_my_row;
            unsigned long long b = 0ull;
            if (tid == 0) b = atomicAdd(P.work_counter + my_row, 1ull);
            b = __shfl_sync(0xffffffffu, b, 0);
            if (b < P.batches_per_row) return ((unsigned long long)my_row << P.n_fast) + b * KO_BATCH;
            int found = -1;
            for (int base = 1; base < P.n_rows && found < 0; base += 32) {
                const int off = base + tid;
                int r = my_row + off;
                r = r >= P.n_rows ? r - P.n_rows : r;
                const bool has = off < P.n_rows && *(volatile unsigned long long*)(P.work_counter + r) < P.batches_per_row;
                const unsigned int m = __ballot_sync(0xffffffffu, has);
                if (m) {
                    found = my_row + base + (__ffs(m) - 1);
                    found = found >= P.n_rows ? found - P.n_rows : found;
                }
            }
            if (found < 0) return DONE;
            __syncwarp();
            if (tid == 0) s_my_row = found;
            __syncwarp();
        }
    };
    double sum = 0.0, mn = INFINITY;
    if (tid < 32) {
        const unsigned long long gb = next_batch();
        if (tid < KO_BATCH && gb != DONE && gb + tid < P.n_chunks) make_desc(P, gb + tid, &desc[0][tid]);
        if (tid == 0) s_batch[0] = gb;
    }
    __syncthreads();
    for (int buf = 0;; buf ^= 1) {
        const unsigned long long gb = s_batch[buf];
        if (gb == DONE) break;
        if (tid < 32) {  // fetch and describe the next batch while this one streams
            const unsigned long long gn = next_batch();
            if (tid < KO_BATCH && gn != DONE && gn + tid < P.n_chunks) make_desc(P, gn + tid, &desc[buf ^ 1][tid]);
            if (tid == 0) s_batch[buf ^ 1] = gn;
        }
        const unsigned long long row_end = ((gb >> P.n_fast) + 1ull) << P.n_fast;
        const int nb = (int)((row_end - gb) < KO_BATCH ? (row_end - gb) : KO_BATCH);
        for (int b = 0; b < nb; ++b) {
            const ChunkDesc& D = desc[buf][b];
            if (FV > 0) {
                bool reload = false;
#pragma unroll
                for (int f = 0; f < FV; ++f) reload |= (D.hi[f] != loaded[f]);
                if (reload) {  // uniform across the CTA; rare when the chunk order is good
                    __syncthreads();
#pragma unroll
                    for (int f = 0; f < FV; ++f) {
                        if (D.hi[f] != loaded[f]) {
                            const double* src = P.table[f] + ((unsigned long long)D.hi[f] << P.nlo[f]);
                            double* dst = rows + P.row_off[f];
                            for (int i = tid; i < (1 << P.nlo[f]); i += KO_THREADS) dst[i] = __ldg(src + i);
                            loaded[f] = D.hi[f];
                        }
                    }
                    __syncthreads();
                    // y_lo = (e << 10) | (tid << 2) | j, and pext splits over disjoint bit ranges: the tid part (the only
                    // one that needs a loop) once per fragment, the two-bit parts of j and e in closed form.  (A
                    // soft_pext per entry made a row change cost ~1 300 instructions per thread - several us each
                    // time a CTA moves to another row, which is what the CTAs do at the end of a launch.)
                    static_assert(KO_THREADS == 256 && KO_ITEMS == 4 && KO_CHUNK_BITS == 12, "y_lo = (e << 10) | (tid << 2) | j");
                    unsigned int tpart[FV > 0 ? FV : 1], mj[FV > 0 ? FV : 1], me[FV > 0 ? FV : 1], se[FV > 0 ? FV : 1];
#pragma unroll
                    for (int f = 0; f < FV; ++f) {
                        const unsigned int m = P.lo_mask[f];
                        mj[f] = m & 3u;
                        me[f] = (m >> 10) & 3u;
                        const unsigned int mt = (m >> 2) & 0xffu;
                        const int sj = __popc(mj[f]);
                        tpart[f] = (unsigned int)soft_pext((unsigned int)tid, mt) << sj;
                        se[f] = (unsigned int)(sj + __popc(mt));
                    }
                    auto pext2 = [](unsigned int x, unsigned int m) -> unsigned int {  // x, m < 4
                        return m == 3u ? x : (m == 1u ? (x & 1u) : (m == 2u ? (x >> 1) : 0u));
                    };
#pragma unroll
                    for (int e = 0; e < KO_ITEMS; ++e)
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            double v = rows[P.row_off[0] + (pext2(j, mj[0]) | tpart[0] | (pext2(e, me[0]) << se[0]))];
#pragma unroll
                            for (int f = 1; f < FV; ++f)
                                v *= rows[P.row_off[f] + (pext2(j, mj[f]) | tpart[f] | (pext2(e, me[f]) << se[f]))];
                            pv[e][j] = v;
                        }
                    pv_sum = 0.0;
                    pv_min = INFINITY;
                    pv_max = -INFINITY;
#pragma unroll
                    for (int e = 0; e < KO_ITEMS; ++e)
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            pv_sum += pv[e][j];
                            pv_min = pv[e][j] < pv_min ? pv[e][j] : pv_min;
                            pv_max = pv[e][j] > pv_max ? pv[e][j] : pv_max;
                        }
                }
            }
            const double sc = D.scal;
            double* dst = WRITE ? P.out + ((D.y_hi << KO_CHUNK_BITS) - P.y_begin) + 4 * tid : nullptr;
#pragma unroll
            for (int e = 0; e < KO_ITEMS; ++e) {
                const double v0 = pv[e][0] * sc, v1 = pv[e][1] * sc, v2 = pv[e][2] * sc, v3 = pv[e][3] * sc;
                if (WRITE) st_stream4(dst + 4 * e * KO_THREADS, v0, v1, v2, v3);
            }
            sum = fma(pv_sum, sc, sum);
            const double cand = (sc >= 0.0 ? pv_min : pv_max) * sc;
            mn = cand < mn ? cand : mn;
        }
        __syncthreads();
    }
    // deterministic CTA reduction -> partials[blockIdx][3]
    __shared__ double red[2][KO_THREADS / 32];
    sum = warp_sum(sum);
    mn = warp_min(mn);
    if ((tid & 31) == 0) {
        red[0][tid >> 5] = sum;
        red[1][tid >> 5] = mn;
    }
    __syncthreads();
    if (tid == 0 && P.partials) {
        double s = 0.0, m = INFINITY;
        for (int w = 0; w < KO_THREADS / 32; ++w) {
            s += red[0][w];
            m = fmin(m, red[1][w]);
        }
        P.partials[3 * blockIdx.x + 0] = s;
        P.partials[3 * blockIdx.x + 1] = m;
        P.partials[3 * blockIdx.x + 2] = -1.0;  // nnz is not tracked on the streaming path
    }
    knit_outer_tail(P);
}

// generic fallback: one thread per element (small or unaligned ranges, many vector fragments)
struct OuterSimpleParams {
    int n_frag;
    const double* table[KO_MAXF];
    unsigned long long mask[KO_MAXF];
    unsigned long long y_begin, y_end;
    double* out;
    double* partials;
};

__global__ void __launch_bounds__(256) knit_outer_simple_kernel(const __grid_constant__ OuterSimpleParams P) {
    double sum = 0.0, mn = INFINITY, nnz = 0.0;
    const unsigned long long n = P.y_end - P.y_begin;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long y = P.y_begin + i;
        double v = 1.0;
        for (int f = 0; f < P.n_frag; ++f) v *= __ldg(P.table[f] + soft_pext(y, P.mask[f]));
        if (P.out) P.out[i] = v;
        sum += v;
        mn = fmin(mn, v);
        nnz += (v != 0.0 ? 1.0 : 0.0);
    }
    __shared__ double red[3][8];
    sum = warp_sum(sum);
    mn = warp_min(mn);
    nnz = warp_sum(nnz);
    if ((threadIdx.x & 31) == 0) {
        red[0][threadIdx.x >> 5] = sum;
        red[1][threadIdx.x >> 5] = mn;
        red[2][threadIdx.x >> 5] = nnz;
    }
    __syncthreads();
    if (threadIdx.x == 0 && P.partials) {
        double s = 0.0, m = INFINITY, z = 0.0;
        for (int w = 0; w < 8; ++w) {
            s += red[0][w];
            m = fmin(m, red[1][w]);
            z += red[2][w];
        }
        P.partials[3 * blockIdx.x + 0] = s;
        P.partials[3 * blockIdx.x + 1] = m;
        P.partials[3 * blockIdx.x + 2] = z;
    }
}

__global__ void finalize_stats_kernel(const double* __restrict__ partials, int n, qck_stats* stats) {
    // one warp, fixed order -> bitwise reproducible
    double s = 0.0, m = INFINITY, z = 0.0, zmin = 0.0;
    for (int i = threadIdx.x; i < n; i += 32) {
        s += partials[3 * i + 0];
        m = fmin(m, partials[3 * i + 1]);
        z += partials[3 * i + 2];
        zmin = fmin(zmin, partials[3 * i + 2]);
    }
    s = warp_sum(s);
    m = warp_min(m);
    z = warp_sum(z);
    zmin = warp_min(zmin);
    if (threadIdx.x == 0) {
        stats->sum = s;
        stats->min = m;
        stats->sum_sqrt = 0.0;
        stats->nnz = zmin < 0.0 ? -1.0 : z;  // -1: not tracked (streaming path)
    }
}

int qck_ensure_partials(qck_handle* h, size_t count);  // api.cu

template <int FV, bool WRITE>
static cudaError_t launch_outer_one(int grid, size_t smem, cudaStream_t st, const OuterParams& P) {
    knit_outer_kernel<FV, WRITE><<<grid, KO_THREADS, smem, st>>>(P);
    return cudaSuccess;
}

template <int FV>
static cudaError_t outer_attr(int limit) {
    cudaError_t e = qck_allow_max_smem(knit_outer_kernel<FV, true>, limit);
    if (e != cudaSuccess) return e;
    return qck_allow_max_smem(knit_outer_kernel<FV, false>, limit);
}

// see qck_sim_init: opt-in shared-memory limits are set once per process, not per launch
int qck_knit_init(qck_handle* h) {
    QCK_CUDA(h, outer_attr<0>(h->max_smem_optin));
    QCK_CUDA(h, outer_attr<1>(h->max_smem_optin));
    QCK_CUDA(h, outer_attr<2>(h->max_smem_optin));
    QCK_CUDA(h, outer_attr<3>(h->max_smem_optin));
    QCK_CUDA(h, outer_attr<4>(h->max_smem_optin));
    return QCK_OK;
}

template <bool WRITE>
static cudaError_t launch_outer(int n_vec, int grid, size_t smem, cudaStream_t st, const OuterParams& P) {
    switch (n_vec) {
        case 0: return launch_outer_one<0, WRITE>(grid, smem, st, P);
        case 1: return launch_outer_one<1, WRITE>(grid, smem, st, P);
        case 2: return launch_outer_one<2, WRITE>(grid, smem, st, P);
        case 3: return launch_outer_one<3, WRITE>(grid, smem, st, P);
        default: return launch_outer_one<4, WRITE>(grid, smem, st, P);
    }
}

extern "C" int qck_knit_outer(qck_handle* h, int n_frag, const double* const* d_tables, const uint64_t* masks,
                              int n_out_bits, uint64_t y_begin, uint64_t y_end, double* d_out, qck_stats* d_stats,
                              qck_stream stream) {
    return qck_knit_outer_exchange(h, n_frag, d_tables, masks, n_out_bits, y_begin, y_end, d_out, d_stats, 0, 1, nullptr,
                                   stream);
}

extern "C" int qck_knit_outer_exchange(qck_handle* h, int n_frag, const double* const* d_tables, const uint64_t* masks,
                                       int n_out_bits, uint64_t y_begin, uint64_t y_end, double* d_out,
                                       qck_stats* d_stats, int rank, int world, void* const* d_mailboxes,
                                       qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    const bool exchange = world > 1;
    if (exchange && (!d_stats || !d_mailboxes || world > QCK_MAX_RANKS || rank < 0 || rank >= world))
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "bad stats exchange arguments");
    if (n_frag < 1 || n_frag > KO_MAXF) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_frag=%d out of range [1,%d]", n_frag, KO_MAXF);
    if (!d_tables || !masks) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "tables / masks NULL");
    if (n_out_bits < 0 || n_out_bits > QCK_MAX_OUT_BITS) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_out_bits=%d", n_out_bits);
    const uint64_t full = n_out_bits >= 64 ? ~0ull : ((1ull << n_out_bits) - 1ull);
    for (int f = 0; f < n_frag; ++f) {
        if (!d_tables[f]) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "table %d is NULL", f);
        if (masks[f] & ~full) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "mask %d has bits >= n_out_bits", f);
    }
    if (y_end < y_begin || y_end > (1ull << n_out_bits)) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "bad output range");
    if ((y_end == y_begin || (!d_out && !d_stats)) && !exchange) return QCK_OK;
    if (y_end == y_begin) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "an exchange needs a non-empty slice on every rank");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;

    const uint64_t span = y_end - y_begin;
    const bool pow2_block = (span & (span - 1)) == 0 && (y_begin % span) == 0;
    int n_vec = 0;
    for (int f = 0; f < n_frag; ++f)
        if (masks[f] & ((1ull << KO_CHUNK_BITS) - 1ull)) ++n_vec;
    int r = 0;
    while ((1ull << r) < span) ++r;
    const bool fast = pow2_block && r >= KO_CHUNK_BITS && n_vec <= KO_MAXV && (n_out_bits - KO_CHUNK_BITS) <= 32 &&
                      (d_out == nullptr || (reinterpret_cast<uintptr_t>(d_out) % 32) == 0);
    int grid;
    if (fast) {
        OuterParams P;
        memset(&P, 0, sizeof(P));
        // vector fragments first (largest row first), then scalars
        int order_f[KO_MAXF], nf = 0;
        for (int pass = 0; pass < 2; ++pass)
            for (int f = 0; f < n_frag; ++f) {
                bool vec = (masks[f] & ((1ull << KO_CHUNK_BITS) - 1ull)) != 0;
                if (vec == (pass == 0)) order_f[nf++] = f;
            }
        P.n_frag = n_frag;
        P.n_vec = n_vec;
        int off = 0;
        for (int i = 0; i < n_frag; ++i) {
            int f = order_f[i];
            P.table[i] = d_tables[f];
            P.hi_mask[i] = masks[f] >> KO_CHUNK_BITS;
            P.lo_mask[i] = (unsigned int)(masks[f] & ((1ull << KO_CHUNK_BITS) - 1ull));
            P.nlo[i] = __builtin_popcount(P.lo_mask[i]);
            P.row_off[i] = off;
            if (i < n_vec) off += (1 << P.nlo[i]);
        }
        // free high bits, fastest first: bits owned by fragments with the smallest rows
        const int n_free = r - KO_CHUNK_BITS;
        int weight[64];
        for (int b = 0; b < n_free; ++b) {
            int w = 0;  // largest row among the fragments that own this bit
            for (int i = 0; i < n_frag; ++i)
                if ((P.hi_mask[i] >> b) & 1ull) w = w > P.nlo[i] ? w : P.nlo[i];
            weight[b] = w;
        }
        int cnt = 0;
        for (int w = 0; w <= KO_CHUNK_BITS; ++w)
            for (int b = 0; b < n_free; ++b)
                if (weight[b] == w) P.order[cnt++] = b;
        P.n_free = n_free;
        P.y_hi_base = y_begin >> KO_CHUNK_BITS;
        P.n_chunks = span >> KO_CHUNK_BITS;
        P.y_begin = y_begin;
        P.out = d_out;
        size_t smem = (size_t)off * sizeof(double);
        if ((int)smem + 4096 > h->max_smem_optin)
            QCK_FAIL(h, QCK_ERR_UNSUPPORTED, "knit_outer: fragment rows (%zu bytes) do not fit shared memory", smem);
        int per_sm = 2;  // resident CTAs per SM; QCK_KO_CTAS_PER_SM overrides (tuning knob)
        if (const char* env = getenv("QCK_KO_CTAS_PER_SM")) {
            int v = atoi(env);
            if (v >= 1 && v <= 8) per_sm = v;
        }
        grid = h->sm_count * per_sm;
        if ((unsigned long long)grid > P.n_chunks) grid = (int)P.n_chunks;
        // rows = values of the free bits owned by vector fragments (they come last in `order`)
        int n_fast = 0;
        while (n_fast < n_free && weight[P.order[n_fast]] == 0) ++n_fast;
        int lg_batch = 0;
        while ((1 << lg_batch) < KO_BATCH) ++lg_batch;
        if (n_fast < lg_batch) n_fast = n_free < lg_batch ? n_free : lg_batch;   // rows of >= 1 batch
        if (n_free - n_fast > 10) n_fast = n_free - 10;                          // at most 1024 counters
        P.n_fast = n_fast;
        P.n_rows = 1 << (n_free - n_fast);
        P.batches_per_row = ((1ull << n_fast) + KO_BATCH - 1) / KO_BATCH;
        int rc = qck_ensure_partials(h, (size_t)grid * 3);
        if (rc) return rc;
        if (P.n_rows > 1024) QCK_FAIL(h, QCK_ERR_UNSUPPORTED, "knit_outer: %d work rows", P.n_rows);
        P.partials = d_stats ? h->d_partials : nullptr;
        P.work_counter = h->knit_ctr;          // zero between launches (the last CTA of a launch resets them)
        P.ticket = h->knit_ctr + 1024;
        P.stats = d_stats;
        P.exchange = exchange ? 1 : 0;
        if (exchange) {
            for (int r2 = 0; r2 < world; ++r2) {
                if (!d_mailboxes[r2]) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "mailbox of rank %d is NULL", r2);
                P.xp.box[r2] = reinterpret_cast<StatsSlot*>(reinterpret_cast<char*>(d_mailboxes[r2]) + 64);
            }
            P.xp.rank = rank;
            P.xp.world = world;
            P.seq_counter = reinterpret_cast<unsigned long long*>(d_mailboxes[rank]);
        }
        QCK_CUDA(h, d_out ? launch_outer<true>(n_vec, grid, smem, st, P) : launch_outer<false>(n_vec, grid, smem, st, P));
        QCK_CHECK_LAUNCH(h);
        return QCK_OK;
    } else {
        OuterSimpleParams P;
        memset(&P, 0, sizeof(P));
        P.n_frag = n_frag;
        for (int f = 0; f < n_frag; ++f) {
            P.table[f] = d_tables[f];
            P.mask[f] = masks[f];
        }
        P.y_begin = y_begin;
        P.y_end = y_end;
        P.out = d_out;
        unsigned long long want = (span + 255) / 256;
        grid = (int)(want < (unsigned long long)h->sm_count * 8 ? want : (unsigned long long)h->sm_count * 8);
        int rc = qck_ensure_partials(h, (size_t)grid * 3);
        if (rc) return rc;
        P.partials = d_stats ? h->d_partials : nullptr;
        knit_outer_simple_kernel<<<grid, 256, 0, st>>>(P);
        QCK_CHECK_LAUNCH(h);
    }
    if (d_stats) {
        finalize_stats_kernel<<<1, 32, 0, st>>>(h->d_partials, grid, d_stats);
        QCK_CHECK_LAUNCH(h);
    }
    if (exchange) return qck_stats_exchange(h, d_stats, rank, world, d_mailboxes, stream);
    return QCK_OK;
}

// ====================================================================== knit_contract
// prep: w[l] = prod_k coef[k][digit_k(l)], rows[f][l] = sum_k digit_k(l) * frag_stride[f][k]
struct PrepParams {
    int n_digits, n_frag;
    int radix[QCK_MAX_DIGITS];
    double coef[QCK_MAX_DIGITS][QCK_MAX_VARIANTS];
    int stride[KO_MAXF][QCK_MAX_DIGITS];
    long long l_begin, count;
    double* w;
    int* rows;  // [n_frag][count]
};

__global__ void contract_prep_kernel(const __grid_constant__ PrepParams P) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < P.count;
         i += (long long)gridDim.x * blockDim.x) {
        long long rem = P.l_begin + i;
        double w = 1.0;
        int rows[KO_MAXF];
#pragma unroll
        for (int f = 0; f < KO_MAXF; ++f) rows[f] = 0;
        // digits from the last (fastest) to the first; the weight is multiplied in the order
        // k = 0..K-1 on the host reference, the product of <= 16 doubles differs by O(1e-16)
        int digit[QCK_MAX_DIGITS];
        for (int k = P.n_digits - 1; k >= 0; --k) {
            digit[k] = (int)(rem % P.radix[k]);
            rem /= P.radix[k];
        }
        for (int k = 0; k < P.n_digits; ++k) {
            w *= P.coef[k][digit[k]];
#pragma unroll
            for (int f = 0; f < KO_MAXF; ++f)
                if (f < P.n_frag) rows[f] += digit[k] * P.stride[f][k];
        }
        P.w[i] = w;
        for (int f = 0; f < P.n_frag; ++f) P.rows[(long long)f * P.count + i] = rows[f];
    }
}

struct ContractParams {
    int n_frag;
    const double* table[KO_MAXF];
    unsigned long long mask[KO_MAXF];
    long long row_stride[KO_MAXF];
    int n_out_bits;
    long long count;  // labels
    const double* w;
    const int* rows;
    double* out;
    int accumulate;
};

// generic: one thread per output entry, loops over the labels
__global__ void __launch_bounds__(256) contract_generic_kernel(const __grid_constant__ ContractParams P) {
    const unsigned long long n = 1ull << P.n_out_bits;
    for (unsigned long long y = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; y < n;
         y += (unsigned long long)gridDim.x * blockDim.x) {
        const double* base[KO_MAXF];
        for (int f = 0; f < P.n_frag; ++f) base[f] = P.table[f] + soft_pext(y, P.mask[f]);
        double acc = 0.0;
        for (long long l = 0; l < P.count; ++l) {
            double t = __ldg(P.w + l);
            for (int f = 0; f < P.n_frag; ++f)
                t *= __ldg(base[f] + (long long)__ldg(P.rows + (long long)f * P.count + l) * P.row_stride[f]);
            acc += t;
        }
        P.out[y] = P.accumulate ? P.out[y] + acc : acc;
    }
}

// two fragments: C[i][j] = sum_l w[l] A[rowA[l]][i] B[rowB[l]][j]  (64x64 tile, split over l)
#define GT 64
#define GK 16
// on FP64 tensor cores (sm_100a: mma.sync.aligned.m8n8k4.f64 = DMMA; tcgen05 has no FP64 kind).
// 64x64 output tile per CTA, 8 warps, each warp owns a 32x16 sub-tile = 4x2 DMMA tiles (16 accumulator
// registers).  Per k-step of 4 labels a warp issues 8 DMMAs (2048 FMA) against 6 LDS.64 per thread:
// 0.75 B of shared-memory traffic per FMA instead of 4 B on an FMA-pipe tile, which was measured
// shared-memory bound and removed.  As/Bs rows are padded to 72 doubles so that a fragment load (lanes
// vary the row by lane>>2 and k by lane&3) needs exactly two 128-byte wavefronts.
#define GP 72
__device__ __forceinline__ void dmma_m8n8k4(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(256) contract_dmma_kernel(const __grid_constant__ ContractParams P, int n_split,
                                                            double* __restrict__ partial, int M, int N, int Mr,
                                                            int Nr) {
    __shared__ double As[GK][GP];
    __shared__ double Bs[GK][GP];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wi = (warp >> 2) * 32, wj = (warp & 3) * 16;  // warp sub-tile origin inside the CTA tile
    const int gid = lane >> 2, tig = lane & 3;
    const int i0 = blockIdx.x * GT, j0 = blockIdx.y * GT;
    const long long per = (P.count + n_split - 1) / n_split;
    const long long lb = per * blockIdx.z, le = (lb + per < P.count) ? lb + per : P.count;
    const int* rowA = P.rows;
    const int* rowB = P.rows + P.count;
    double acc[4][2][2];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 2; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;
    for (long long l0 = lb; l0 < le; l0 += GK) {
#pragma unroll
        for (int k = 0; k < (GK * GT) / 256; ++k) {
            const int e = tid + 256 * k, rr = e / GT, cc = e % GT;
            const long long l = l0 + rr;
            double a = 0.0, b = 0.0;
            if (l < le) {  // Mr / Nr: real row lengths (a fragment with fewer than 6 output bits fills part of a tile)
                if (i0 + cc < Mr)
                    a = __ldg(P.w + l) * __ldg(P.table[0] + (long long)__ldg(rowA + l) * P.row_stride[0] + i0 + cc);
                if (j0 + cc < Nr) b = __ldg(P.table[1] + (long long)__ldg(rowB + l) * P.row_stride[1] + j0 + cc);
            }
            As[rr][cc] = a;
            Bs[rr][cc] = b;
        }
        __syncthreads();
#pragma unroll
        for (int k4 = 0; k4 < GK; k4 += 4) {
            double af[4], bf[2];
#pragma unroll
            for (int a = 0; a < 4; ++a) af[a] = As[k4 + tig][wi + 8 * a + gid];  // A[m = gid][k = tig]
#pragma unroll
            for (int b = 0; b < 2; ++b) bf[b] = Bs[k4 + tig][wj + 8 * b + gid];  // B[k = tig][n = gid]
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 2; ++b) dmma_m8n8k4(acc[a][b][0], acc[a][b][1], af[a], bf[b]);
        }
        __syncthreads();
    }
    // C fragment: thread holds C[gid][2 * tig + {0, 1}] of every 8x8 tile
    double* dst = partial + (long long)blockIdx.z * M * N;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 2; ++b) {
            const long long r = i0 + wi + 8 * a + gid, c = j0 + wj + 8 * b + 2 * tig;
            dst[r * N + c] = acc[a][b][0];
            dst[r * N + c + 1] = acc[a][b][1];
        }
}

// The same contraction with the gather PIPELINED (ncu, round 1: the kernel above keeps the DMMA pipe 32 % busy -
// gather -> barrier -> multiply -> barrier per 16 labels, and the weight multiplication sits in the gather).
// Here the table rows of the next two label chunks are in flight (cp.async.cg, 16 bytes per request, zero-fill
// for padding) while the tensor cores work on the current one; the label weights are applied to the A fragments
// as they leave shared memory, so both operands are plain copies.  Three stages of [16 labels][64 + 8] doubles
// per operand = 54 KiB of dynamic shared memory.
// Tile size (round 2, second half): at 64x64 every 16-label chunk brings 16 KiB from L2 for 131 kflop - 8 flop per
// gathered byte, which makes the kernel an L2-gather kernel (ncu: DMMA 41 % of its peak on hwe-16 d5's 256x256
// output, 304 CTAs each re-reading a quarter of both tables).  TT = 128 halves the bytes per flop and quarters the
// barriers per flop: 16 warps of 32x32 (4x4 DMMA tiles, 8 LDS.64 for 16 DMMAs per k-step; the DMMA pipe 61 % busy
// on hwe-16 d5, against 59 % with 8 warps of 64x32, which were removed), one CTA per SM.  Used when both padded dimensions are multiples of 128 and there are at least 4096 labels.
#define GS 3
template <int TT>
struct ContractStage {
    double A[GK][TT + 8];
    double B[GK][TT + 8];
    double W[GK];
};
__device__ __forceinline__ void cp_async16_zfill(void* dst, const void* src, bool valid) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
    const int bytes = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(bytes) : "memory");
}

template <int TT, int NW>
__global__ void __launch_bounds__(32 * NW)
    contract_dmma_pipe_kernel(const __grid_constant__ ContractParams P, int n_split, double* __restrict__ partial, int M,
                              int N, int Mr, int Nr) {
    constexpr int WR = NW / 4;                              // warps: WR rows x 4 columns
    constexpr int NA = TT / WR / 8, NB = TT / 4 / 8;        // DMMA tiles per warp: rows (x 8), columns (x 8)
    constexpr int NT = 32 * NW;
    extern __shared__ __align__(16) unsigned char cps_raw[];
    ContractStage<TT>* stage = reinterpret_cast<ContractStage<TT>*>(cps_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wi = (warp >> 2) * (TT / WR), wj = (warp & 3) * (TT / 4);
    const int gid = lane >> 2, tig = lane & 3;
    const int i0 = blockIdx.x * TT, j0 = blockIdx.y * TT;
    const long long per = (P.count + n_split - 1) / n_split;
    const long long lb = per * blockIdx.z, le = (lb + per < P.count) ? lb + per : P.count;
    const int* rowA = P.rows;
    const int* rowB = P.rows + P.count;
    const long long n_chunks = le > lb ? (le - lb + GK - 1) / GK : 0;
    // this thread's share of a stage: requests of 16 bytes (2 doubles) - rows rr, columns cc..cc+1
    auto issue = [&](long long chunk) {
        ContractStage<TT>& S = stage[chunk % GS];
        const long long l0 = lb + chunk * GK;
#pragma unroll
        for (int k = 0; k < GK * (TT / 2) / NT; ++k) {
            const int e = tid + NT * k;            // GK * TT / 2 requests per operand
            const int rr = e / (TT / 2), cc = (e % (TT / 2)) * 2;
            const long long l = l0 + rr;
            const bool in = l < le;
            const long long ra = in ? (long long)__ldg(rowA + l) : 0, rb = in ? (long long)__ldg(rowB + l) : 0;
            cp_async16_zfill(&S.A[rr][cc], P.table[0] + ra * P.row_stride[0] + i0 + cc, in && (i0 + cc < Mr));
            cp_async16_zfill(&S.B[rr][cc], P.table[1] + rb * P.row_stride[1] + j0 + cc, in && (j0 + cc < Nr));
        }
        if (tid < GK) {
            const long long l = l0 + tid;
            S.W[tid] = l < le ? __ldg(P.w + l) : 0.0;
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    double acc[NA][NB][2];
#pragma unroll
    for (int a = 0; a < NA; ++a)
#pragma unroll
        for (int b = 0; b < NB; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;
    for (int c = 0; c < GS - 1; ++c) {
        if (c < n_chunks) issue(c);
        else asm volatile("cp.async.commit_group;" ::: "memory");
    }
    for (long long c = 0; c < n_chunks; ++c) {
        asm volatile("cp.async.wait_group %0;" ::"n"(GS - 2) : "memory");
        __syncthreads();  // chunk c has landed for everyone; everyone is done with chunk c - 1's buffer
        if (c + GS - 1 < n_chunks) issue(c + GS - 1);
        else asm volatile("cp.async.commit_group;" ::: "memory");
        const ContractStage<TT>& S = stage[c % GS];
#pragma unroll
        for (int k4 = 0; k4 < GK; k4 += 4) {
            const double w = S.W[k4 + tig];
            double af[NA], bf[NB];
#pragma unroll
            for (int a = 0; a < NA; ++a) af[a] = w * S.A[k4 + tig][wi + 8 * a + gid];
#pragma unroll
            for (int b = 0; b < NB; ++b) bf[b] = S.B[k4 + tig][wj + 8 * b + gid];
#pragma unroll
            for (int a = 0; a < NA; ++a)
#pragma unroll
                for (int b = 0; b < NB; ++b) dmma_m8n8k4(acc[a][b][0], acc[a][b][1], af[a], bf[b]);
        }
    }
    double* dst = partial + (long long)blockIdx.z * M * N;
#pragma unroll
    for (int a = 0; a < NA; ++a)
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            const long long r = i0 + wi + 8 * a + gid, cidx = j0 + wj + 8 * b + 2 * tig;
            dst[r * N + cidx] = acc[a][b][0];
            dst[r * N + cidx + 1] = acc[a][b][1];
        }
}

// Sum of the split partials (fixed order) -> out.  One thread per TILE entry: the partials are read in their own
// order (consecutive lanes, consecutive addresses; one thread per OUTPUT entry read 32 different rows per warp and
// split - 10 us for hwe-16 d5's 19 splits) and the 8-byte results go to their pdep positions.  The masks cover the
// output exactly (full_cover), so every output entry is written once; padded tile entries have none.
__global__ void __launch_bounds__(256) contract_scatter_kernel(const double* __restrict__ partial, int n_split, int M,
                                                               int N, int Mr, int Nr, unsigned long long maskA,
                                                               unsigned long long maskB, double* __restrict__ out,
                                                               int accumulate) {
    const long long total = (long long)M * N;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long i = idx / N, j = idx - i * N;
        if (i >= Mr || j >= Nr) continue;
        double acc = 0.0;
        for (int s = 0; s < n_split; ++s) acc += partial[(long long)s * total + idx];
        const unsigned long long y = soft_pdep((unsigned long long)i, maskA) | soft_pdep((unsigned long long)j, maskB);
        out[y] = accumulate ? out[y] + acc : acc;
    }
}

// Three and more fragments (virtual_circuit.py:139-163 handles any number; Cutter.py:40 maxNPartitions): the
// fragments are split into two GROUPS and the rows of a group with several members are multiplied out once per
// group label - merged[lg][c] = prod_{f in g} Q_f[row_f(lg)][pext(c, mask_f inside the group)] - so that the
// label contraction itself is the two-operand tensor-core tile kernel above (the per-output generic kernel walks
// all labels serially: 19.5 ms against 0.3 ms on 32 768 labels in round 1).
struct MergeParams {
    int n_frag, n_digits, m_bits;
    const double* table[KO_MAXF];
    long long row_stride[KO_MAXF];
    unsigned long long cmask[KO_MAXF];     // the fragment's output bits among the group's
    int stride[KO_MAXF][QCK_MAX_DIGITS];   // fragment label strides of the digits
    int radix[QCK_MAX_DIGITS];
    int touched[QCK_MAX_DIGITS];           // digit is part of the group label
    long long n_labels;
    double* out;                           // [n_labels][2^m_bits]
};

__global__ void __launch_bounds__(256) contract_merge_kernel(const __grid_constant__ MergeParams P) {
    __shared__ long long row[KO_MAXF];
    const long long cols = 1ll << P.m_bits;
    for (long long lg = blockIdx.x; lg < P.n_labels; lg += gridDim.x) {
        __syncthreads();
        if (threadIdx.x < P.n_frag) {
            long long rem = lg, r = 0;
            for (int k = P.n_digits - 1; k >= 0; --k) {
                if (!P.touched[k]) continue;
                r += (rem % P.radix[k]) * P.stride[threadIdx.x][k];
                rem /= P.radix[k];
            }
            row[threadIdx.x] = r * P.row_stride[threadIdx.x];
        }
        __syncthreads();
        for (long long c = threadIdx.x; c < cols; c += blockDim.x) {
            double v = 1.0;
            for (int f = 0; f < P.n_frag; ++f) v *= __ldg(P.table[f] + row[f] + soft_pext((unsigned long long)c, P.cmask[f]));
            P.out[lg * cols + c] = v;
        }
    }
}

static unsigned long long compress_mask(unsigned long long mask, unsigned long long within) {
    unsigned long long out = 0;
    int j = 0;
    for (int b = 0; b < 64; ++b)
        if ((within >> b) & 1ull) {
            if ((mask >> b) & 1ull) out |= 1ull << j;
            ++j;
        }
    return out;
}

int qck_ensure_scratch(qck_handle* h, size_t bytes, void** out);  // api.cu

// w[i] and rows[f][i] of the labels l_begin + i, i < count (also the label decode of qck_knit_terms, observe.cu)
int qck_contract_prep(qck_handle* h, int n_frag, int n_digits, const int32_t* radix, const double* coef,
                      const int32_t* frag_stride, long long l_begin, long long count, double* d_w, int* d_rows,
                      cudaStream_t st) {
    PrepParams pp;
    memset(&pp, 0, sizeof(pp));
    pp.n_digits = n_digits;
    pp.n_frag = n_frag;
    for (int k = 0; k < n_digits; ++k) {
        pp.radix[k] = radix[k];
        for (int v = 0; v < QCK_MAX_VARIANTS; ++v) pp.coef[k][v] = coef[k * QCK_MAX_VARIANTS + v];
        for (int f = 0; f < n_frag; ++f) pp.stride[f][k] = frag_stride[f * QCK_MAX_DIGITS + k];
    }
    pp.l_begin = l_begin;
    pp.count = count;
    pp.w = d_w;
    pp.rows = d_rows;
    int pgrid = (int)((count + 255) / 256 < 1024 ? (count + 255) / 256 : 1024);
    contract_prep_kernel<<<pgrid, 256, 0, st>>>(pp);
    QCK_CHECK_LAUNCH(h);
    return QCK_OK;
}

extern "C" int qck_knit_contract(qck_handle* h, int n_frag, const double* const* d_tables, const uint64_t* masks,
                                 const int64_t* row_strides, int n_out_bits, int n_digits, const int32_t* radix,
                                 const double* coef, const int32_t* frag_stride, int64_t l_begin, int64_t l_end,
                                 double* d_out, int accumulate, qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    if (n_frag < 1 || n_frag > KO_MAXF) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_frag=%d out of range", n_frag);
    if (n_digits < 0 || n_digits > QCK_MAX_DIGITS) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_digits=%d out of range", n_digits);
    if (!d_tables || !masks || !row_strides || !d_out || (n_digits > 0 && (!radix || !coef || !frag_stride)))
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "NULL argument");
    if (n_out_bits < 0 || n_out_bits > 34) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_out_bits=%d out of range", n_out_bits);
    long long total = 1;
    for (int k = 0; k < n_digits; ++k) {
        if (radix[k] < 1 || radix[k] > QCK_MAX_VARIANTS) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "radix[%d]=%d", k, radix[k]);
        total *= radix[k];
    }
    if (l_begin < 0 || l_end > total || l_end < l_begin) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "bad label range");
    uint64_t seen = 0;
    for (int f = 0; f < n_frag; ++f) {
        if (masks[f] & seen) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "fragment masks overlap");
        seen |= masks[f];
    }
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    const long long count = l_end - l_begin;
    if (count == 0) {
        if (!accumulate) QCK_CUDA(h, cudaMemsetAsync(d_out, 0, sizeof(double) << n_out_bits, st));
        return QCK_OK;
    }
    // ---- three and more fragments: two groups (see contract_merge_kernel)
    const bool full_cover = seen == (n_out_bits >= 64 ? ~0ull : (1ull << n_out_bits) - 1ull);
    const char* group_env = getenv("QCK_CONTRACT_GROUPS");
    const double* eff_tables[2];
    uint64_t eff_masks[2];
    int64_t eff_row_strides[2];
    int32_t eff_stride[2 * QCK_MAX_DIGITS];
    size_t merged_bytes[2] = {0, 0};
    long long group_labels[2] = {0, 0};
    int group_of_frag = 0;  // bit f set: fragment f belongs to group 1
    bool grouped = false;
    if (n_frag >= 3 && full_cover && !(group_env && atoi(group_env) == 0)) {
        double best = -1.0;
        for (int pick = 1; pick < (1 << (n_frag - 1)); ++pick) {  // fragment n_frag-1 always in group 0
            double cost = 0.0;
            int bits[2] = {0, 0};
            bool ok = true;
            for (int g = 0; g < 2; ++g) {
                int members = 0;
                long long lg = 1;
                for (int f = 0; f < n_frag; ++f)
                    if (((pick >> f) & 1) == g) {
                        ++members;
                        bits[g] += __builtin_popcountll(masks[f]);
                    }
                for (int k = 0; k < n_digits; ++k) {
                    bool touched = false;
                    for (int f = 0; f < n_frag; ++f)
                        if (((pick >> f) & 1) == g && frag_stride[f * QCK_MAX_DIGITS + k] != 0) touched = true;
                    if (touched) lg *= radix[k];
                    if (lg >= (1ll << 31)) ok = false;
                }
                if (members > 1) cost += 2.0 * (double)lg * (double)(1ull << bits[g]);
            }
            const int pa = bits[0] < 6 ? 6 : bits[0], pb = bits[1] < 6 ? 6 : bits[1];
            cost += (double)count * (double)(1ull << (pa + pb)) / 6.0;
            if (ok && (best < 0 || cost < best)) best = cost, group_of_frag = pick;
        }
        grouped = best >= 0;
        if (grouped) {
            for (int g = 0; g < 2 && grouped; ++g) {
                int members = 0, bits = 0, last = -1;
                uint64_t gmask = 0;
                long long acc = 1;
                for (int f = 0; f < n_frag; ++f)
                    if (((group_of_frag >> f) & 1) == g) ++members, bits += __builtin_popcountll(masks[f]), gmask |= masks[f], last = f;
                for (int k = n_digits - 1; k >= 0; --k) {
                    bool touched = false;
                    for (int f = 0; f < n_frag; ++f)
                        if (((group_of_frag >> f) & 1) == g && frag_stride[f * QCK_MAX_DIGITS + k] != 0) touched = true;
                    eff_stride[g * QCK_MAX_DIGITS + k] = touched ? (int32_t)acc : 0;
                    if (touched) acc *= radix[k];
                }
                eff_masks[g] = gmask;
                group_labels[g] = acc;
                if (members == 1) {
                    eff_tables[g] = d_tables[last];
                    eff_row_strides[g] = row_strides[last];
                    for (int k = 0; k < n_digits; ++k) eff_stride[g * QCK_MAX_DIGITS + k] = frag_stride[last * QCK_MAX_DIGITS + k];
                } else {
                    eff_tables[g] = nullptr;  // filled once the scratch is known
                    eff_row_strides[g] = 1ll << bits;
                    merged_bytes[g] = (((size_t)acc << bits) * sizeof(double) + 255) & ~(size_t)255;
                }
            }
            if (merged_bytes[0] + merged_bytes[1] > ((size_t)16 << 30)) grouped = false;  // fall back: generic kernel
        }
    }
    const int n_eff = grouped ? 2 : n_frag;
    const double* const* tabs = grouped ? eff_tables : d_tables;
    const uint64_t* msk = grouped ? eff_masks : masks;
    const int64_t* rstr = grouped ? eff_row_strides : row_strides;
    const int32_t* fstr = grouped ? eff_stride : frag_stride;
    // scratch: w[count] + rows[n_frag][count] (+ split partials for the GEMM path, + merged group tables)
    const int mA = __builtin_popcountll(msk[0]);
    const int mB = n_eff >= 2 ? __builtin_popcountll(msk[1]) : 0;
    // two fragments always take the tile kernels: rows shorter than a tile (a fragment with fewer than 6 output
    // bits, e.g. the 5-bit side of aqft-16 with five wire cuts) are padded with zeros inside the tile - the
    // per-output generic kernel walks all labels serially (19.5 ms against 0.3 ms for those 32 768 labels)
    const bool gemm = (n_eff == 2);
    const int mAp = mA < 6 ? 6 : mA, mBp = mB < 6 ? 6 : mB;
    int n_split = 1;
    bool big_tile = false;
    size_t partial_bytes = 0;
    if (gemm) {
        // 128x128 tiles (one CTA per SM) when both padded dimensions allow it and there are labels enough to keep
        // the three-stage ring busy; else 64x64 tiles, ~2 CTAs per SM (QCK_CONTRACT_TILE=64 / 128 forces one)
        const char* tile_env = getenv("QCK_CONTRACT_TILE");
        big_tile = mAp >= 7 && mBp >= 7 && count >= 4096;
        if (tile_env) big_tile = atoi(tile_env) == 128 && mAp >= 7 && mBp >= 7;
        const int tb = big_tile ? 7 : 6;
        long long tiles = (1ll << (mAp - tb)) * (1ll << (mBp - tb));
        // the pipelined kernel hides its own latency, more splits only add partial-sum traffic
        const char* split_env = getenv("QCK_CONTRACT_CTAS_PER_SM");
        const long long per_sm = split_env ? atoi(split_env) : (big_tile ? 1 : 2);
        long long want = ((per_sm > 0 ? per_sm : 2) * h->sm_count + tiles - 1) / tiles;
        if (big_tile && !split_env) want = h->sm_count / tiles > 0 ? h->sm_count / tiles : 1;  // one wave, never two
        long long maxs = (count + 4 * GK - 1) / (4 * GK);
        n_split = (int)(want < maxs ? want : maxs);
        if (n_split < 1) n_split = 1;
        if (n_split > 64) n_split = 64;
        partial_bytes = (size_t)n_split * sizeof(double) << (mAp + mBp);
    }
    size_t w_bytes = ((size_t)count * sizeof(double) + 255) & ~(size_t)255;
    size_t r_bytes = ((size_t)count * n_eff * sizeof(int) + 255) & ~(size_t)255;
    partial_bytes = (partial_bytes + 255) & ~(size_t)255;
    void* scratch = nullptr;
    int rc = qck_ensure_scratch(h, w_bytes + r_bytes + partial_bytes + merged_bytes[0] + merged_bytes[1], &scratch);
    if (rc) return rc;
    double* d_w = (double*)scratch;
    int* d_rows = (int*)((char*)scratch + w_bytes);
    double* d_partial = (double*)((char*)scratch + w_bytes + r_bytes);
    if (grouped) {
        char* at = (char*)scratch + w_bytes + r_bytes + partial_bytes;
        for (int g = 0; g < 2; ++g) {
            if (!merged_bytes[g]) continue;
            MergeParams mp;
            memset(&mp, 0, sizeof(mp));
            mp.n_digits = n_digits;
            mp.m_bits = __builtin_popcountll(eff_masks[g]);
            for (int f = 0; f < n_frag; ++f)
                if (((group_of_frag >> f) & 1) == g) {
                    const int j = mp.n_frag++;
                    mp.table[j] = d_tables[f];
                    mp.row_stride[j] = row_strides[f];
                    mp.cmask[j] = compress_mask(masks[f], eff_masks[g]);
                    for (int k = 0; k < n_digits; ++k) mp.stride[j][k] = frag_stride[f * QCK_MAX_DIGITS + k];
                }
            for (int k = 0; k < n_digits; ++k) {
                mp.radix[k] = radix[k];
                mp.touched[k] = eff_stride[g * QCK_MAX_DIGITS + k] != 0;
            }
            mp.n_labels = group_labels[g];
            mp.out = (double*)at;
            eff_tables[g] = (const double*)at;
            at += merged_bytes[g];
            const long long want = group_labels[g] < (long long)h->sm_count * 16 ? group_labels[g] : (long long)h->sm_count * 16;
            contract_merge_kernel<<<(int)want, 256, 0, st>>>(mp);
            QCK_CHECK_LAUNCH(h);
        }
    }

    rc = qck_contract_prep(h, n_eff, n_digits, radix, coef, fstr, l_begin, count, d_w, d_rows, st);
    if (rc) return rc;

    ContractParams cp;
    memset(&cp, 0, sizeof(cp));
    cp.n_frag = n_eff;
    for (int f = 0; f < n_eff; ++f) {
        cp.table[f] = tabs[f];
        cp.mask[f] = msk[f];
        cp.row_stride[f] = rstr[f];
    }
    cp.n_out_bits = n_out_bits;
    cp.count = count;
    cp.w = d_w;
    cp.rows = d_rows;
    cp.out = d_out;
    cp.accumulate = accumulate;
    const unsigned long long n = 1ull << n_out_bits;
    int ggrid = (int)((n + 255) / 256 < (unsigned long long)h->sm_count * 8 ? (n + 255) / 256
                                                                           : (unsigned long long)h->sm_count * 8);
    if (gemm && full_cover) {
        const int M = 1 << mAp, N = 1 << mBp, Mr = 1 << mA, Nr = 1 << mB;
        dim3 grid(M / GT, N / GT, n_split);
        // pipelined gather (cp.async, 16-byte requests): rows must start on 16-byte boundaries and be even
        const char* pipe_env = getenv("QCK_CONTRACT_PIPE");
        const bool aligned = ((reinterpret_cast<uintptr_t>(tabs[0]) | reinterpret_cast<uintptr_t>(tabs[1])) & 15) == 0 &&
                             ((rstr[0] | rstr[1]) & 1) == 0 && Mr >= 2 && Nr >= 2;
        if (aligned && !(pipe_env && atoi(pipe_env) == 0)) {
            static bool attr_set = false;  // process-wide function attributes, same values from every thread
            if (!attr_set) {
                QCK_CUDA(h, cudaFuncSetAttribute(contract_dmma_pipe_kernel<64, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)(GS * sizeof(ContractStage<64>))));
                QCK_CUDA(h, cudaFuncSetAttribute(contract_dmma_pipe_kernel<128, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)(GS * sizeof(ContractStage<128>))));
                attr_set = true;
            }
            if (big_tile)
                contract_dmma_pipe_kernel<128, 16><<<dim3(M / 128, N / 128, n_split), 512, GS * sizeof(ContractStage<128>), st>>>(
                    cp, n_split, d_partial, M, N, Mr, Nr);
            else
                contract_dmma_pipe_kernel<64, 8><<<grid, 256, GS * sizeof(ContractStage<64>), st>>>(cp, n_split, d_partial, M, N,
                                                                                                   Mr, Nr);
        }
        else
            contract_dmma_kernel<<<grid, 256, 0, st>>>(cp, n_split, d_partial, M, N, Mr, Nr);
        QCK_CHECK_LAUNCH(h);
        const long long tile_entries = (long long)M * N;
        const int sgrid = (int)((tile_entries + 255) / 256 < (long long)h->sm_count * 8 ? (tile_entries + 255) / 256
                                                                                       : (long long)h->sm_count * 8);
        contract_scatter_kernel<<<sgrid, 256, 0, st>>>(d_partial, n_split, M, N, Mr, Nr, msk[0], msk[1], d_out, accumulate);
        QCK_CHECK_LAUNCH(h);
    } else {
        contract_generic_kernel<<<ggrid, 256, 0, st>>>(cp);
        QCK_CHECK_LAUNCH(h);
    }
    return QCK_OK;
}

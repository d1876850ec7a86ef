// QuasiDistr.nearest_probability_distribution (third_party/qvm/qvm/quasi_distr.py:28-43) on a dense
// vector, without sorting and without a host round trip (sm_100a).
//
// The reference sorts ascending and drops the j-th smallest value while
//     v_(j) + (sum of the j-1 smaller ones) / (N - j + 1) < 0   <=>   g(j) = v_(j) (N - j + 1) + S_(j-1) < 0.
// g(j) = G(v_(j)) with G(t) = sum_i min(v_i, t), a continuous non-decreasing function of t, so an entry is
// dropped <=> v < t0 = inf{t : G(t) >= 0}; the survivors get v + beta / num (beta = sum of the dropped
// entries, num = number of survivors).  Only the PARTITION of the data at t0 matters.
//
// t0 is located by radix refinement on the order-preserving integer image ("key") of the doubles:
//   stats   sum S, minimum, sum of the negative entries; min >= 0 -> identity.  S >= 0 implies
//           G(|neg_sum|) >= 0, so t0 lies in [min, |neg_sum|] (the entries above are certainly kept);
//   level l the key range (lo, hi] known to hold t0 is cut into <= 8192 bins; one pass counts the entries
//           per bin and sums them as integers, q = llrint((v - val(lo + 1)) * 2^qexp) (order independent,
//           hence deterministic; exact once the range is narrow), and sums the entries at or below lo as
//           doubles in a fixed order.  The tail (the last CTA to finish, or a one-CTA launch when the
//           bins are all-reduced across ranks in between) evaluates G at every bin boundary and keeps the
//           first bin whose upper boundary has G >= 0.  An empty bin or a one-key bin ends the search:
//           the dropped set is {key <= lo}.  13 bits per level: at most 5 levels.
//   final   one more pass of the same kernel recomputes (sum, count) of {key <= lo} in doubles -> beta, num;
//   apply   v -> v + beta / num for the survivors, 0 for the rest.
// Every launch is enqueued unconditionally and looks at the state left by the previous one (a launch
// with nothing to do returns at once): 8 launches, no cudaStreamSynchronize, against the ~66 probe +
// read-back round trips of a host-driven bisection.
#include "qck_common.cuh"

#include <cooperative_groups.h>
#include <math.h>

#define NPD_BINS 8192
#define NPD_BIN_BITS 13
#define NPD_LEVELS 5
#define NPD_GRID_MAX 2048
#define NPD_THREADS 256

// status values of NpdState::status
#define NPD_SEARCH 0
#define NPD_IDENTITY 1
#define NPD_SOLVED 2
#define NPD_NEGATIVE_TOTAL 3
#define NPD_LOCATED 4  // the partition key is known, (sum, count) of the dropped entries still to be taken

struct NpdState {  // 8-byte slots; the first QCK_NPD_STATE_SLOTS of the workspace (qck.h documents them)
    double sum, vmin, neg_sum, alive, neg_cnt;  // 0-4: statistics over alive entries (|v| > acc)
    long long status;                           // 5
    long long lo, hi;                           // 6, 7: t0's key lies in (lo, hi]
    long long shift;                            // 8: bin of a key = (key - lo - 1) >> shift
    long long qexp;                             // 9: q = llrint((v - val(lo + 1)) * 2^qexp)
    double under_sum, under_cnt;                // 10, 11: over alive entries with key <= lo
    long long sel_cnt;                          // 12: upper bound of the entries with key in (lo, hi]
    double t0, shift_val, beta, num;            // 13-16: result (t0 = smallest kept value's lower bound)
    unsigned long long ticket;                  // 17
    long long level;                            // 18: levels done
    long long pad[13];
};
static_assert(sizeof(NpdState) == 8 * QCK_NPD_STATE_SLOTS, "NpdState must fill the documented slots");

__host__ __device__ __forceinline__ long long npd_key(double d) {
#ifdef __CUDA_ARCH__
    long long b = __double_as_longlong(d);
#else
    long long b;
    memcpy(&b, &d, 8);
#endif
    return b < 0 ? (long long)(0x8000000000000000ull - (unsigned long long)b) : b;
}
__host__ __device__ __forceinline__ double npd_val(long long o) {
    long long b = o < 0 ? (long long)(0x8000000000000000ull - (unsigned long long)o) : o;
#ifdef __CUDA_ARCH__
    return __longlong_as_double(b);
#else
    double d;
    memcpy(&d, &b, 8);
    return d;
#endif
}

struct NpdWs {
    NpdState* st;
    unsigned long long* bin_cnt;  // [NPD_BINS]
    long long* bin_q;             // [NPD_BINS]
    double* partials;             // [NPD_GRID_MAX * 8]
};
__host__ __device__ __forceinline__ NpdWs npd_ws(void* ws) {
    NpdWs w;
    char* b = reinterpret_cast<char*>(ws);
    w.st = reinterpret_cast<NpdState*>(b);
    w.bin_cnt = reinterpret_cast<unsigned long long*>(b + sizeof(NpdState));
    w.bin_q = reinterpret_cast<long long*>(b + sizeof(NpdState) + 8 * NPD_BINS);
    w.partials = reinterpret_cast<double*>(b + sizeof(NpdState) + 16 * NPD_BINS);
    return w;
}
static const size_t NPD_WS_BYTES = sizeof(NpdState) + 16 * NPD_BINS + 8 * 8 * NPD_GRID_MAX;

// ---- block helpers (fixed reduction order: deterministic)
__device__ __forceinline__ double block_sum(double v, double* red) {  // red: >= 8 doubles of shared memory
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
    return s;
}
__device__ __forceinline__ double block_min(double v, double* red) {
    v = warp_min(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = INFINITY;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s = fmin(s, red[w]);
    return s;
}
// true in every thread of exactly one CTA: the last one to get here (its view of global memory is complete)
__device__ __forceinline__ bool last_cta(unsigned long long* ticket) {
    __shared__ int is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned long long t = atomicAdd(ticket, 1ull);
        is_last = (t == (unsigned long long)gridDim.x - 1ull);
        if (is_last) *ticket = 0ull;
    }
    __syncthreads();
    if (is_last) __threadfence();
    return is_last != 0;
}

// bins and quantisation of the current range (one thread)
__device__ void npd_set_level(NpdState* s, int bin_bits = NPD_BIN_BITS) {
    const unsigned long long width = (unsigned long long)s->hi - (unsigned long long)s->lo;  // >= 1
    int bits = 64 - __clzll((long long)(width - 1ull));                                      // ceil(log2(width))
    if (width <= 1ull) bits = 0;
    s->shift = bits > bin_bits ? bits - bin_bits : 0;
    const double w = npd_val(s->hi) - npd_val(s->lo + 1);
    long long cnt = s->sel_cnt < 1 ? 1 : s->sel_cnt;
    const int cbits = 64 - __clzll(cnt);  // cnt < 2^cbits
    int e = 0;
    if (w > 0.0 && isfinite(w)) e = 61 - cbits - (ilogb(w) + 1);  // cnt * w * 2^e < 2^61
    s->qexp = e;
}

// after the statistics: identity / error / first range
__device__ void npd_plan_tail(NpdWs w) {
    NpdState* s = w.st;
    for (int i = threadIdx.x; i < NPD_BINS; i += blockDim.x) {
        w.bin_cnt[i] = 0ull;
        w.bin_q[i] = 0ll;
    }
    if (threadIdx.x == 0) {
        s->level = 0;
        s->under_sum = 0.0;
        s->under_cnt = 0.0;
        s->beta = 0.0;
        s->num = s->alive;
        s->shift_val = 0.0;
        s->t0 = -INFINITY;
        if (!(s->alive > 0.0) || !(s->vmin < 0.0)) {
            s->status = NPD_IDENTITY;
        } else if (s->sum < 0.0) {
            s->status = NPD_NEGATIVE_TOTAL;  // the reference ends up dividing by zero here
        } else {
            s->status = NPD_SEARCH;
            const double t_ub = -s->neg_sum * (1.0 + 1e-9);
            s->lo = npd_key(s->vmin) - 1;
            s->hi = npd_key(t_ub);
            s->sel_cnt = (long long)s->alive;
            npd_set_level(s);
        }
    }
}

// after a histogram pass: pick the bin that holds t0, or finish
__device__ void npd_select_tail(NpdWs w) {
    NpdState* s = w.st;
    __shared__ unsigned long long sc[NPD_THREADS];
    __shared__ long long sq[NPD_THREADS];
    __shared__ int found;
    const int status = (int)s->status;
    if (status == NPD_LOCATED) {  // this pass only took (sum, count) of the dropped entries
        if (threadIdx.x == 0) {
            s->beta = s->under_sum;
            s->num = s->alive - s->under_cnt;
            s->shift_val = s->num > 0.0 ? s->beta / s->num : 0.0;
            s->t0 = npd_val(s->lo + 1);
            s->status = NPD_SOLVED;
        }
        return;
    }
    if (status != NPD_SEARCH) return;
    constexpr int PER = NPD_BINS / NPD_THREADS;  // consecutive bins per thread
    static_assert(PER == 32, "the second search level is one warp wide");
    const int b0 = threadIdx.x * PER;
    unsigned long long c = 0ull;
    long long q = 0ll;
    for (int i = 0; i < PER; ++i) {
        c += w.bin_cnt[b0 + i];
        q += w.bin_q[b0 + i];
    }
    // exclusive prefix over the threads (integers: any order is exact) - warp scans + one pass over the warp
    // totals.  (The serial form, thread t adding t shared-memory entries, was ~4 us per level: half of the time
    // of a level at 2^16 entries.)
    __shared__ unsigned long long wc[NPD_THREADS / 32];
    __shared__ long long wq[NPD_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long c_in = c;
    long long q_in = q;
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long cu = __shfl_up_sync(0xffffffffu, c_in, o);
        const long long qu = __shfl_up_sync(0xffffffffu, q_in, o);
        if (lane >= o) {
            c_in += cu;
            q_in += qu;
        }
    }
    if (lane == 31) {
        wc[warp] = c_in;
        wq[warp] = q_in;
    }
    if (threadIdx.x == 0) found = NPD_BINS;
    __syncthreads();
    unsigned long long c_ex = c_in - c;
    long long q_ex = q_in - q;
    for (int t = 0; t < warp; ++t) {
        c_ex += wc[t];
        q_ex += wq[t];
    }
    sc[threadIdx.x] = c_ex;  // exclusive prefixes: what precedes thread t's block of bins
    sq[threadIdx.x] = q_ex;
    const long long lo = s->lo, hi = s->hi;
    const int shift = (int)s->shift;
    const double lo_val = npd_val(lo + 1);
    const int qexp = (int)s->qexp;
    const double rest = s->alive - s->under_cnt, under = s->under_sum;
    const unsigned long long width = (unsigned long long)hi - (unsigned long long)lo;
    // G at the upper boundary of bin j, given the entries (count c, integer sum q) of bins 0..j
    auto g_at = [&](int j, unsigned long long c, long long q, bool* is_last) -> double {
        unsigned long long off = ((unsigned long long)(j + 1)) << shift;  // keys up to lo + off belong to bins <= j
        if (off > width || (shift > 0 && (off >> shift) != (unsigned long long)(j + 1))) off = width;
        *is_last = off == width;
        const double ub = npd_val(lo + (long long)off);
        return under + ((double)c * lo_val + scalbn((double)q, -qexp)) + ub * (rest - (double)c);
    };
    // two-level search (G is non-decreasing): first the 32-bin block whose END has G >= 0 - one evaluation
    // per thread -, then the bin inside that block - one evaluation per lane of warp 0
    __shared__ int found_block;
    if (threadIdx.x == 0) found_block = NPD_THREADS;
    __syncthreads();
    {
        bool is_last;
        const double g = g_at(b0 + PER - 1, c_ex + c, q_ex + q, &is_last);
        if (g >= 0.0 || is_last) atomicMin(&found_block, (int)threadIdx.x);
    }
    __syncthreads();
    const int blk = found_block;
    int mine = NPD_BINS;
    if (threadIdx.x < PER) {  // (PER == 32: warp 0) - inclusive scan of the block's 32 bins on top of its prefix
        unsigned long long cb = w.bin_cnt[blk * PER + (int)threadIdx.x];
        long long qb = w.bin_q[blk * PER + (int)threadIdx.x];
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long cu = __shfl_up_sync(0xffffffffu, cb, o);
            const long long qu = __shfl_up_sync(0xffffffffu, qb, o);
            if (lane >= o) {
                cb += cu;
                qb += qu;
            }
        }
        cb += sc[blk];
        qb += sq[blk];
        bool is_last;
        const double g = g_at(blk * PER + (int)threadIdx.x, cb, qb, &is_last);
        if (g >= 0.0 || is_last) mine = blk * PER + (int)threadIdx.x;
    }
    atomicMin(&found, mine);
    __syncthreads();
    const int j = found;
    if (threadIdx.x == 0) {
        unsigned long long off_lo = ((unsigned long long)j) << shift;
        unsigned long long off_hi = ((unsigned long long)(j + 1)) << shift;
        if (off_hi > width || (shift > 0 && (off_hi >> shift) != (unsigned long long)(j + 1))) off_hi = width;
        const unsigned long long cnt_j = w.bin_cnt[j];
        s->lo = lo + (long long)off_lo;
        s->hi = lo + (long long)off_hi;
        s->sel_cnt = (long long)cnt_j;
        s->level += 1;
        if (cnt_j == 0ull || off_hi - off_lo <= 1ull) {
            s->status = NPD_LOCATED;  // dropped = {key <= lo}; the next pass sums them
        } else {
            npd_set_level(s);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < NPD_BINS; i += blockDim.x) {
        w.bin_cnt[i] = 0ull;
        w.bin_q[i] = 0ll;
    }
}

// ---- pass 1: statistics
__global__ void __launch_bounds__(NPD_THREADS) npd_stats_kernel(const double* __restrict__ p, unsigned long long n,
                                                                double acc, void* ws_raw, int fuse_tail) {
    NpdWs w = npd_ws(ws_raw);
    __shared__ double red[8];
    double s = 0.0, m = INFINITY, ns = 0.0, z = 0.0, nz = 0.0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const double v = p[i];
        if (fabs(v) > acc) {
            s += v;
            m = fmin(m, v);
            z += 1.0;
            if (v < 0.0) {
                ns += v;
                nz += 1.0;
            }
        }
    }
    s = block_sum(s, red);
    m = block_min(m, red);
    ns = block_sum(ns, red);
    z = block_sum(z, red);
    nz = block_sum(nz, red);
    if (threadIdx.x == 0) {
        double* o = w.partials + 8 * blockIdx.x;
        o[0] = s; o[1] = m; o[2] = ns; o[3] = z; o[4] = nz;
    }
    if (!last_cta(&w.st->ticket)) return;
    s = 0.0; m = INFINITY; ns = 0.0; z = 0.0; nz = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) {
        const double* o = w.partials + 8 * i;
        s += o[0]; m = fmin(m, o[1]); ns += o[2]; z += o[3]; nz += o[4];
    }
    s = block_sum(s, red);
    m = block_min(m, red);
    ns = block_sum(ns, red);
    z = block_sum(z, red);
    nz = block_sum(nz, red);
    if (threadIdx.x == 0) {
        w.st->sum = s; w.st->vmin = m; w.st->neg_sum = ns; w.st->alive = z; w.st->neg_cnt = nz;
    }
    __syncthreads();
    if (fuse_tail) npd_plan_tail(w);
}

// ---- levels: histogram of the current range + (sum, count) below it
extern __shared__ __align__(16) unsigned char npd_smem[];

__global__ void __launch_bounds__(NPD_THREADS) npd_hist_kernel(const double* __restrict__ p, unsigned long long n,
                                                               double acc, void* ws_raw, int fuse_tail) {
    NpdWs w = npd_ws(ws_raw);
    const int status = (int)w.st->status;
    if (status != NPD_SEARCH && status != NPD_LOCATED) return;  // uniform over the grid
    __shared__ double red[8];
    unsigned int* h_cnt = reinterpret_cast<unsigned int*>(npd_smem);
    unsigned long long* h_q = reinterpret_cast<unsigned long long*>(npd_smem + 4 * NPD_BINS);
    const bool bins = status == NPD_SEARCH;
    if (bins) {
        for (int i = threadIdx.x; i < NPD_BINS; i += blockDim.x) {
            h_cnt[i] = 0u;
            h_q[i] = 0ull;
        }
    }
    const long long lo = w.st->lo, hi = w.st->hi;
    const int shift = (int)w.st->shift;
    const double lo_val = npd_val(lo + 1);
    const int qexp = (int)w.st->qexp;
    __syncthreads();
    double us = 0.0, uc = 0.0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const double v = p[i];
        if (!(fabs(v) > acc)) continue;
        const long long k = npd_key(v);
        if (k <= lo) {
            us += v;
            uc += 1.0;
        } else if (bins && k <= hi) {
            const unsigned int b = (unsigned int)(((unsigned long long)k - (unsigned long long)lo - 1ull) >> shift);
            atomicAdd(&h_cnt[b], 1u);
            atomicAdd(&h_q[b], (unsigned long long)__double2ll_rn(scalbn(v - lo_val, qexp)));
        }
    }
    us = block_sum(us, red);
    uc = block_sum(uc, red);
    if (threadIdx.x == 0) {
        w.partials[8 * blockIdx.x + 0] = us;
        w.partials[8 * blockIdx.x + 1] = uc;
    }
    if (bins) {
        __syncthreads();
        for (int i = threadIdx.x; i < NPD_BINS; i += blockDim.x) {
            const unsigned int c = h_cnt[i];
            if (c) {
                atomicAdd(&w.bin_cnt[i], (unsigned long long)c);
                atomicAdd(reinterpret_cast<unsigned long long*>(&w.bin_q[i]), h_q[i]);
            }
        }
    }
    if (!last_cta(&w.st->ticket)) return;
    us = 0.0;
    uc = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) {
        us += w.partials[8 * i + 0];
        uc += w.partials[8 * i + 1];
    }
    us = block_sum(us, red);
    uc = block_sum(uc, red);
    if (threadIdx.x == 0) {
        w.st->under_sum = us;
        w.st->under_cnt = uc;
    }
    __syncthreads();
    if (fuse_tail) npd_select_tail(w);
}

// one-CTA launches of the tails (multi-rank runs reduce the statistics / bins across ranks in between)
__global__ void __launch_bounds__(NPD_THREADS) npd_plan_kernel(void* ws_raw) { npd_plan_tail(npd_ws(ws_raw)); }
__global__ void __launch_bounds__(NPD_THREADS) npd_select_kernel(void* ws_raw) { npd_select_tail(npd_ws(ws_raw)); }

// ---- apply
__global__ void __launch_bounds__(NPD_THREADS) npd_apply_kernel(double* __restrict__ p, unsigned long long n, double acc,
                                                                const void* ws_raw) {
    const NpdState* s = reinterpret_cast<const NpdState*>(ws_raw);
    const int status = (int)s->status;
    if (status == NPD_IDENTITY && !(acc > 0.0)) return;
    if (status != NPD_IDENTITY && status != NPD_SOLVED) return;  // unsolved / negative total: the caller checks
    const long long lo = status == NPD_SOLVED ? s->lo : (long long)0x8000000000000000ull;
    const double shift = status == NPD_SOLVED ? s->shift_val : 0.0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const double v = p[i];
        p[i] = (fabs(v) > acc && npd_key(v) > lo) ? v + shift : 0.0;
    }
}

// ---- vectors of at most 2^16 entries (every 16-qubit configuration): the whole search as ONE launch of ONE
// thread-block cluster.  Eight CTAs hold the vector in registers (16 entries per thread); the passes are separated
// by cluster barriers instead of launches; the bins (2048 per level: 11 key bits) live in shared memory.  After a
// pass CTA r adds up bins [256 r, 256 r + 256) of all eight CTAs through distributed shared memory, the slice totals
// tell every CTA which slice holds t0, the CTA owning that slice picks the bin and writes the new search state into
// the shared memory of all eight.  Nothing but the vector itself and the final state touches global memory.
// (Every CTA reading all eight histograms was tried first: 196 KB through a 17-21 B/clk DSMEM port per level.)
// Same definitions as the staged kernels above (key ranges, integer quantisation, G at the bin boundaries, the
// under-range sums in a fixed order): the partition is the same set, beta may differ in the last bit (another
// summation order).
#define NPC_CTAS 8
#define NPC_THREADS 512
#define NPC_WARPS (NPC_THREADS / 32)
#define NPC_VPT 16
#define NPC_BINS 2048
#define NPC_BIN_BITS 11
#define NPC_SLICE (NPC_BINS / NPC_CTAS)
#define NPC_LEVELS 6
#define NPC_CAPACITY (NPC_CTAS * NPC_THREADS * NPC_VPT)
static_assert(NPC_SLICE == 256 && NPC_BINS % NPC_THREADS == 0 && NPC_LEVELS * NPC_BIN_BITS >= 64, "npd cluster kernel geometry");

struct NpcShared {
    unsigned int cnt[NPC_BINS];           // bins of this CTA's entries
    unsigned int q_lo[NPC_BINS], q_hi[NPC_BINS];  // integer sums (64 bits in two words)
    double part[8];                       // this CTA's statistics / (sum, count) of its entries at or below lo
    long long slice_tot[2];               // (count, integer sum) of this CTA's slice of the bins, all CTAs added
    double gathered[NPC_CTAS * 5];
    long long gathered_slices[NPC_CTAS * 2];
    double red[NPC_WARPS][5];
    long long wtot[NPC_SLICE / 32][2];
    int found;
    NpdState st;                          // every CTA keeps a copy of the search state
};

// sums (index 1: minimum) of N per-thread values over the CTA in a fixed order -> out[0..N) (valid after the next barrier)
template <int N>
__device__ __forceinline__ void npc_block_reduce(double (&x)[N], NpcShared& S, double* out, bool second_is_min) {
    const int tid = threadIdx.x;
#pragma unroll
    for (int i = 0; i < N; ++i) x[i] = (second_is_min && i == 1) ? warp_min(x[i]) : warp_sum(x[i]);
    if ((tid & 31) == 0)
#pragma unroll
        for (int i = 0; i < N; ++i) S.red[tid >> 5][i] = x[i];
    __syncthreads();
    if (tid < N) {
        double a = (second_is_min && tid == 1) ? INFINITY : 0.0;
        for (int w = 0; w < NPC_WARPS; ++w) a = (second_is_min && tid == 1) ? fmin(a, S.red[w][tid]) : a + S.red[w][tid];
        out[tid] = a;
    }
}

__global__ void __cluster_dims__(NPC_CTAS, 1, 1) __launch_bounds__(NPC_THREADS)
    npd_cluster_kernel(double* __restrict__ p, unsigned long long n, double acc, void* ws_raw) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    NpcShared& S = *reinterpret_cast<NpcShared*>(npd_smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned int rank = cluster.block_rank();
    NpdState* s = &S.st;

    // the vector, 16 entries per thread (entry i of the vector: CTA i / 8192, then coalesced)
    double v[NPC_VPT];
    unsigned int alive = 0u;
    const unsigned long long base = (unsigned long long)rank * (NPC_THREADS * NPC_VPT) + tid;
#pragma unroll
    for (int j = 0; j < NPC_VPT; ++j) {
        const unsigned long long i = base + (unsigned long long)j * NPC_THREADS;
        v[j] = i < n ? p[i] : 0.0;
        if (i < n && fabs(v[j]) > acc) alive |= 1u << j;
    }
    // statistics: sum, minimum, sum of the negative entries, number of alive / negative entries
    {
        double x[5] = {0.0, INFINITY, 0.0, 0.0, 0.0};
#pragma unroll
        for (int j = 0; j < NPC_VPT; ++j)
            if (alive >> j & 1u) {
                x[0] += v[j];
                x[1] = fmin(x[1], v[j]);
                x[3] += 1.0;
                if (v[j] < 0.0) {
                    x[2] += v[j];
                    x[4] += 1.0;
                }
            }
        npc_block_reduce<5>(x, S, S.part, true);
    }
    cluster.sync();
    if (tid < NPC_CTAS * 5) S.gathered[tid] = cluster.map_shared_rank(S.part, tid / 5)[tid % 5];
    __syncthreads();
    if (tid == 0) {  // rank order: the same bits in every CTA
        double sm = 0.0, m = INFINITY, ns = 0.0, z = 0.0, nz = 0.0;
        for (int r = 0; r < NPC_CTAS; ++r) {
            sm += S.gathered[5 * r + 0];
            m = fmin(m, S.gathered[5 * r + 1]);
            ns += S.gathered[5 * r + 2];
            z += S.gathered[5 * r + 3];
            nz += S.gathered[5 * r + 4];
        }
        memset(s, 0, sizeof(NpdState));
        s->sum = sm; s->vmin = m; s->neg_sum = ns; s->alive = z; s->neg_cnt = nz;
        s->num = z;
        s->t0 = -INFINITY;
        if (!(z > 0.0) || !(m < 0.0)) {
            s->status = NPD_IDENTITY;
        } else if (sm < 0.0) {
            s->status = NPD_NEGATIVE_TOTAL;
        } else {
            s->status = NPD_SEARCH;
            // G(0) = neg_sum < 0: t0 > 0, every entry <= 0 is dropped - the search starts above zero
            s->lo = 0ll;
            s->hi = npd_key(-ns * (1.0 + 1e-9));
            s->sel_cnt = (long long)z;
            npd_set_level(s, NPC_BIN_BITS);
        }
    }
    cluster.sync();  // (also: S.part has been read by every CTA before the first pass overwrites it)

    for (int level = 0; level <= NPC_LEVELS + 1; ++level) {
        const int status = (int)s->status;
        if (status != NPD_SEARCH && status != NPD_LOCATED) break;  // the same decision in every CTA
        const bool bins = status == NPD_SEARCH;
        if (bins) {
#pragma unroll
            for (int i = 0; i < NPC_BINS / NPC_THREADS; ++i) {
                S.cnt[tid + i * NPC_THREADS] = 0u;
                S.q_lo[tid + i * NPC_THREADS] = 0u;
                S.q_hi[tid + i * NPC_THREADS] = 0u;
            }
        }
        const long long lo = s->lo, hi = s->hi;
        const int shift = (int)s->shift;
        const double lo_val = npd_val(lo + 1);
        const int qexp = (int)s->qexp;
        const double alive_total = s->alive;
        __syncthreads();
        double x[2] = {0.0, 0.0};
#pragma unroll
        for (int j = 0; j < NPC_VPT; ++j) {
            const long long k = npd_key(v[j]);
            const bool a = alive >> j & 1u;
            if (a && k <= lo) {
                x[0] += v[j];
                x[1] += 1.0;
            }
            if (bins && a && k > lo && k <= hi) {
                const unsigned int b = (unsigned int)(((unsigned long long)k - (unsigned long long)lo - 1ull) >> shift);
                const unsigned long long qv = (unsigned long long)__double2ll_rn(scalbn(v[j] - lo_val, qexp));  // < 2^61
                // 64-bit integer sum as two native 32-bit shared-memory atomics, the carry added by the thread whose
                // addition wrapped (a 64-bit atomicAdd on shared memory compiles to a compare-and-swap spin loop).
                // (Adding up lanes with the same bin inside the warp first - __match_any_sync, or the bin of the first
                // pending lane - was slower on every knitted result tried: rounding noise spreads over many binades.)
                atomicAdd(&S.cnt[b], 1u);
                const unsigned int ql = (unsigned int)qv, qh = (unsigned int)(qv >> 32);
                const unsigned int old = atomicAdd(&S.q_lo[b], ql);
                const unsigned int carry = old + ql < old ? 1u : 0u;
                if (qh + carry) atomicAdd(&S.q_hi[b], qh + carry);
            }
        }
        npc_block_reduce<2>(x, S, S.part, false);
        cluster.sync();  // bins and partial sums of every CTA are complete
        if (tid < NPC_CTAS * 2) S.gathered[tid] = cluster.map_shared_rank(S.part, tid / 2)[tid % 2];
        unsigned int c_bin = 0u;
        long long q_bin = 0ll, c_in = 0ll, q_in = 0ll;
        if (bins && tid < NPC_SLICE) {  // my slice of the bins, all CTAs added (integers)
            const int bin = (int)rank * NPC_SLICE + tid;
#pragma unroll
            for (int r = 0; r < NPC_CTAS; ++r) {
                c_bin += cluster.map_shared_rank(S.cnt, r)[bin];
                q_bin += (long long)(((unsigned long long)cluster.map_shared_rank(S.q_hi, r)[bin] << 32) +
                                     (unsigned long long)cluster.map_shared_rank(S.q_lo, r)[bin]);
            }
            // inclusive prefix inside the slice: warp scans, then the warp totals
            c_in = (long long)c_bin;
            q_in = q_bin;
            for (int o = 1; o < 32; o <<= 1) {
                const long long cu = __shfl_up_sync(0xffffffffu, c_in, o);
                const long long qu = __shfl_up_sync(0xffffffffu, q_in, o);
                if (lane >= o) {
                    c_in += cu;
                    q_in += qu;
                }
            }
            if (lane == 31) {
                S.wtot[warp][0] = c_in;
                S.wtot[warp][1] = q_in;
            }
        }
        __syncthreads();
        if (tid == 0) {
            double a = 0.0, b = 0.0;
            for (int r = 0; r < NPC_CTAS; ++r) {
                a += S.gathered[2 * r + 0];
                b += S.gathered[2 * r + 1];
            }
            s->under_sum = a;
            s->under_cnt = b;
            if (!bins) {  // this pass only took (sum, count) of the dropped entries
                s->beta = a;
                s->num = s->alive - b;
                s->shift_val = s->num > 0.0 ? s->beta / s->num : 0.0;
                s->t0 = npd_val(s->lo + 1);
                s->status = NPD_SOLVED;
            } else {
                long long ct = 0ll, qt = 0ll;
                for (int w = 0; w < NPC_SLICE / 32; ++w) {
                    ct += S.wtot[w][0];
                    qt += S.wtot[w][1];
                }
                S.slice_tot[0] = ct;
                S.slice_tot[1] = qt;
            }
            S.found = NPC_BINS;
        }
        if (!bins) {
            __syncthreads();
            continue;  // every CTA has computed the same state
        }
        cluster.sync();  // slice totals
        if (tid < NPC_CTAS * 2) S.gathered_slices[tid] = cluster.map_shared_rank(S.slice_tot, tid / 2)[tid % 2];
        __syncthreads();
        const double rest = alive_total - s->under_cnt, under = s->under_sum;
        const unsigned long long width = (unsigned long long)hi - (unsigned long long)lo;
        // G at the upper boundary of bin j, given the entries (count cc, integer sum qq) of bins 0..j
        auto g_at = [&](int j, long long cc, long long qq, bool* is_last) -> double {
            unsigned long long off = ((unsigned long long)(j + 1)) << shift;
            if (off > width || (shift > 0 && (off >> shift) != (unsigned long long)(j + 1))) off = width;
            *is_last = off == width;
            const double ub = npd_val(lo + (long long)off);
            return under + ((double)cc * lo_val + scalbn((double)qq, -qexp)) + ub * (rest - (double)cc);
        };
        // the slice that holds t0: the first one whose END has G >= 0 (G is non-decreasing) - the same in every CTA
        int owner = NPC_CTAS - 1;
        long long c_before = 0ll, q_before = 0ll;
        {
            long long cc = 0ll, qq = 0ll;
            for (int r = 0; r < NPC_CTAS; ++r) {
                const long long c0 = cc, q0 = qq;
                cc += S.gathered_slices[2 * r + 0];
                qq += S.gathered_slices[2 * r + 1];
                bool is_last;
                const double g = g_at(r * NPC_SLICE + NPC_SLICE - 1, cc, qq, &is_last);
                if (g >= 0.0 || is_last || r == NPC_CTAS - 1) {
                    owner = r;
                    c_before = c0;
                    q_before = q0;
                    break;
                }
            }
        }
        if ((int)rank == owner) {
            if (tid < NPC_SLICE) {
                for (int w = 0; w < warp; ++w) {
                    c_in += S.wtot[w][0];
                    q_in += S.wtot[w][1];
                }
                bool is_last;
                const double g = g_at(owner * NPC_SLICE + tid, c_before + c_in, q_before + q_in, &is_last);
                if (g >= 0.0 || is_last) atomicMin(&S.found, owner * NPC_SLICE + tid);
            }
            __syncthreads();
            const int j = S.found;  // (always set: the last bin of the slice qualifies by the choice of the owner)
            if (tid == j - owner * NPC_SLICE) {
                unsigned long long off_lo = ((unsigned long long)j) << shift;
                unsigned long long off_hi = ((unsigned long long)(j + 1)) << shift;
                if (off_hi > width || (shift > 0 && (off_hi >> shift) != (unsigned long long)(j + 1))) off_hi = width;
                s->lo = lo + (long long)off_lo;
                s->hi = lo + (long long)off_hi;
                s->sel_cnt = (long long)c_bin;
                s->level += 1;
                if (c_bin == 0u || off_hi - off_lo <= 1ull) {
                    s->status = NPD_LOCATED;  // dropped = {key <= lo}; the next pass sums them
                } else {
                    npd_set_level(s, NPC_BIN_BITS);
                }
            }
            __syncthreads();
            // the new state into every CTA's copy (8-byte slots)
            constexpr int SLOTS = (int)(sizeof(NpdState) / 8);
            if (tid < NPC_CTAS * SLOTS && tid / SLOTS != owner)
                reinterpret_cast<long long*>(cluster.map_shared_rank(s, tid / SLOTS))[tid % SLOTS] =
                    reinterpret_cast<const long long*>(s)[tid % SLOTS];
        }
        cluster.sync();  // new state everywhere
    }
    // apply
    const int status = (int)s->status;
    if (status == NPD_SOLVED || (status == NPD_IDENTITY && acc > 0.0)) {
        const long long lo = status == NPD_SOLVED ? s->lo : (long long)0x8000000000000000ull;
        const double shift_val = status == NPD_SOLVED ? s->shift_val : 0.0;
#pragma unroll
        for (int j = 0; j < NPC_VPT; ++j) {
            const unsigned long long i = base + (unsigned long long)j * NPC_THREADS;
            if (i < n) p[i] = ((alive >> j & 1u) && npd_key(v[j]) > lo) ? v[j] + shift_val : 0.0;
        }
    }
    if (rank == 0 && tid < (int)(sizeof(NpdState) / 8) && tid != 17)  // (slot 17 = the ticket of the staged kernels)
        reinterpret_cast<long long*>(ws_raw)[tid] = reinterpret_cast<const long long*>(s)[tid];
    cluster.sync();  // no CTA leaves while its shared memory may still be read
}

// ------------------------------------------------------------------ host side
// (4 elements per thread.  Fewer, fatter CTAs - 32 per thread, 8 CTAs at n = 2^16 - measured slower: every
// pass is latency bound, 0.087 -> 0.121 ms for the eight launches of hwe-16 d5's npd.)
static int npd_grid(qck_handle* h, unsigned long long n) {
    unsigned long long want = (n + NPD_THREADS * 4 - 1) / (NPD_THREADS * 4);
    unsigned long long cap = (unsigned long long)h->sm_count * 8;
    if (cap > NPD_GRID_MAX) cap = NPD_GRID_MAX;
    return (int)(want < cap ? (want ? want : 1) : cap);
}

int qck_npd_init(qck_handle* h) {
    QCK_CUDA(h, cudaFuncSetAttribute(npd_hist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 12 * NPD_BINS));
    QCK_CUDA(h, cudaFuncSetAttribute(npd_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(NpcShared)));
    QCK_CUDA(h, cudaMalloc(&h->npd_ws, NPD_WS_BYTES));
    QCK_CUDA(h, cudaMemset(h->npd_ws, 0, NPD_WS_BYTES));
    return QCK_OK;
}

extern "C" size_t qck_npd_workspace_bytes(void) { return NPD_WS_BYTES; }

extern "C" int qck_npd_stage(qck_handle* h, int stage, double* d_p, uint64_t n, double acc, void* d_ws, int fuse_tail,
                             qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    if (!d_p && n > 0 && (stage == QCK_NPD_STATS || stage == QCK_NPD_LEVEL || stage == QCK_NPD_APPLY))
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "NULL argument");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    void* ws = d_ws ? d_ws : h->npd_ws;
    const int grid = npd_grid(h, n);
    switch (stage) {
        case QCK_NPD_STATS: npd_stats_kernel<<<grid, NPD_THREADS, 0, st>>>(d_p, n, acc, ws, fuse_tail); break;
        case QCK_NPD_PLAN: npd_plan_kernel<<<1, NPD_THREADS, 0, st>>>(ws); break;
        case QCK_NPD_LEVEL: npd_hist_kernel<<<grid, NPD_THREADS, 12 * NPD_BINS, st>>>(d_p, n, acc, ws, fuse_tail); break;
        case QCK_NPD_SELECT: npd_select_kernel<<<1, NPD_THREADS, 0, st>>>(ws); break;
        case QCK_NPD_APPLY: npd_apply_kernel<<<grid, NPD_THREADS, 0, st>>>(d_p, n, acc, ws); break;
        default: QCK_FAIL(h, QCK_ERR_INVALID_ARG, "unknown npd stage %d", stage);
    }
    QCK_CHECK_LAUNCH(h);
    return QCK_OK;
}

extern "C" int qck_npd_async(qck_handle* h, double* d_p, uint64_t n, double acc, void* d_ws, qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    if (!d_p && n > 0) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "NULL argument");
    // n <= 2^16: one launch of one 8-CTA cluster, the vector in registers, bins in (distributed) shared memory
    // (QCK_NPD_CLUSTER=0: the staged launches below)
    const char* cluster_env = getenv("QCK_NPD_CLUSTER");
    if (n <= NPC_CAPACITY && !(cluster_env && atoi(cluster_env) == 0)) {
        DeviceGuard guard(h->device);
        void* ws = d_ws ? d_ws : h->npd_ws;
        npd_cluster_kernel<<<NPC_CTAS, NPC_THREADS, sizeof(NpcShared), (cudaStream_t)stream>>>(d_p, n, acc, ws);
        QCK_CHECK_LAUNCH(h);
        return QCK_OK;
    }
    int rc = qck_npd_stage(h, QCK_NPD_STATS, d_p, n, acc, d_ws, 1, stream);
    for (int l = 0; l <= NPD_LEVELS && !rc; ++l) rc = qck_npd_stage(h, QCK_NPD_LEVEL, d_p, n, acc, d_ws, 1, stream);
    if (!rc) rc = qck_npd_stage(h, QCK_NPD_APPLY, d_p, n, acc, d_ws, 1, stream);
    return rc;
}

extern "C" int qck_npd(qck_handle* h, double* d_p, uint64_t n, double acc, double* host_beta, double* host_num,
                       qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    if (!d_p) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "NULL argument");
    int rc = qck_npd_async(h, d_p, n, acc, nullptr, stream);
    if (rc) return rc;
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    NpdState* hs = reinterpret_cast<NpdState*>(h->h_pinned);
    QCK_CUDA(h, cudaMemcpyAsync(hs, h->npd_ws, sizeof(NpdState), cudaMemcpyDeviceToHost, st));
    QCK_CUDA(h, cudaStreamSynchronize(st));
    if (hs->status == NPD_NEGATIVE_TOTAL)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "nearest_probability_distribution: total mass %.3e is negative", hs->sum);
    if (hs->status != NPD_IDENTITY && hs->status != NPD_SOLVED)
        QCK_FAIL(h, QCK_ERR_CUDA, "nearest_probability_distribution: threshold search did not finish (status %lld)",
                 hs->status);
    if (host_beta) *host_beta = hs->beta;
    if (host_num) *host_num = hs->num;
    return QCK_OK;
}

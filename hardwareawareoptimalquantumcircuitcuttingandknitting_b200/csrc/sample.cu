// Finite-shot sampling of fragment-table rows (qck_rows_sample): a multinomial of `shots` over every row, drawn as
// a descent of binomial splits down the row's pairwise sum tree (the definition is in qck.h; tests/
// sampling_reference.py restates it in numpy, bit for bit).
//
// The tree is cut into tiles of 2^12 leaves.  A row of 2^m columns, m <= 13, is one tile: one CTA per row holds its
// whole sum tree in shared memory and descends it.  A wider row is a pyramid: level 0 is the row, level L + 1 holds
// the sums of the 2^12-entry tiles of level L (sp_up_kernel: the row is read once), until a level of <= 2^13
// entries, which is one tile.  The descent (sp_down_kernel) then walks the levels top down; a tile whose count is 0
// is not read again, so a 2^32-entry row with 20 000 shots costs about one read of the row.
//
// Every draw takes its random numbers from Philox4x32-10 at a counter made of (stream id, row label, tree level,
// node index, call index): the counts depend on nothing else (not on the CTA mapping, the launch or the rank).
// This file is compiled with -fmad=false: the binomial sampler's arithmetic must round as the restatement does.
#include "qck_common.cuh"

int qck_ensure_scratch(qck_handle* h, size_t bytes, void** out);  // api.cu

#define SP_THREADS 512
#define SP_TILE_BITS 12        // tile of a pyramid level
#define SP_SINGLE_BITS 13      // widest row (and top level) that is one tile
#define SP_ST_ENTRY 1ull       // an entry is negative, NaN or infinite
#define SP_ST_TOTAL 2ull       // a row total is not > 0 or not finite

// The uniforms of one node's draw: Philox call t gives two, (w0, w1) then (w2, w3) (qck_uniform).
struct NodeRng {
    uint32_t c0, c1, c2, c3, k0, k1;
    uint32_t w[4];
    int used;  // uniforms taken so far
    __device__ NodeRng(unsigned long long seed, uint32_t stream_id, uint32_t row_label, int level,
                       unsigned long long node)
        : c0((uint32_t)node), c1((uint32_t)(node >> 32) | ((uint32_t)level << 16)), c2(row_label),
          c3(stream_id << 20), k0((uint32_t)seed), k1((uint32_t)(seed >> 32)), used(0) {}
    __device__ double uniform() {
        const int half = used & 1;
        if (!half) philox4x32_10(c0, c1, c2, c3 + (uint32_t)(used >> 1), k0, k1, w);
        ++used;
        return qck_uniform(w[2 * half], w[2 * half + 1]);
    }
};

// ---------------------------------------------------------------------------------------------------- binomial
// ATen's sample_binomial (Distributions.h: inversion below count * prob = 10, else BTRS; prob > 1/2 by symmetry).
__constant__ double sp_tail[10] = {0.0810614667953272,  0.0413406959554092,  0.0276779256849983,
                                   0.02079067210376509, 0.0166446911898211,  0.0138761288230707,
                                   0.0118967099458917,  0.0104112652619720,  0.00925546218271273,
                                   0.00833056343336287};
__device__ double sp_stirling_tail(double k) {
    if (k < 10.0) return sp_tail[(int)k];
    const double kp1sq = (k + 1) * (k + 1);
    return (1.0 / 12 - (1.0 / 360 - 1.0 / 1260 / kp1sq) / kp1sq) / (k + 1);
}

__device__ double sp_inversion(double count, double prob, NodeRng& rng) {
    double geom_sum = 0.0, num_geom = 0.0;
    const double logprob = log1p(-prob);
    while (true) {
        const double U = rng.uniform();
        const double geom = ceil(log(U) / logprob);
        geom_sum += geom;
        if (geom_sum > count) break;
        num_geom = num_geom + 1;
    }
    return num_geom;
}

__device__ double sp_btrs(double count, double prob, NodeRng& rng) {
    const double stddev = sqrt(count * prob * (1 - prob));
    const double b = 1.15 + 2.53 * stddev;
    const double a = -0.0873 + 0.0248 * b + 0.01 * prob;
    const double c = count * prob + 0.5;
    const double v_r = 0.92 - 4.2 / b;
    const double r = prob / (1 - prob);
    const double alpha = (2.83 + 5.1 / b) * stddev;
    const double m = floor((count + 1) * prob);
    while (true) {
        const double U = rng.uniform() - 0.5;
        double V = rng.uniform();
        const double us = 0.5 - fabs(U);
        const double k = floor((2 * a / us + b) * U + c);
        if (k < 0 || k > count) continue;
        if (us >= 0.07 && V <= v_r) return k;
        V = log(V * alpha / (a / (us * us) + b));
        const double upperbound = ((m + 0.5) * log((m + 1) / (r * (count - m + 1))) +
                                   (count + 1) * log((count - m + 1) / (count - k + 1)) +
                                   (k + 0.5) * log(r * (count - k + 1) / (k + 1)) + sp_stirling_tail(m) +
                                   sp_stirling_tail(count - m) - sp_stirling_tail(k) - sp_stirling_tail(count - k));
        if (V <= upperbound) return k;
    }
}

// B(count, prob) for 0 < prob < 1 (the caller handles prob = 0 and prob = 1 without a draw)
__device__ long long sp_binomial(long long n, double prob, NodeRng& rng) {
    const double count = (double)n;
    if (prob <= 0.5) {
        if (count * prob >= 10.0) return (long long)sp_btrs(count, prob, rng);
        return (long long)sp_inversion(count, prob, rng);
    }
    const double q = 1.0 - prob;
    if (count * q >= 10.0) return n - (long long)sp_btrs(count, q, rng);
    return n - (long long)sp_inversion(count, q, rng);
}

// ---------------------------------------------------------------------------------------------------- kernels
struct SampleParams {
    const double* in;               // level 0: the table
    long long n_rows, row_stride;
    int m_bits;
    long long shots;
    unsigned long long seed;
    uint32_t stream_id;
    long long row_label_begin;
    double* out;                    // table output (may be null)
    long long out_row_stride;
    int fold_bits;
    long long* shot_list;           // [n_rows][shots] (may be null)
    unsigned long long* status;
    // pyramid: level L >= 1 has 2^lvl_bits[L] entries per row; sums, counts and shot offsets in scratch
    int n_levels;                   // top level index
    int lvl_bits[4];
    double* sums[4];
    int* cnt[4];
    long long* off[4];
};

// Sums of the 2^12-entry tiles of level L -> level L + 1.  Thread e adds its 8 consecutive entries pairwise in
// registers, the warp its 32 partial sums, warp 0 the 16 warp sums: the pairing of the definition throughout.
__global__ void __launch_bounds__(SP_THREADS) sp_up_kernel(const __grid_constant__ SampleParams P, int L) {
    __shared__ double s[SP_THREADS / 16];
    const int bits = L == 0 ? P.m_bits : P.lvl_bits[L];
    const long long tiles_per_row = 1ll << (bits - SP_TILE_BITS);
    const long long n_tiles = P.n_rows * tiles_per_row;
    const double* base = L == 0 ? P.in : P.sums[L];
    const long long stride = L == 0 ? P.row_stride : (1ll << bits);
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long r = tile / tiles_per_row, t = tile - r * tiles_per_row;
        const double2* src = reinterpret_cast<const double2*>(base + r * stride + (t << SP_TILE_BITS)) + 4 * threadIdx.x;
        const double2 a = __ldcs(src), b = __ldcs(src + 1), c = __ldcs(src + 2), d = __ldcs(src + 3);
        if (L == 0) {
            bool bad = false;
            const double v[8] = {a.x, a.y, b.x, b.y, c.x, c.y, d.x, d.y};
#pragma unroll
            for (int i = 0; i < 8; ++i) bad |= !(v[i] >= 0.0) || isinf(v[i]);
            if (bad) atomicOr(P.status, SP_ST_ENTRY);
        }
        // xor butterflies add the pairs of the definition (a + b == b + a exactly): lane sums of 2^5 partials
        double v = ((a.x + a.y) + (b.x + b.y)) + ((c.x + c.y) + (d.x + d.y));
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0) s[SP_THREADS / 32 + (threadIdx.x >> 5)] = v;
        __syncthreads();
        if (threadIdx.x < 32) {
            for (int d0 = SP_THREADS / 64; d0 >= 1; d0 >>= 1) {
                if (threadIdx.x < d0) s[d0 + threadIdx.x] = s[2 * (d0 + threadIdx.x)] + s[2 * (d0 + threadIdx.x) + 1];
                __syncwarp();
            }
        }
        if (threadIdx.x == 0) P.sums[L + 1][(r << (bits - SP_TILE_BITS)) + t] = s[1];
        __syncthreads();
    }
}

// Block-wide exclusive scan of one int per thread (the partial sums are < 2^31: the total is `shots`).
__device__ int sp_block_exclusive_scan(int v, int* warp_tot) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_tot[warp] = x;
    __syncthreads();
    if (warp == 0) {
        int w = lane < SP_THREADS / 32 ? warp_tot[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += y;
        }
        if (lane < SP_THREADS / 32) warp_tot[lane] = w;
    }
    __syncthreads();
    const int before = warp ? warp_tot[warp - 1] : 0;
    __syncthreads();
    return before + x - v;
}

// One tile of level L per CTA iteration: its sum tree in shared memory (heap order: node k has children 2k, 2k + 1,
// leaves at 2^b + x), the count of its root from the level above (`shots` at the top), the descent, then the
// children's counts and shot offsets (L > 0) or the outputs (L = 0).
__global__ void __launch_bounds__(SP_THREADS) sp_down_kernel(const __grid_constant__ SampleParams P, int L) {
    extern __shared__ double sm[];
    __shared__ int warp_tot[SP_THREADS / 32];
    __shared__ int bad_row;
    const bool top = L == P.n_levels;
    const int bits = L == 0 ? P.m_bits : P.lvl_bits[L];
    const int b = top ? bits : SP_TILE_BITS;
    const int nleaf = 1 << b;
    double* s = sm;                                       // [2 * nleaf]
    int* cnt = reinterpret_cast<int*>(sm + 2 * nleaf);    // [2 * nleaf]
    const long long tiles_per_row = 1ll << (bits - b);
    const long long n_tiles = P.n_rows * tiles_per_row;
    const int jL = SP_TILE_BITS * L;
    const int fb = P.fold_bits, xb = P.m_bits - P.fold_bits;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long r = tile / tiles_per_row, t = tile - r * tiles_per_row;
        const long long gidx = (r << (bits - b)) + t;     // this tile's entry at level L + 1
        const long long c = top ? P.shots : (long long)P.cnt[L + 1][gidx];
        const long long off0 = top ? 0 : P.off[L + 1][gidx];
        if (c == 0) {                                     // not read again: zero children / zero output columns
            for (int x = threadIdx.x; x < nleaf; x += SP_THREADS) {
                if (L > 0) P.cnt[L][(gidx << b) + x] = 0;
                else if (P.out && fb == 0) P.out[r * P.out_row_stride + (t << b) + x] = 0.0;
            }
            continue;
        }
        const double* src = L == 0 ? P.in + r * P.row_stride + (t << b) : P.sums[L] + (gidx << b);
        bool bad = false;
        for (int x = threadIdx.x; x < nleaf; x += SP_THREADS) {
            const double v = L == 0 ? __ldcs(src + x) : src[x];
            if (L == 0 && top) bad |= !(v >= 0.0) || isinf(v);
            s[nleaf + x] = v;
        }
        if (bad) atomicOr(P.status, SP_ST_ENTRY);
        __syncthreads();
        for (int d = b - 1; d >= 0; --d) {
            for (int k = (1 << d) + threadIdx.x; k < (2 << d); k += SP_THREADS) s[k] = s[2 * k] + s[2 * k + 1];
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            bad_row = top && !(s[1] > 0.0 && !isinf(s[1]));
            if (bad_row) atomicOr(P.status, SP_ST_TOTAL);
            cnt[1] = bad_row ? 0 : (int)c;
        }
        __syncthreads();
        const uint32_t label = (uint32_t)(P.row_label_begin + r);
        for (int d = 0; d < b; ++d) {
            const int h = b - d;
            for (int k = (1 << d) + threadIdx.x; k < (2 << d); k += SP_THREADS) {
                const int cc = cnt[k];
                int left = 0;
                if (cc > 0) {
                    const double p = s[2 * k] / s[k];
                    if (!(p > 0.0)) left = 0;                 // also NaN (rows the status flags)
                    else if (!(p < 1.0)) left = cc;
                    else {
                        NodeRng rng(P.seed, P.stream_id, label, jL + h, ((unsigned long long)t << d) + (k - (1 << d)));
                        left = (int)sp_binomial(cc, p, rng);
                    }
                }
                cnt[2 * k] = left;
                cnt[2 * k + 1] = cc - left;
            }
            __syncthreads();
        }
        // shot offsets of the leaves: exclusive scan over contiguous chunks of leaves per thread
        const int per = nleaf > SP_THREADS ? nleaf / SP_THREADS : 1;
        const int x0 = threadIdx.x * per;
        int local = 0;
        if (x0 < nleaf)
            for (int i = 0; i < per; ++i) local += cnt[nleaf + x0 + i];
        long long o = off0 + sp_block_exclusive_scan(local, warp_tot);
        if (x0 < nleaf) {
            for (int i = 0; i < per; ++i) {
                const int x = x0 + i;
                const int k = cnt[nleaf + x];
                if (L > 0) {
                    P.cnt[L][(gidx << b) + x] = k;
                    P.off[L][(gidx << b) + x] = o;
                } else {
                    const long long col = (t << b) + x;
                    if (P.shot_list)
                        for (int q = 0; q < k; ++q) P.shot_list[r * P.shots + o + q] = col;
                    if (P.out && fb == 0) {
                        P.out[r * P.out_row_stride + col] = (double)k / (double)P.shots;
                    } else if (P.out && !top && k) {           // folded pyramid row: integer accumulation
                        const long long signed_k = (__popcll((unsigned long long)col >> xb) & 1) ? -k : k;
                        atomicAdd(reinterpret_cast<unsigned long long*>(P.out + r * P.out_row_stride) +
                                      (col & ((1ll << xb) - 1)), (unsigned long long)signed_k);
                    }
                }
                o += k;
            }
        }
        if (L == 0 && top && P.out && fb > 0) {          // folded single-tile row: fold the counts here
            __syncthreads();
            for (int x = threadIdx.x; x < (1 << xb); x += SP_THREADS) {
                long long acc = 0;
                for (int cf = 0; cf < (1 << fb); ++cf) {
                    const int k = cnt[nleaf + x + (cf << xb)];
                    acc += (__popc(cf) & 1) ? -k : k;
                }
                P.out[r * P.out_row_stride + x] = (double)acc / (double)P.shots;
            }
        }
        __syncthreads();
    }
}

// folded pyramid rows: zero the integer accumulators before the descent, turn them into count / shots after it
__global__ void sp_fold_zero_kernel(double* out, long long n_rows, long long stride, int xb) {
    const long long n = n_rows << xb;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        reinterpret_cast<long long*>(out)[(i >> xb) * stride + (i & ((1ll << xb) - 1))] = 0;
}
__global__ void sp_fold_finish_kernel(double* out, long long n_rows, long long stride, int xb, long long shots) {
    const long long n = n_rows << xb;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        double* p = out + (i >> xb) * stride + (i & ((1ll << xb) - 1));
        *p = (double)*reinterpret_cast<long long*>(p) / (double)shots;
    }
}

static int sp_grid(const qck_handle* h, long long work, int per_sm) {
    const long long cap = (long long)h->sm_count * per_sm;
    return (int)(work < 1 ? 1 : work < cap ? work : cap);
}

extern "C" int qck_rows_sample(qck_handle* h, const double* d_in, int64_t n_rows, int64_t row_stride, int m_bits,
                               int64_t shots, uint64_t seed, uint32_t stream_id, int64_t row_label_begin,
                               double* d_out, int64_t out_row_stride, int fold_bits, int64_t* d_shot_list,
                               uint64_t* d_status, qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    if (!d_in || !d_status || (!d_out && !d_shot_list)) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "NULL argument");
    if (m_bits < 0 || m_bits > QCK_MAX_OUT_BITS) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "m_bits=%d out of range", m_bits);
    if (fold_bits < 0 || fold_bits > m_bits) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "fold_bits=%d out of range", fold_bits);
    if (n_rows < 0) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_rows=%lld", (long long)n_rows);
    if (shots < 1 || shots > INT32_MAX) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "shots=%lld: need 1 <= shots < 2^31", (long long)shots);
    if (stream_id >= (1u << 12)) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "stream_id=%u: need < 4096", stream_id);
    if (row_label_begin < 0 || row_label_begin + n_rows > (1ll << 32))
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "row labels [%lld, %lld) outside [0, 2^32)", (long long)row_label_begin,
                 (long long)(row_label_begin + n_rows));
    if (n_rows > 1 && row_stride < (1ll << m_bits))
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "row stride shorter than a row of 2^%d columns", m_bits);
    if (d_out && n_rows > 1 && out_row_stride < (1ll << (m_bits - fold_bits)))
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "output row stride shorter than a row of 2^%d columns", m_bits - fold_bits);
    if (m_bits > SP_SINGLE_BITS && ((uintptr_t)d_in & 15 || row_stride & 1))
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "rows wider than 2^%d columns must start 16-byte aligned", SP_SINGLE_BITS);
    if (n_rows == 0) return QCK_OK;
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    SampleParams P;
    memset(&P, 0, sizeof(P));
    P.in = d_in;
    P.n_rows = n_rows;
    P.row_stride = row_stride;
    P.m_bits = m_bits;
    P.shots = shots;
    P.seed = seed;
    P.stream_id = stream_id;
    P.row_label_begin = row_label_begin;
    P.out = d_out;
    P.out_row_stride = out_row_stride;
    P.fold_bits = d_out ? fold_bits : 0;
    P.shot_list = (long long*)d_shot_list;
    P.status = (unsigned long long*)d_status;
    // pyramid levels: 2^m, 2^(m-12), ... until one of <= 2^13 entries
    int bits = m_bits, L = 0;
    size_t scratch_bytes = 0;
    size_t level_off[4] = {0, 0, 0, 0};
    while (bits > SP_SINGLE_BITS) {
        bits -= SP_TILE_BITS;
        ++L;
        P.lvl_bits[L] = bits;
        level_off[L] = scratch_bytes;
        scratch_bytes += (size_t)n_rows << bits << 4;      // sums (8 B) + offsets (8 B)
        scratch_bytes += (((size_t)n_rows << bits << 2) + 255) & ~(size_t)255;   // counts (4 B)
    }
    P.n_levels = L;
    if (L > 0) {
        void* scratch = nullptr;
        int rc = qck_ensure_scratch(h, scratch_bytes, &scratch);
        if (rc) return rc;
        for (int l = 1; l <= L; ++l) {
            char* base = (char*)scratch + level_off[l];
            const size_t n = (size_t)n_rows << P.lvl_bits[l];
            P.sums[l] = (double*)base;
            P.off[l] = (long long*)(base + 8 * n);
            P.cnt[l] = (int*)(base + 16 * n);
        }
    }
    const int xb = m_bits - P.fold_bits;
    const bool fold_pyramid = d_out && P.fold_bits > 0 && L > 0;
    if (fold_pyramid) {
        sp_fold_zero_kernel<<<sp_grid(h, ((long long)n_rows << xb) / 256 + 1, 8), 256, 0, st>>>(d_out, n_rows,
                                                                                               out_row_stride, xb);
        QCK_CHECK_LAUNCH(h);
    }
    for (int l = 0; l < L; ++l) {
        const int lb = l == 0 ? m_bits : P.lvl_bits[l];
        sp_up_kernel<<<sp_grid(h, (long long)n_rows << (lb - SP_TILE_BITS), 4), SP_THREADS, 0, st>>>(P, l);
        QCK_CHECK_LAUNCH(h);
    }
    for (int l = L; l >= 0; --l) {
        const int lb = l == 0 ? m_bits : P.lvl_bits[l];
        const int b = l == L ? lb : SP_TILE_BITS;
        const size_t smem = (size_t)12 << (b + 1);
        if (smem > 48 * 1024) QCK_CUDA(h, cudaFuncSetAttribute(sp_down_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                                 (int)smem));
        const int per_sm = smem <= 24 * 1024 ? 4 : smem <= 100 * 1024 ? 2 : 1;
        sp_down_kernel<<<sp_grid(h, (long long)n_rows << (lb - b), per_sm), SP_THREADS, smem, st>>>(P, l);
        QCK_CHECK_LAUNCH(h);
    }
    if (fold_pyramid) {
        sp_fold_finish_kernel<<<sp_grid(h, ((long long)n_rows << xb) / 256 + 1, 8), 256, 0, st>>>(
            d_out, n_rows, out_row_stride, xb, shots);
        QCK_CHECK_LAUNCH(h);
    }
    return QCK_OK;
}

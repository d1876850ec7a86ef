// Observables straight from the fragment tables (observables.py), without the dense 2^n_out distribution.
//
//   rows_wht      out[r][s] = sum_x in[r][x] (-1)^popcount(x & s)           (HBM / L2 bound: m adds per entry)
//   rows_marginal out[r][c] = sum_{x : pext(x, keep) = c} in[r][x]           (one read of the table)
//   knit_terms    out[p] = sum_l w(l) prod_f T_f[lf(l)][cols[f][p]]          (gathers from L2-resident tables)
//
// The knit is linear in every fragment table and the fragments' output masks are disjoint, so <Z_S> is the label sum
// of products of per-fragment Walsh-Hadamard entries, a probability out[y] the same sum of table entries, and a
// marginal the dense knit of the tables with the other columns summed out.  Every sum runs in a fixed order: results
// are deterministic.
#include "qck_common.cuh"

int qck_ensure_scratch(qck_handle* h, size_t bytes, void** out);  // api.cu
int qck_contract_prep(qck_handle* h, int n_frag, int n_digits, const int32_t* radix, const double* coef,
                      const int32_t* frag_stride, long long l_begin, long long count, double* d_w, int* d_rows,
                      cudaStream_t st);  // knit.cu

#define OB_THREADS 256
#define OB_TILE_BITS 12                                 // on-chip tile: 4096 doubles = 32 KiB
#define OB_ITEMS ((1 << OB_TILE_BITS) / OB_THREADS)     // entries per thread
#define OB_RUN_BITS 6                                   // global passes: runs of 64 doubles = 512 bytes
#define OB_GROUP_BITS 6                                 // bits transformed per global pass

// ====================================================================== Walsh-Hadamard transform
// The low min(m, 12) bits of every row: one 4096-entry tile per CTA, which is one row, a 4096-column segment of a
// longer row, or 2^(12-m) short rows.  Entry e of the tile is v[i] of thread e & 255 with i = e >> 8: bits 0-4 of
// the column are lanes (shuffle butterflies), bits 8-11 are register indices (butterflies inside a thread), bits 5-7
// go through shared memory.  Stages on different bits commute; their order here is fixed.
__global__ void __launch_bounds__(OB_THREADS) rows_wht_tile_kernel(const double* __restrict__ in, long long n_rows,
                                                                   long long row_stride, int m_bits,
                                                                   double* __restrict__ out, long long out_row_stride) {
    __shared__ double s[1 << OB_TILE_BITS];
    const int tb = m_bits < OB_TILE_BITS ? m_bits : OB_TILE_BITS;  // bits transformed here
    const int hb = m_bits - tb;                                     // 2^hb segments per row
    const long long n_seg = n_rows << hb;
    const long long seg0 = (long long)blockIdx.x << (OB_TILE_BITS - tb);
    const int tid = threadIdx.x, lane = tid & 31;
    const long long seg_mask = (1ll << hb) - 1;
    double v[OB_ITEMS];
#pragma unroll
    for (int i = 0; i < OB_ITEMS; ++i) {
        const int e = tid + i * OB_THREADS;
        const long long q = seg0 + (e >> tb);
        v[i] = 0.0;
        if (q < n_seg) v[i] = __ldg(in + (q >> hb) * row_stride + ((q & seg_mask) << tb) + (e & ((1 << tb) - 1)));
    }
#pragma unroll
    for (int b = 0; b < 5; ++b) {
        if (b < tb) {
            const bool upper = (lane >> b) & 1;
#pragma unroll
            for (int i = 0; i < OB_ITEMS; ++i) {
                const double o = __shfl_xor_sync(0xffffffffu, v[i], 1 << b);
                v[i] = upper ? o - v[i] : v[i] + o;
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (8 + j < tb) {
#pragma unroll
            for (int i = 0; i < OB_ITEMS; ++i) {
                if (!((i >> j) & 1)) {
                    const double a = v[i], c = v[i | (1 << j)];
                    v[i] = a + c;
                    v[i | (1 << j)] = a - c;
                }
            }
        }
    }
    if (tb > 5) {
#pragma unroll
        for (int i = 0; i < OB_ITEMS; ++i) s[tid + i * OB_THREADS] = v[i];
        __syncthreads();
        for (int b = 5; b < 8 && b < tb; ++b) {
            for (int p = tid; p < (1 << (OB_TILE_BITS - 1)); p += OB_THREADS) {
                const uint32_t e0 = insert_zero((uint32_t)p, b), e1 = e0 | (1u << b);
                const double a = s[e0], c = s[e1];
                s[e0] = a + c;
                s[e1] = a - c;
            }
            __syncthreads();
        }
#pragma unroll
        for (int i = 0; i < OB_ITEMS; ++i) v[i] = s[tid + i * OB_THREADS];
    }
#pragma unroll
    for (int i = 0; i < OB_ITEMS; ++i) {
        const int e = tid + i * OB_THREADS;
        const long long q = seg0 + (e >> tb);
        if (q < n_seg) out[(q >> hb) * out_row_stride + ((q & seg_mask) << tb) + (e & ((1 << tb) - 1))] = v[i];
    }
}

// Bits [lo, lo + g) of every row, in place (lo >= 12, g <= 6): a tile is 2^g runs of 64 contiguous doubles (the
// column bits 0-5), one run per value of the group bits; the other column bits number the tiles.
__global__ void __launch_bounds__(OB_THREADS) rows_wht_pass_kernel(double* __restrict__ out, long long n_rows,
                                                                   long long row_stride, int m_bits, int lo, int g) {
    __shared__ double s[1 << (OB_RUN_BITS + OB_GROUP_BITS)];
    const int n = 1 << (OB_RUN_BITS + g);
    const int mid = lo - OB_RUN_BITS;               // tile bits below the group
    const int rest = m_bits - OB_RUN_BITS - g;      // tile bits per row
    const long long tiles = n_rows << rest;
    for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
        const long long r = t >> rest, u = t & ((1ll << rest) - 1);
        double* base = out + r * row_stride + ((u & ((1ll << mid) - 1)) << OB_RUN_BITS) + ((u >> mid) << (lo + g));
        for (int e = threadIdx.x; e < n; e += OB_THREADS)
            s[e] = base[(e & ((1 << OB_RUN_BITS) - 1)) + ((long long)(e >> OB_RUN_BITS) << lo)];
        __syncthreads();
        for (int b = OB_RUN_BITS; b < OB_RUN_BITS + g; ++b) {
            for (int p = threadIdx.x; p < (n >> 1); p += OB_THREADS) {
                const uint32_t e0 = insert_zero((uint32_t)p, b), e1 = e0 | (1u << b);
                const double a = s[e0], c = s[e1];
                s[e0] = a + c;
                s[e1] = a - c;
            }
            __syncthreads();
        }
        for (int e = threadIdx.x; e < n; e += OB_THREADS)
            base[(e & ((1 << OB_RUN_BITS) - 1)) + ((long long)(e >> OB_RUN_BITS) << lo)] = s[e];
        __syncthreads();
    }
}

static int grid_for(const qck_handle* h, long long work) {
    const long long cap = (long long)h->sm_count * 8;
    return (int)(work < 1 ? 1 : work < cap ? work : cap);
}

extern "C" int qck_rows_wht(qck_handle* h, const double* d_in, int64_t n_rows, int64_t row_stride, int m_bits,
                            double* d_out, int64_t out_row_stride, qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    if (!d_in || !d_out) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "NULL argument");
    if (m_bits < 0 || m_bits > QCK_MAX_OUT_BITS) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "m_bits=%d out of range", m_bits);
    if (n_rows < 0) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_rows=%lld", (long long)n_rows);
    if (n_rows > 1 && (row_stride < (1ll << m_bits) || out_row_stride < (1ll << m_bits)))
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "row strides shorter than a row of 2^%d columns", m_bits);
    if (n_rows == 0) return QCK_OK;
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    const int tb = m_bits < OB_TILE_BITS ? m_bits : OB_TILE_BITS;
    const long long n_seg = (long long)n_rows << (m_bits - tb);
    const long long per_cta = 1ll << (OB_TILE_BITS - tb);
    rows_wht_tile_kernel<<<(unsigned)((n_seg + per_cta - 1) / per_cta), OB_THREADS, 0, st>>>(
        d_in, n_rows, row_stride, m_bits, d_out, out_row_stride);
    QCK_CHECK_LAUNCH(h);
    // the bits above the tile: as few global passes as groups of <= 6 bits allow, of near-equal width
    const int rest = m_bits - tb;
    const int passes = (rest + OB_GROUP_BITS - 1) / OB_GROUP_BITS;
    int lo = tb;
    for (int p = 0; p < passes; ++p) {
        const int g = (rest - (lo - tb)) / (passes - p);
        rows_wht_pass_kernel<<<grid_for(h, (long long)n_rows << (m_bits - OB_RUN_BITS - g)), OB_THREADS, 0, st>>>(
            d_out, n_rows, out_row_stride, m_bits, lo, g);
        QCK_CHECK_LAUNCH(h);
        lo += g;
    }
    return QCK_OK;
}

// ====================================================================== marginal
// One read of the table, any row length.  A warp reads 32 consecutive entries: the lb = min(m, 5) low column bits
// are lanes (with m < 5 the lanes above them are 32 >> m consecutive rows).  A GROUP = (row block, value c_hi of the
// kept column bits above the lanes); the wpg warps of a group walk disjoint consecutive ranges of the summed bits
// above the lanes in ascending order, then the summed lane bits are added with butterflies and the warps' sums in
// warp order.
struct MarginalParams {
    const double* in;
    double* out;
    long long n_rows, row_stride;
    int m_bits, lb, k_lo, k_hi, wpg_log;
    unsigned long long keep_hi, sum_hi;  // over the column bits above the lanes
    unsigned keep_lo;
    long long per_warp;                  // summed values each warp of a group walks
    long long n_groups;
};

__device__ __forceinline__ unsigned long long next_subset(unsigned long long x, unsigned long long mask) {
    return ((x | ~mask) + 1ull) & mask;
}

__global__ void __launch_bounds__(OB_THREADS) rows_marginal_kernel(const __grid_constant__ MarginalParams P) {
    __shared__ double part[OB_THREADS / 32][32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int gpc = (OB_THREADS / 32) >> P.wpg_log;  // groups per CTA
    const int wig = warp & ((1 << P.wpg_log) - 1);   // warp in group
    const int rows_per_warp_log = 5 - P.lb;
    const long long hi_count = 1ll << P.k_hi;
    const unsigned lane_col = lane & ((1u << P.lb) - 1u);
    for (long long g0 = (long long)blockIdx.x * gpc; g0 < P.n_groups; g0 += (long long)gridDim.x * gpc) {
        const long long grp = g0 + (warp >> P.wpg_log);
        double acc = 0.0;
        long long row = -1;
        if (grp < P.n_groups) {
            const long long rb = grp / hi_count, c_hi = grp - rb * hi_count;
            row = (rb << rows_per_warp_log) + (lane >> P.lb);
            if (row < P.n_rows) {
                const double* src = P.in + row * P.row_stride + lane_col;
                const unsigned long long kept = soft_pdep((unsigned long long)c_hi, P.keep_hi);
                unsigned long long s = soft_pdep((unsigned long long)(wig * P.per_warp), P.sum_hi);
#pragma unroll 4
                for (long long i = 0; i < P.per_warp; ++i) {
                    acc += __ldg(src + ((long long)(kept | s) << P.lb));
                    s = next_subset(s, P.sum_hi);
                }
            }
        }
        for (int b = 0; b < P.lb; ++b)
            if (!((P.keep_lo >> b) & 1u)) acc += __shfl_xor_sync(0xffffffffu, acc, 1 << b);
        part[warp][lane] = acc;
        __syncthreads();
        if (wig == 0 && grp < P.n_groups && row < P.n_rows && (lane_col & ~P.keep_lo) == 0) {
            double sum = part[warp][lane];
            for (int w = 1; w < (1 << P.wpg_log); ++w) sum += part[warp + w][lane];
            const long long c_hi = grp % hi_count;
            const long long c = (c_hi << P.k_lo) | (long long)soft_pext(lane_col, P.keep_lo);
            P.out[(row << (P.k_lo + P.k_hi)) + c] = sum;
        }
        __syncthreads();
    }
}

extern "C" int qck_rows_marginal(qck_handle* h, const double* d_in, int64_t n_rows, int64_t row_stride, int m_bits,
                                 uint64_t keep_mask, double* d_out, qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    if (!d_in || !d_out) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "NULL argument");
    if (m_bits < 0 || m_bits > QCK_MAX_OUT_BITS) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "m_bits=%d out of range", m_bits);
    if (n_rows < 0) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_rows=%lld", (long long)n_rows);
    if (keep_mask >> m_bits) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "keep_mask has bits >= m_bits");
    if (n_rows > 1 && row_stride < (1ll << m_bits))
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "row stride shorter than a row of 2^%d columns", m_bits);
    if (n_rows == 0) return QCK_OK;
    DeviceGuard guard(h->device);
    MarginalParams P;
    memset(&P, 0, sizeof(P));
    P.in = d_in;
    P.out = d_out;
    P.n_rows = n_rows;
    P.row_stride = row_stride;
    P.m_bits = m_bits;
    P.lb = m_bits < 5 ? m_bits : 5;
    P.keep_lo = (unsigned)(keep_mask & ((1ull << P.lb) - 1ull));
    P.keep_hi = keep_mask >> P.lb;
    P.sum_hi = ((1ull << (m_bits - P.lb)) - 1ull) & ~P.keep_hi;
    P.k_lo = __builtin_popcount(P.keep_lo);
    P.k_hi = __builtin_popcountll(P.keep_hi);
    const int s_bits = __builtin_popcountll(P.sum_hi);
    P.wpg_log = s_bits < 3 ? s_bits : 3;  // up to the 8 warps of a CTA share one group
    P.per_warp = 1ll << (s_bits - P.wpg_log);
    const long long row_blocks = (n_rows + (32 >> P.lb) - 1) / (32 >> P.lb);
    P.n_groups = row_blocks << P.k_hi;
    const long long gpc = (OB_THREADS / 32) >> P.wpg_log;
    rows_marginal_kernel<<<grid_for(h, (P.n_groups + gpc - 1) / gpc), OB_THREADS, 0, (cudaStream_t)stream>>>(P);
    QCK_CHECK_LAUNCH(h);
    return QCK_OK;
}

// ====================================================================== label sum at given columns
// Grid (term blocks, label splits): thread p of a block walks the labels of its split once, the weights and the row
// offsets staged in shared memory 256 labels at a time; the splits' partial sums are added in split order.
#define OB_LABELS 256
struct TermsParams {
    int n_frag;
    const double* table[QCK_MAX_FRAGMENTS];
    long long row_stride[QCK_MAX_FRAGMENTS];
    const int64_t* cols;  // [n_frag][n_terms]
    long long n_terms, count;
    const double* w;      // [count]
    const int* rows;      // [n_frag][count]
    double* partial;      // [n_split][n_terms]; with one split the output itself
    int n_split;
};

__global__ void __launch_bounds__(OB_THREADS) knit_terms_kernel(const __grid_constant__ TermsParams P) {
    __shared__ double sw[OB_LABELS];
    __shared__ long long soff[QCK_MAX_FRAGMENTS][OB_LABELS];
    const long long p = (long long)blockIdx.x * OB_THREADS + threadIdx.x;
    const long long per = (P.count + P.n_split - 1) / P.n_split;
    const long long lb = per * blockIdx.y, le = lb + per < P.count ? lb + per : P.count;
    const double* base[QCK_MAX_FRAGMENTS];
#pragma unroll
    for (int f = 0; f < QCK_MAX_FRAGMENTS; ++f)
        base[f] = (f < P.n_frag && p < P.n_terms) ? P.table[f] + __ldg(P.cols + f * P.n_terms + p) : nullptr;
    double acc = 0.0;
    for (long long l0 = lb; l0 < le; l0 += OB_LABELS) {
        const int n = (int)(le - l0 < OB_LABELS ? le - l0 : OB_LABELS);
        __syncthreads();
        for (int j = threadIdx.x; j < n; j += OB_THREADS) {
            sw[j] = __ldg(P.w + l0 + j);
            for (int f = 0; f < P.n_frag; ++f) soff[f][j] = (long long)__ldg(P.rows + f * P.count + l0 + j) * P.row_stride[f];
        }
        __syncthreads();
        if (p < P.n_terms) {
            for (int j = 0; j < n; ++j) {
                double t = sw[j];
#pragma unroll
                for (int f = 0; f < QCK_MAX_FRAGMENTS; ++f)
                    if (f < P.n_frag) t *= __ldg(base[f] + soff[f][j]);
                acc += t;
            }
        }
    }
    if (p < P.n_terms) P.partial[(long long)blockIdx.y * P.n_terms + p] = acc;
}

__global__ void __launch_bounds__(OB_THREADS) knit_terms_sum_kernel(const double* __restrict__ partial, int n_split,
                                                                    long long n_terms, double* __restrict__ out) {
    for (long long p = (long long)blockIdx.x * OB_THREADS + threadIdx.x; p < n_terms;
         p += (long long)gridDim.x * OB_THREADS) {
        double acc = 0.0;
        for (int s = 0; s < n_split; ++s) acc += partial[(long long)s * n_terms + p];
        out[p] = acc;
    }
}

extern "C" int qck_knit_terms(qck_handle* h, int n_frag, const double* const* d_tables, const int64_t* row_strides,
                              int n_digits, const int32_t* radix, const double* coef, const int32_t* frag_stride,
                              int64_t n_terms, const int64_t* d_cols, double* d_out, qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    if (n_frag < 1 || n_frag > QCK_MAX_FRAGMENTS) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_frag=%d out of range", n_frag);
    if (n_digits < 0 || n_digits > QCK_MAX_DIGITS) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_digits=%d out of range", n_digits);
    if (!d_tables || !row_strides || (n_terms > 0 && (!d_cols || !d_out)) ||
        (n_digits > 0 && (!radix || !coef || !frag_stride)))
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "NULL argument");
    if (n_terms < 0) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_terms=%lld", (long long)n_terms);
    long long count = 1;
    for (int k = 0; k < n_digits; ++k) {
        if (radix[k] < 1 || radix[k] > QCK_MAX_VARIANTS) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "radix[%d]=%d", k, radix[k]);
        count *= radix[k];
    }
    for (int f = 0; f < n_frag; ++f) {
        if (!d_tables[f]) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "table %d is NULL", f);
        if (row_strides[f] < 1) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "row_strides[%d]=%lld", f, (long long)row_strides[f]);
    }
    if (n_terms == 0) return QCK_OK;
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    const long long term_blocks = (n_terms + OB_THREADS - 1) / OB_THREADS;
    // about four CTAs per SM, at least 32 labels per split
    long long n_split = ((long long)h->sm_count * 4 + term_blocks - 1) / term_blocks;
    const long long max_split = (count + 31) / 32;
    if (n_split > max_split) n_split = max_split;
    if (n_split > 1024) n_split = 1024;
    if (n_split < 1) n_split = 1;
    const size_t w_bytes = ((size_t)count * sizeof(double) + 255) & ~(size_t)255;
    const size_t r_bytes = ((size_t)count * n_frag * sizeof(int) + 255) & ~(size_t)255;
    const size_t p_bytes = n_split > 1 ? (size_t)n_split * n_terms * sizeof(double) : 0;
    void* scratch = nullptr;
    int rc = qck_ensure_scratch(h, w_bytes + r_bytes + p_bytes, &scratch);
    if (rc) return rc;
    double* d_w = (double*)scratch;
    int* d_rows = (int*)((char*)scratch + w_bytes);
    rc = qck_contract_prep(h, n_frag, n_digits, radix, coef, frag_stride, 0, count, d_w, d_rows, st);
    if (rc) return rc;
    TermsParams P;
    memset(&P, 0, sizeof(P));
    P.n_frag = n_frag;
    for (int f = 0; f < n_frag; ++f) {
        P.table[f] = d_tables[f];
        P.row_stride[f] = row_strides[f];
    }
    P.cols = d_cols;
    P.n_terms = n_terms;
    P.count = count;
    P.w = d_w;
    P.rows = d_rows;
    P.partial = n_split > 1 ? (double*)((char*)scratch + w_bytes + r_bytes) : d_out;
    P.n_split = (int)n_split;
    knit_terms_kernel<<<dim3((unsigned)term_blocks, (unsigned)n_split), OB_THREADS, 0, st>>>(P);
    QCK_CHECK_LAUNCH(h);
    if (n_split > 1) {
        knit_terms_sum_kernel<<<grid_for(h, term_blocks), OB_THREADS, 0, st>>>(P.partial, (int)n_split, n_terms, d_out);
        QCK_CHECK_LAUNCH(h);
    }
    return QCK_OK;
}

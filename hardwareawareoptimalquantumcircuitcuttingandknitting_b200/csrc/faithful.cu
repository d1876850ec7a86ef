// Reference-faithful knit (ACCURACY > 0) as one fused evaluation per output bitstring.
//
// The reference prunes |v| <= ACCURACY after EVERY QuasiDistr operation
// (third_party/qvm/qvm/quasi_distr.py:3,7-10): from_counts, each merge fold
// (virtual_circuit.py:216-228), each half of split, and every + / - / scalar * of the per-gate
// knit formulas (virtual_gates.py:105-124,179-194,262-286), which are evaluated left to right, one
// virtual gate per level from the last to the first (virtual_circuit.py:59-68).  All of it is
// elementwise in the output bitstring x: the value of level k at (x, config bits c_0..c_{k-1}) is a
// fixed expression of the level-(k+1) values of its n_k children at c_k = 0 and 1.  So instead of
// materialising 2^(n_cl+K)-entry dictionaries per label, every thread evaluates that expression
// tree for its own x by recursion over the label digits, reading the UNFOLDED fragment tables
// (config bits kept as extra row bits).  Subtrees with c_k = 1 under a variant that measures
// nothing are identically zero and are skipped.
//
// Parallelism: level 0 is split off - one thread per (x, variant of gate 0, c_0) evaluates the
// subtree below it, a second small kernel applies gate 0's formula.
#include "qck_common.cuh"

#define FA_MAXF QCK_MAX_FRAGMENTS
#define FA_MAXK QCK_MAX_DIGITS
#define FA_MAXV QCK_MAX_VARIANTS

struct FaithParams {
    int n_frag, K, n_out_bits;
    const double* table[FA_MAXF];
    unsigned long long mask[FA_MAXF];
    long long row_stride[FA_MAXF];
    int m_bits[FA_MAXF];
    int radix[FA_MAXK];
    int form[FA_MAXK];                  // 0: signed chain (move / cz / cx / cy), 1: rzz family
    int degenerate[FA_MAXK];            // rzz: 0 full, 1: |cos| < eps -> r * sin^2, 2: |sin| < eps -> r * cos^2
    double sign[FA_MAXK][FA_MAXV];      // chain: +1 / -1 per variant
    double c1[FA_MAXK], s1[FA_MAXK];    // rzz: cos(m/2), sin(m/2)
    double c2[FA_MAXK], s2[FA_MAXK];    // rzz: cos^2, sin^2 (as Python's ** 2)
    int frag_stride[FA_MAXF][FA_MAXK];  // fragment label = sum_k digit_k * stride
    long long row_step[FA_MAXF][FA_MAXK];  // frag_stride * row_stride: table offset per unit of digit k
    int cfg_bit[FA_MAXF][FA_MAXK];      // position of gate k's config bit among f's extra row bits, -1: untouched
    unsigned char measures[FA_MAXF][FA_MAXK][FA_MAXV];  // does f's instance measure gate k under variant v
    unsigned char any_measure[FA_MAXK][FA_MAXV];
    double acc;
    int part, n_parts;  // this call evaluates part `part` of `n_parts` of the outputs (the others stay +0)
};

__device__ __forceinline__ double prn(double v, double acc) { return fabs(v) > acc ? v : 0.0; }

struct EvalCtx {
    const FaithParams* P;
    unsigned long long xf[FA_MAXF];  // x restricted to each fragment's output bits (compact)
    long long off[FA_MAXF];          // table offset of the fragment's row under the current digits
    unsigned long long cf[FA_MAXF];  // config bits of the fragment's row index under the current path
    int d[FA_MAXK];
};

// the path below gate k takes variant i with config bit `bit`: row offsets and config bits follow incrementally
// (recomputing them at every leaf - K multiply-adds per fragment - was most of the leaf's cost)
__device__ __forceinline__ void enter(EvalCtx& C, int k, int i, int bit) {
    const FaithParams& P = *C.P;
    const int delta = i - C.d[k];
    C.d[k] = i;
    for (int f = 0; f < P.n_frag; ++f) {
        C.off[f] += (long long)delta * P.row_step[f][k];
        if (bit && P.cfg_bit[f][k] >= 0 && P.measures[f][k][i]) C.cf[f] |= 1ull << P.cfg_bit[f][k];
    }
}
__device__ __forceinline__ void leave(EvalCtx& C, int k, int bit) {
    const FaithParams& P = *C.P;
    if (bit)
        for (int f = 0; f < P.n_frag; ++f)
            if (P.cfg_bit[f][k] >= 0) C.cf[f] &= ~(1ull << P.cfg_bit[f][k]);
}

// merged_l(x, c): left fold over the fragments of prune(p_f) with a prune after each product.  (A config bit is
// only ever set under a variant that measures it somewhere - knit_formula skips the other children - so no leaf
// needs the "does anybody measure this bit" test.)
__device__ __forceinline__ double leaf(EvalCtx& C) {
    const FaithParams& P = *C.P;
    double v = 0.0;
    for (int f = 0; f < P.n_frag; ++f) {
        const double pf = prn(__ldg(P.table[f] + C.off[f] + (C.xf[f] | (C.cf[f] << P.m_bits[f]))), P.acc);
        v = f == 0 ? pf : prn(v * pf, P.acc);
    }
    return v;
}

__device__ double eval(EvalCtx& C, int k);

// apply gate k's knit formula given a functor child(i, bit) -> level-(k+1) value
template <typename Child>
__device__ __forceinline__ double knit_formula(const FaithParams& P, int k, Child child) {
    const double acc = P.acc;
    if (P.form[k] == 0) {
        double total = 0.0;
        for (int i = 0; i < P.radix[k]; ++i) {
            const double r0 = prn(child(i, 0), acc);
            const double r1 = P.any_measure[k][i] ? prn(child(i, 1), acc) : 0.0;
            const double diff = prn(r0 - r1, acc);
            total = i == 0 ? diff : prn(P.sign[k][i] > 0.0 ? total + diff : total - diff, acc);
        }
        return prn(0.5 * total, acc);
    }
    if (P.degenerate[k] == 1) return prn(prn(child(0, 0), acc) * P.s2[k], acc);
    if (P.degenerate[k] == 2) return prn(prn(child(0, 0), acc) * P.c2[k], acc);
    const double r0 = prn(child(0, 0), acc), r1 = prn(child(1, 0), acc);
    const double r23_0 = prn(child(2, 0) + child(3, 0), acc);
    const double r23_1 = prn((P.any_measure[k][2] ? child(2, 1) : 0.0) + (P.any_measure[k][3] ? child(3, 1) : 0.0), acc);
    const double r45_0 = prn(child(4, 0) + child(5, 0), acc);
    const double r45_1 = prn((P.any_measure[k][4] ? child(4, 1) : 0.0) + (P.any_measure[k][5] ? child(5, 1) : 0.0), acc);
    const double mixed = prn(prn(prn(r23_0 - r23_1, acc) - r45_0, acc) + r45_1, acc);
    const double head = prn(prn(r0 * P.c2[k], acc) + prn(r1 * P.s2[k], acc), acc);
    return prn(head + prn(prn(mixed * P.c1[k], acc) * P.s1[k], acc), acc);
}

__device__ double eval(EvalCtx& C, int k) {
    const FaithParams& P = *C.P;
    if (k == P.K) return leaf(C);
    return knit_formula(P, k, [&](int i, int bit) {
        enter(C, k, i, bit);
        const double v = eval(C, k + 1);
        leave(C, k, bit);
        return v;
    });
}

__device__ __forceinline__ void init_ctx(EvalCtx& C, const FaithParams& P, unsigned long long x) {
    C.P = &P;
    for (int f = 0; f < P.n_frag; ++f) C.xf[f] = soft_pext(x, P.mask[f]), C.off[f] = 0, C.cf[f] = 0;
    for (int k = 0; k < FA_MAXK; ++k) C.d[k] = 0;
}

// stage 1: scratch[(i * 2 + bit) << n_out | x] = level-1 value under gate 0's variant i, c_0 = bit
__global__ void __launch_bounds__(128) faith_subtree_kernel(const __grid_constant__ FaithParams P,
                                                            double* __restrict__ scratch) {
    const unsigned long long n = 1ull << P.n_out_bits;
    const unsigned long long x0 = n / P.n_parts * P.part, x1 = P.part + 1 == P.n_parts ? n : n / P.n_parts * (P.part + 1);
    const unsigned long long total = n * (unsigned long long)(2 * P.radix[0]);
    for (unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long x = t & (n - 1);
        if (x < x0 || x >= x1) continue;
        const int j = (int)(t >> P.n_out_bits), i = j >> 1, bit = j & 1;
        double v = 0.0;
        if (!bit || P.any_measure[0][i]) {
            EvalCtx C;
            init_ctx(C, P, x);
            enter(C, 0, i, bit);
            v = eval(C, 1);
        }
        scratch[t] = v;
    }
}

// stage 2: gate 0's formula over the stored subtrees
__global__ void __launch_bounds__(256) faith_top_kernel(const __grid_constant__ FaithParams P,
                                                        const double* __restrict__ scratch, double* __restrict__ out) {
    const unsigned long long n = 1ull << P.n_out_bits;
    const unsigned long long x0 = n / P.n_parts * P.part, x1 = P.part + 1 == P.n_parts ? n : n / P.n_parts * (P.part + 1);
    for (unsigned long long x = x0 + (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; x < x1;
         x += (unsigned long long)gridDim.x * blockDim.x)
        out[x] = knit_formula(P, 0, [&](int i, int bit) { return scratch[((unsigned long long)(2 * i + bit) << P.n_out_bits) | x]; });
}

// no virtual gates: the pruned merge only
__global__ void __launch_bounds__(256) faith_leaf_kernel(const __grid_constant__ FaithParams P, double* __restrict__ out) {
    const unsigned long long n = 1ull << P.n_out_bits;
    const unsigned long long x0 = n / P.n_parts * P.part, x1 = P.part + 1 == P.n_parts ? n : n / P.n_parts * (P.part + 1);
    for (unsigned long long x = x0 + (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; x < x1;
         x += (unsigned long long)gridDim.x * blockDim.x) {
        EvalCtx C;
        init_ctx(C, P, x);
        out[x] = leaf(C);
    }
}

// ---- sparsity: the reference's dictionaries simply do not hold pruned entries (quasi_distr.py:7-10), which is
// where its speed on concentrated distributions (hwe) comes from.  Dense counterpart: a leaf is a pruned product
// with one factor per fragment taken from COLUMN pext(x, mask_f) of that fragment's table, so when a column holds
// no entry above the threshold in any row (any label, any config bits) every leaf under x is 0 and so is every
// level above it (each formula maps zeros to +0).  The alive columns of every fragment are listed once; the
// expression trees are evaluated only for the product set of the lists, the other outputs are +0 from a memset.
struct AliveParams {
    int n_frag;
    const double* table[FA_MAXF];
    long long n_rows[FA_MAXF], row_stride[FA_MAXF];
    int m_bits[FA_MAXF];
    unsigned* flags[FA_MAXF];  // [2^m_bits], zeroed
    double acc;
};

__global__ void __launch_bounds__(256) faith_alive_kernel(const __grid_constant__ AliveParams A) {
    const int f = blockIdx.y;
    if (f >= A.n_frag) return;
    const long long total = A.n_rows[f] * A.row_stride[f];
    const long long cmask = (1ll << A.m_bits[f]) - 1;
    const double* __restrict__ t = A.table[f];
    unsigned* __restrict__ fl = A.flags[f];
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x)
        if (fabs(__ldg(t + e)) > A.acc) {
            const long long col = (e % A.row_stride[f]) & cmask;
            if (!fl[col]) fl[col] = 1u;  // every writer stores the same value
        }
}

// ascending list of the set flags + their number (one CTA per fragment: the order is fixed)
__global__ void __launch_bounds__(1024) faith_compact_kernel(const __grid_constant__ AliveParams A, int* __restrict__ lists,
                                                             long long list_stride, int* __restrict__ counts) {
    __shared__ int warp_tot[32];
    __shared__ int base;
    const int f = blockIdx.x;
    const long long n_cols = 1ll << A.m_bits[f];
    const unsigned* fl = A.flags[f];
    int* list = lists + f * list_stride;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    for (long long c0 = 0; c0 < n_cols; c0 += blockDim.x) {
        const long long c = c0 + threadIdx.x;
        const int on = (c < n_cols && fl[c]) ? 1 : 0;
        const unsigned ballot = __ballot_sync(0xffffffffu, on);
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        if (lane == 0) warp_tot[warp] = __popc(ballot);
        __syncthreads();
        int before = base;
        for (int w = 0; w < warp; ++w) before += warp_tot[w];
        if (on) list[before + __popc(ballot & ((1u << lane) - 1u))] = (int)c;
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = 0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += warp_tot[w];
            base += t;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) counts[f] = base;
}

struct SparseCtx {
    const int* lists;
    long long list_stride;
    const int* counts;
};

// j-th element of the product set -> x and the per-fragment columns
__device__ __forceinline__ unsigned long long alive_point(const FaithParams& P, const SparseCtx& S, unsigned long long j,
                                                          EvalCtx& C) {
    unsigned long long x = 0;
    C.P = &P;
    for (int f = 0; f < P.n_frag; ++f) {
        const unsigned long long cnt = (unsigned long long)S.counts[f];
        const unsigned long long col = (unsigned long long)S.lists[f * S.list_stride + (long long)(j % cnt)];
        j /= cnt;
        C.xf[f] = col;
        C.off[f] = 0;
        C.cf[f] = 0;
        unsigned long long m = P.mask[f], src = col;  // deposit the column's bits at the mask's positions
        while (m) {
            const unsigned long long low = m & (~m + 1ull);
            if (src & 1ull) x |= low;
            src >>= 1;
            m ^= low;
        }
    }
    for (int k = 0; k < FA_MAXK; ++k) C.d[k] = 0;
    return x;
}
__device__ __forceinline__ unsigned long long alive_total(const FaithParams& P, const SparseCtx& S) {
    unsigned long long t = 1;
    for (int f = 0; f < P.n_frag; ++f) t *= (unsigned long long)S.counts[f];
    return t;
}

__global__ void __launch_bounds__(128) faith_subtree_sparse_kernel(const __grid_constant__ FaithParams P, const SparseCtx S,
                                                                   double* __restrict__ scratch) {
    const unsigned long long all = alive_total(P, S);
    const unsigned long long j0 = all / P.n_parts * P.part, j1 = P.part + 1 == P.n_parts ? all : all / P.n_parts * (P.part + 1);
    const unsigned long long alive = j1 - j0;
    const unsigned long long total = alive * (unsigned long long)(2 * P.radix[0]);
    for (unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (unsigned long long)gridDim.x * blockDim.x) {
        const int j = (int)(t / alive), i = j >> 1, bit = j & 1;
        EvalCtx C;
        const unsigned long long x = alive_point(P, S, j0 + t % alive, C);
        double v = 0.0;
        if (!bit || P.any_measure[0][i]) {
            enter(C, 0, i, bit);
            v = eval(C, 1);
        }
        scratch[((unsigned long long)j << P.n_out_bits) | x] = v;
    }
}

// Two levels split off (K >= 2): one thread per (alive entry, variant and config bit of gate 0, of gate 1).  A
// concentrated distribution leaves few alive entries (hwe-16 d5: a few hundred) and 2 * n_0 subtrees per entry are
// too few threads for 148 SMs - the evaluation then lasts as long as ONE thread's walk over the other K - 1 levels.
__global__ void __launch_bounds__(128) faith_subtree2_sparse_kernel(const __grid_constant__ FaithParams P, const SparseCtx S,
                                                                    double* __restrict__ scratch2) {
    const unsigned long long all = alive_total(P, S);
    const unsigned long long j0 = all / P.n_parts * P.part, j1 = P.part + 1 == P.n_parts ? all : all / P.n_parts * (P.part + 1);
    const unsigned long long alive = j1 - j0;
    const int w0 = 2 * P.radix[0], w1 = 2 * P.radix[1];
    const unsigned long long total = alive * (unsigned long long)(w0 * w1);
    for (unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (unsigned long long)gridDim.x * blockDim.x) {
        const int c = (int)(t / alive), c0 = c / w1, c1 = c % w1;
        const int i0 = c0 >> 1, b0 = c0 & 1, i1 = c1 >> 1, b1 = c1 & 1;
        EvalCtx C;
        const unsigned long long x = alive_point(P, S, j0 + t % alive, C);
        double v = 0.0;
        if ((!b0 || P.any_measure[0][i0]) && (!b1 || P.any_measure[1][i1])) {
            enter(C, 0, i0, b0);
            enter(C, 1, i1, b1);
            v = eval(C, 2);
        }
        scratch2[((unsigned long long)c << P.n_out_bits) | x] = v;
    }
}

// gate 1's formula over the stored subtrees -> the level-1 values the top kernel reads
__global__ void __launch_bounds__(256) faith_mid_sparse_kernel(const __grid_constant__ FaithParams P, const SparseCtx S,
                                                               const double* __restrict__ scratch2, double* __restrict__ scratch) {
    const unsigned long long all = alive_total(P, S);
    const unsigned long long j0 = all / P.n_parts * P.part, j1 = P.part + 1 == P.n_parts ? all : all / P.n_parts * (P.part + 1);
    const unsigned long long alive = j1 - j0;
    const int w0 = 2 * P.radix[0], w1 = 2 * P.radix[1];
    const unsigned long long total = alive * (unsigned long long)w0;
    for (unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (unsigned long long)gridDim.x * blockDim.x) {
        const int c0 = (int)(t / alive), i0 = c0 >> 1, b0 = c0 & 1;
        EvalCtx C;
        const unsigned long long x = alive_point(P, S, j0 + t % alive, C);
        double v = 0.0;
        if (!b0 || P.any_measure[0][i0])
            v = knit_formula(P, 1, [&](int i, int bit) {
                return scratch2[((unsigned long long)(c0 * w1 + 2 * i + bit) << P.n_out_bits) | x];
            });
        scratch[((unsigned long long)c0 << P.n_out_bits) | x] = v;
    }
}

__global__ void __launch_bounds__(256) faith_top_sparse_kernel(const __grid_constant__ FaithParams P, const SparseCtx S,
                                                               const double* __restrict__ scratch, double* __restrict__ out) {
    const unsigned long long all = alive_total(P, S);
    const unsigned long long j0 = all / P.n_parts * P.part, j1 = P.part + 1 == P.n_parts ? all : all / P.n_parts * (P.part + 1);
    for (unsigned long long j = j0 + (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; j < j1;
         j += (unsigned long long)gridDim.x * blockDim.x) {
        EvalCtx C;
        const unsigned long long x = alive_point(P, S, j, C);
        out[x] = knit_formula(P, 0, [&](int i, int bit) { return scratch[((unsigned long long)(2 * i + bit) << P.n_out_bits) | x]; });
    }
}

__global__ void __launch_bounds__(256) faith_leaf_sparse_kernel(const __grid_constant__ FaithParams P, const SparseCtx S,
                                                                double* __restrict__ out) {
    const unsigned long long all = alive_total(P, S);
    const unsigned long long j0 = all / P.n_parts * P.part, j1 = P.part + 1 == P.n_parts ? all : all / P.n_parts * (P.part + 1);
    for (unsigned long long j = j0 + (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; j < j1;
         j += (unsigned long long)gridDim.x * blockDim.x) {
        EvalCtx C;
        const unsigned long long x = alive_point(P, S, j, C);
        out[x] = leaf(C);
    }
}

int qck_ensure_scratch(qck_handle* h, size_t bytes, void** out);  // api.cu

extern "C" int qck_knit_faithful(qck_handle* h, int n_frag, const double* const* d_tables, const uint64_t* masks,
                                 const int64_t* row_strides, int n_out_bits, int n_gates, const qck_faithful_gate* gates,
                                 const int32_t* frag_stride, const int32_t* cfg_bit, const uint8_t* measures,
                                 double accuracy, double* d_out, qck_stream stream) {
    return qck_knit_faithful_part(h, n_frag, d_tables, masks, row_strides, n_out_bits, n_gates, gates, frag_stride, cfg_bit,
                                  measures, accuracy, d_out, 0, 1, stream);
}

extern "C" int qck_knit_faithful_part(qck_handle* h, int n_frag, const double* const* d_tables, const uint64_t* masks,
                                      const int64_t* row_strides, int n_out_bits, int n_gates,
                                      const qck_faithful_gate* gates, const int32_t* frag_stride, const int32_t* cfg_bit,
                                      const uint8_t* measures, double accuracy, double* d_out, int part, int n_parts,
                                      qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    if (n_parts < 1 || n_parts > 64 || part < 0 || part >= n_parts) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "part %d of %d", part, n_parts);
    if (n_frag < 1 || n_frag > FA_MAXF) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_frag=%d out of range", n_frag);
    if (n_gates < 0 || n_gates > FA_MAXK) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_gates=%d out of range", n_gates);
    if (!d_tables || !masks || !row_strides || !d_out || (n_gates > 0 && (!gates || !frag_stride || !cfg_bit || !measures)))
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "NULL argument");
    if (n_out_bits < 0 || n_out_bits > 30) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_out_bits=%d out of range", n_out_bits);
    if (!(accuracy >= 0.0)) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "accuracy must be >= 0");
    FaithParams P;
    memset(&P, 0, sizeof(P));
    P.n_frag = n_frag;
    P.K = n_gates;
    P.n_out_bits = n_out_bits;
    P.acc = accuracy;
    P.part = part;
    P.n_parts = n_parts;
    uint64_t seen = 0;
    for (int f = 0; f < n_frag; ++f) {
        if (!d_tables[f]) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "table %d is NULL", f);
        if (masks[f] & seen) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "fragment masks overlap");
        seen |= masks[f];
        P.table[f] = d_tables[f];
        P.mask[f] = masks[f];
        P.row_stride[f] = row_strides[f];
        P.m_bits[f] = __builtin_popcountll(masks[f]);
    }
    for (int k = 0; k < n_gates; ++k) {
        const qck_faithful_gate& g = gates[k];
        if (g.n_variants < 1 || g.n_variants > FA_MAXV) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "gate %d: n_variants=%d", k, g.n_variants);
        if (g.form != 0 && g.form != 1) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "gate %d: unknown knit form %d", k, g.form);
        if (g.form == 1 && g.degenerate == 0 && g.n_variants != 6)
            QCK_FAIL(h, QCK_ERR_INVALID_ARG, "gate %d: the rzz form needs 6 variants", k);
        P.radix[k] = g.n_variants;
        P.form[k] = g.form;
        P.degenerate[k] = g.degenerate;
        for (int v = 0; v < FA_MAXV; ++v) P.sign[k][v] = g.sign[v];
        P.c1[k] = g.cos_half;
        P.s1[k] = g.sin_half;
        P.c2[k] = g.cos_half_sq;
        P.s2[k] = g.sin_half_sq;
        for (int f = 0; f < n_frag; ++f) {
            P.frag_stride[f][k] = frag_stride[f * FA_MAXK + k];
            P.row_step[f][k] = (long long)frag_stride[f * FA_MAXK + k] * row_strides[f];
            P.cfg_bit[f][k] = cfg_bit[f * FA_MAXK + k];
            for (int v = 0; v < FA_MAXV; ++v) {
                P.measures[f][k][v] = measures[(f * FA_MAXK + k) * FA_MAXV + v];
                P.any_measure[k][v] |= P.measures[f][k][v];
            }
        }
    }
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned long long n = 1ull << n_out_bits;
    int grid = (int)((n + 255) / 256 < (unsigned long long)h->sm_count * 8 ? (n + 255) / 256 : (unsigned long long)h->sm_count * 8);
    // ---- alive columns (accuracy > 0 and the masks cover the output: else every x is evaluated as before)
    const char* sparse_env = getenv("QCK_FAITHFUL_SPARSE");
    const bool sparse = accuracy > 0.0 && seen == (n_out_bits >= 64 ? ~0ull : (1ull << n_out_bits) - 1ull) &&
                        !(sparse_env && atoi(sparse_env) == 0);
    const unsigned long long total = n_gates ? n * (unsigned long long)(2 * P.radix[0]) : 0;
    size_t tree_bytes = (total * sizeof(double) + 255) & ~(size_t)255, flag_bytes = 0, list_bytes = 0;
    // second split level (sparse path): scratch for the (gate 0, gate 1) subtrees, bounded at 1 GiB
    const unsigned long long total2 = n_gates >= 2 ? total * (unsigned long long)(2 * P.radix[1]) : 0;
    const bool split2 = sparse && n_gates >= 2 && total2 * sizeof(double) <= ((size_t)1 << 30);
    const size_t tree1_bytes = tree_bytes;
    if (split2) tree_bytes += (total2 * sizeof(double) + 255) & ~(size_t)255;
    long long list_stride = 0;
    AliveParams A;
    memset(&A, 0, sizeof(A));
    if (sparse) {
        A.n_frag = n_frag;
        A.acc = accuracy;
        for (int f = 0; f < n_frag; ++f) {
            long long rows = 1;
            for (int k = 0; k < n_gates; ++k)
                if (P.frag_stride[f][k] != 0) rows *= P.radix[k];
            A.table[f] = P.table[f];
            A.n_rows[f] = rows;
            A.row_stride[f] = P.row_stride[f];
            A.m_bits[f] = P.m_bits[f];
            flag_bytes += (sizeof(unsigned) << P.m_bits[f]);
            if ((1ll << P.m_bits[f]) > list_stride) list_stride = 1ll << P.m_bits[f];
        }
        flag_bytes = (flag_bytes + 255) & ~(size_t)255;
        list_bytes = ((size_t)list_stride * n_frag * sizeof(int) + 255) & ~(size_t)255;
    }
    void* scratch = nullptr;
    int rc = qck_ensure_scratch(h, tree_bytes + flag_bytes + list_bytes + 256, &scratch);
    if (rc) return rc;
    SparseCtx S;
    memset(&S, 0, sizeof(S));
    if (sparse) {
        char* at = (char*)scratch + tree_bytes;
        QCK_CUDA(h, cudaMemsetAsync(at, 0, flag_bytes, st));
        for (int f = 0; f < n_frag; ++f) {
            A.flags[f] = (unsigned*)at;
            at += sizeof(unsigned) << P.m_bits[f];
        }
        int* lists = (int*)((char*)scratch + tree_bytes + flag_bytes);
        int* counts = (int*)((char*)scratch + tree_bytes + flag_bytes + list_bytes);
        long long most = 0;
        for (int f = 0; f < n_frag; ++f) most = A.n_rows[f] * A.row_stride[f] > most ? A.n_rows[f] * A.row_stride[f] : most;
        long long want_a = (most + 256 * 8 - 1) / (256 * 8);
        dim3 agrid((unsigned)(want_a < (long long)h->sm_count * 8 ? (want_a < 1 ? 1 : want_a) : (long long)h->sm_count * 8), n_frag);
        faith_alive_kernel<<<agrid, 256, 0, st>>>(A);
        QCK_CHECK_LAUNCH(h);
        faith_compact_kernel<<<n_frag, 1024, 0, st>>>(A, lists, list_stride, counts);
        QCK_CHECK_LAUNCH(h);
        S.lists = lists;
        S.list_stride = list_stride;
        S.counts = counts;
    }
    if (sparse || n_parts > 1) QCK_CUDA(h, cudaMemsetAsync(d_out, 0, n * sizeof(double), st));
    if (n_gates == 0) {
        if (sparse) faith_leaf_sparse_kernel<<<grid, 256, 0, st>>>(P, S, d_out);
        else faith_leaf_kernel<<<grid, 256, 0, st>>>(P, d_out);
        QCK_CHECK_LAUNCH(h);
        return QCK_OK;
    }
    // recursion depth <= K: make sure the per-thread stack can hold it
    size_t stack = 0;
    cudaDeviceGetLimit(&stack, cudaLimitStackSize);
    if (stack < 4096) QCK_CUDA(h, cudaDeviceSetLimit(cudaLimitStackSize, 4096));
    unsigned long long want = (total + 127) / 128;
    int sgrid = (int)(want < (unsigned long long)h->sm_count * 32 ? want : (unsigned long long)h->sm_count * 32);
    if (sparse && split2) {
        double* scratch2 = (double*)((char*)scratch + tree1_bytes);
        const unsigned long long want2 = (total2 + 127) / 128;
        const int sgrid2 = (int)(want2 < (unsigned long long)h->sm_count * 32 ? want2 : (unsigned long long)h->sm_count * 32);
        faith_subtree2_sparse_kernel<<<sgrid2, 128, 0, st>>>(P, S, scratch2);
        QCK_CHECK_LAUNCH(h);
        faith_mid_sparse_kernel<<<sgrid, 128 * 2, 0, st>>>(P, S, scratch2, (double*)scratch);
        QCK_CHECK_LAUNCH(h);
        faith_top_sparse_kernel<<<grid, 256, 0, st>>>(P, S, (const double*)scratch, d_out);
        QCK_CHECK_LAUNCH(h);
        return QCK_OK;
    }
    if (sparse) {
        faith_subtree_sparse_kernel<<<sgrid, 128, 0, st>>>(P, S, (double*)scratch);
        QCK_CHECK_LAUNCH(h);
        faith_top_sparse_kernel<<<grid, 256, 0, st>>>(P, S, (const double*)scratch, d_out);
        QCK_CHECK_LAUNCH(h);
        return QCK_OK;
    }
    faith_subtree_kernel<<<sgrid, 128, 0, st>>>(P, (double*)scratch);
    QCK_CHECK_LAUNCH(h);
    faith_top_kernel<<<grid, 256, 0, st>>>(P, (const double*)scratch, d_out);
    QCK_CHECK_LAUNCH(h);
    return QCK_OK;
}

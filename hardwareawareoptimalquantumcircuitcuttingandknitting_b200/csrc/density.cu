// Density-matrix simulation of fragment instances under a noise model (qck_sim_density; the definition is in
// qck.h, the host lowering in density.py).
//
// rho is 2^(2n) complex128 entries, index r | c << n.  Every op is a superoperator (4x4 or 16x16) on positions of a
// tile of 2^n_tile entries.  Two regimes:
//   - 2n <= 12: one sweep, one CTA per work item; rho is built as |0><0| in shared memory, every op runs there and
//     the diagonal is reduced into the item's columns: rho never touches HBM.
//   - 2n > 12: rho lives in the work buffer (as many items as fit).  Each sweep is one launch of one CTA per
//     (item, tile): load the tile (its low 5 bits are contiguous: 512-byte runs), run the sweep's ops, store it.  The
//     first sweep generates |0><0| instead of loading.  A last launch reduces the diagonal (stride 2^n + 1).
// Then one CTA per row applies the readout butterflies to the unfolded row and folds the configuration bits.
#include "qck_common.cuh"

#define DM_THREADS 512
#define DM_OP_INTS 12

struct DmItem {
    unsigned long long digits;
    int label;
    unsigned branch, col_base, qmask;
};
static_assert(sizeof(DmItem) == 24, "qck_dm item layout");

struct DmQcol {
    int v[QCK_DM_MAX_QUBITS];   // row column of each qubit's diagonal bit
};

struct DmTile {
    int n_tile, n_rest;
    int pos[QCK_DM_MAX_TILE_BITS];
    int rest[2 * QCK_DM_MAX_QUBITS];
};

__device__ __forceinline__ double2 cmul_add(double2 acc, double2 a, double2 b) {
    acc.x = fma(a.x, b.x, acc.x);
    acc.x = fma(-a.y, b.y, acc.x);
    acc.y = fma(a.x, b.y, acc.y);
    acc.y = fma(a.y, b.x, acc.y);
    return acc;
}

// ops [b, e) on the tile in shared memory; mat_s: 256 complex of shared memory for the current matrix
__device__ void dm_apply(double2* tile, double2* mat_s, const int* __restrict__ ops, int b, int e,
                         const double2* __restrict__ mats, const DmItem& it, int n_tile) {
    for (int k = b; k < e; ++k) {
        const int* r = ops + DM_OP_INTS * k;
        const int nq = r[0], dig = r[2], br = r[3];
        const int digit = dig >= 0 ? (int)((it.digits >> (4 * dig)) & 15ull) : 0;
        const int bit = br >= 0 ? (int)((it.branch >> br) & 1u) : 0;
        const int msize = nq == 1 ? 16 : 256;
        const double2* m = mats + r[1] + (size_t)msize * (digit * (br >= 0 ? 2 : 1) + bit);
        __syncthreads();                         // the previous op is done with the tile and the matrix
        for (int i = threadIdx.x; i < msize; i += blockDim.x) mat_s[i] = m[i];
        __syncthreads();
        if (nq == 1) {
            const int p0 = r[4], p1 = r[5], s0 = r[8], s1 = r[9];
            const int groups = 1 << (n_tile - 2);
            for (int g = threadIdx.x; g < groups; g += blockDim.x) {
                const uint32_t base = insert_zero(insert_zero((uint32_t)g, s0), s1);
                uint32_t idx[4];
                double2 v[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    idx[j] = base | ((uint32_t)(j & 1) << p0) | ((uint32_t)(j >> 1) << p1);
                    v[j] = tile[idx[j]];
                }
#pragma unroll
                for (int o = 0; o < 4; ++o) {
                    double2 acc = make_double2(0.0, 0.0);
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc = cmul_add(acc, mat_s[4 * o + j], v[j]);
                    tile[idx[o]] = acc;
                }
            }
        } else {
            const int s0 = r[8], s1 = r[9], s2 = r[10], s3 = r[11];
            const int groups = 1 << (n_tile - 4);
            for (int g = threadIdx.x; g < groups; g += blockDim.x) {
                const uint32_t base = insert_zero(insert_zero(insert_zero(insert_zero((uint32_t)g, s0), s1), s2), s3);
                uint32_t idx[16];
                double2 v[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    idx[j] = base | ((uint32_t)(j & 1) << r[4]) | ((uint32_t)((j >> 1) & 1) << r[5]) |
                             ((uint32_t)((j >> 2) & 1) << r[6]) | ((uint32_t)(j >> 3) << r[7]);
                    v[j] = tile[idx[j]];
                }
#pragma unroll 4
                for (int o = 0; o < 16; ++o) {
                    double2 acc = make_double2(0.0, 0.0);
#pragma unroll
                    for (int j = 0; j < 16; ++j) acc = cmul_add(acc, mat_s[16 * o + j], v[j]);
                    tile[idx[o]] = acc;
                }
            }
        }
    }
    __syncthreads();
}

// Column t (of 2^popcount(qmask)) of an item: the sum of Re rho[i][i] over the qubits outside qmask.
__device__ __forceinline__ void dm_column(const double2* rho, int n, const int* qcol, const DmItem& it, uint32_t t,
                                          double* row) {
    const uint32_t full = (1u << n) - 1u;
    const uint32_t keep = it.qmask & full, rest = full & ~keep;
    uint32_t fixed = 0, col = it.col_base, tt = t;
    for (int q = 0; q < n; ++q) {
        if ((keep >> q) & 1u) {
            const uint32_t b = tt & 1u;
            tt >>= 1;
            fixed |= b << q;
            col |= b << qcol[q];
        }
    }
    const int n_rest = __popc(rest);
    const size_t diag = ((size_t)1 << n) + 1;
    double s = 0.0;
    for (uint32_t u = 0; u < (1u << n_rest); ++u) {
        uint32_t i = fixed, uu = u;
        for (int q = 0; q < n; ++q) {
            if ((rest >> q) & 1u) {
                i |= (uu & 1u) << q;
                uu >>= 1;
            }
        }
        s += rho[(size_t)i * diag].x;
    }
    row[col] = s;
}

struct DmRows {
    double* rows;               // unfolded rows
    long long row_stride;
    long long row_label0;       // label of rows[0]
};

__global__ void __launch_bounds__(DM_THREADS) dm_resident_kernel(const int* __restrict__ ops, int n_ops,
                                                                 const double2* __restrict__ mats,
                                                                 const DmItem* __restrict__ items, long long n_items,
                                                                 int n, DmRows R, DmQcol Q) {
    extern __shared__ double2 dm_smem[];
    const int n2 = 2 * n;
    double2* tile = dm_smem;
    double2* mat_s = dm_smem + (1 << n2);
    __shared__ int qcol[QCK_DM_MAX_QUBITS];
    if (threadIdx.x < QCK_DM_MAX_QUBITS) qcol[threadIdx.x] = Q.v[threadIdx.x];
    for (long long w = blockIdx.x; w < n_items; w += gridDim.x) {
        const DmItem it = items[w];
        __syncthreads();
        for (int i = threadIdx.x; i < (1 << n2); i += blockDim.x) tile[i] = make_double2(i == 0 ? 1.0 : 0.0, 0.0);
        dm_apply(tile, mat_s, ops, 0, n_ops, mats, it, n2);
        double* row = R.rows + (it.label - R.row_label0) * R.row_stride;
        const uint32_t cols = 1u << __popc(it.qmask);
        for (uint32_t t = threadIdx.x; t < cols; t += blockDim.x) dm_column(tile, n, qcol, it, t, row);
    }
}

__device__ __forceinline__ size_t dm_global(uint32_t l, unsigned long long t, const DmTile& T) {
    size_t g = l & 31u;                          // pos[k] = k for the low 5 bits
    for (int k = 5; k < T.n_tile; ++k) g |= (size_t)((l >> k) & 1u) << T.pos[k];
    for (int k = 0; k < T.n_rest; ++k) g |= (size_t)((t >> k) & 1ull) << T.rest[k];
    return g;
}

__global__ void __launch_bounds__(DM_THREADS) dm_sweep_kernel(const int* __restrict__ ops, int op_begin, int op_end,
                                                              const double2* __restrict__ mats,
                                                              const DmItem* __restrict__ items, double2* work,
                                                              int n2, DmTile T, int first) {
    extern __shared__ double2 dm_smem[];
    double2* tile = dm_smem;
    double2* mat_s = dm_smem + (1 << T.n_tile);
    const unsigned long long tiles = 1ull << T.n_rest;
    const unsigned long long item = blockIdx.x / tiles, t = blockIdx.x % tiles;
    const DmItem it = items[item];
    double2* rho = work + (item << n2);
    for (uint32_t l = threadIdx.x; l < (1u << T.n_tile); l += blockDim.x) {
        const size_t g = dm_global(l, t, T);
        tile[l] = first ? make_double2(g == 0 ? 1.0 : 0.0, 0.0) : rho[g];
    }
    dm_apply(tile, mat_s, ops, op_begin, op_end, mats, it, T.n_tile);
    for (uint32_t l = threadIdx.x; l < (1u << T.n_tile); l += blockDim.x) rho[dm_global(l, t, T)] = tile[l];
}

__global__ void dm_diag_kernel(const DmItem* __restrict__ items, const double2* __restrict__ work, int n,
                               DmRows R, DmQcol Q, int blocks_per_item) {
    __shared__ int qcol[QCK_DM_MAX_QUBITS];
    if (threadIdx.x < QCK_DM_MAX_QUBITS) qcol[threadIdx.x] = Q.v[threadIdx.x];
    __syncthreads();
    const long long item = blockIdx.x / blocks_per_item;
    const DmItem it = items[item];
    const uint32_t cols = 1u << __popc(it.qmask);
    double* row = R.rows + (it.label - R.row_label0) * R.row_stride;
    const double2* rho = work + ((size_t)item << (2 * n));
    for (uint32_t t = (blockIdx.x % blocks_per_item) * blockDim.x + threadIdx.x; t < cols;
         t += blocks_per_item * blockDim.x)
        dm_column(rho, n, qcol, it, t, row);
}

__global__ void dm_zero_kernel(DmRows R, long long n_rows, int n_cols) {
    const long long total = n_rows << n_cols;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x)
        R.rows[(i >> n_cols) * R.row_stride + (i & ((1ll << n_cols) - 1))] = 0.0;
}

// one CTA per row: readout butterflies on the unfolded row (in place), then the signed fold into d_out
struct DmRadix {
    int n_digits;
    int radix[QCK_MAX_DIGITS];
};

__global__ void dm_finish_kernel(DmRows R, long long label_begin, int n_cols, const uint32_t* __restrict__ ro_mask,
                                 const double* __restrict__ ro, DmRadix D, int fold_bits, double* out,
                                 long long out_stride) {
    const long long label = label_begin + blockIdx.x;
    double* row = R.rows + (label - R.row_label0) * R.row_stride;
    const uint32_t mask = ro_mask[label];
    const int row_bits = n_cols - D.n_digits;
    for (int j = 0; j < n_cols; ++j) {
        if (!((mask >> j) & 1u)) continue;
        int v = 0;                               // a configuration column: the label's digit picks the measuring qubit
        if (j >= row_bits) {
            long long l = label;
            for (int d = D.n_digits - 1; d > j - row_bits; --d) l /= D.radix[d];
            v = (int)(l % D.radix[j - row_bits]);
        }
        const double* rj = ro + 4 * (QCK_MAX_VARIANTS * j + v);
        const double r00 = rj[0], r01 = rj[1], r10 = rj[2], r11 = rj[3];
        for (uint32_t p = threadIdx.x; p < (1u << (n_cols - 1)); p += blockDim.x) {
            const uint32_t i0 = insert_zero(p, j), i1 = i0 | (1u << j);
            const double u0 = row[i0], u1 = row[i1];
            row[i0] = r00 * u0 + r01 * u1;
            row[i1] = r10 * u0 + r11 * u1;
        }
        __syncthreads();
    }
    if (fold_bits == 0) return;
    const int xb = n_cols - fold_bits;
    for (uint32_t x = threadIdx.x; x < (1u << xb); x += blockDim.x) {
        double s = 0.0;
        for (uint32_t c = 0; c < (1u << fold_bits); ++c) {
            const double v = row[x | (c << xb)];
            s += (__popc(c) & 1) ? -v : v;
        }
        out[label * out_stride + x] = s;
    }
}

QCK_API int qck_sim_density(qck_handle* h, const qck_dm_plan* plan, int64_t label_begin, int64_t label_end,
                            double* d_out, int64_t out_row_stride, double* d_rows, void* d_work, size_t work_bytes,
                            qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    if (!plan || !d_out || !plan->sweeps || !plan->item_begin || !plan->d_ops || !plan->d_mats || !plan->d_items ||
        !plan->d_ro_mask || !plan->d_ro)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "NULL argument");
    const int n = plan->n_qubits, n2 = 2 * n;
    if (n < 1 || n > QCK_DM_MAX_QUBITS) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_qubits=%d out of range", n);
    if (plan->n_sweeps < 1) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "a plan needs at least one sweep");
    if (plan->n_cols < 0 || plan->n_cols > 30 || plan->fold_bits < 0 || plan->fold_bits > plan->n_cols)
        QCK_FAIL(h, QCK_ERR_UNSUPPORTED, "row of 2^%d columns (fold %d) out of range", plan->n_cols, plan->fold_bits);
    if (label_begin < 0 || label_begin > label_end || label_end > plan->n_labels)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "label range [%lld, %lld) outside [0, %lld)", (long long)label_begin,
                 (long long)label_end, (long long)plan->n_labels);
    if (plan->n_digits < 0 || plan->n_digits > QCK_MAX_DIGITS || plan->n_digits > plan->n_cols)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_digits=%d out of range", plan->n_digits);
    for (int d = 0; d < plan->n_digits; ++d)
        if (plan->radix[d] < 1 || plan->radix[d] > QCK_MAX_VARIANTS)
            QCK_FAIL(h, QCK_ERR_INVALID_ARG, "radix[%d]=%d out of range", d, plan->radix[d]);
    if (plan->fold_bits > 0 && !d_rows) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "folding needs d_rows");
    if (out_row_stride < (1ll << (plan->n_cols - plan->fold_bits)) && label_end - label_begin > 1)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "output row stride shorter than a row");
    const bool resident = n2 <= QCK_DM_MAX_TILE_BITS;
    if (resident && plan->n_sweeps != 1)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "a plan of %d qubits (2n <= %d) has one sweep, not %d", n,
                 QCK_DM_MAX_TILE_BITS, plan->n_sweeps);
    for (int s = 0; s < plan->n_sweeps; ++s) {
        const qck_dm_sweep& sw = plan->sweeps[s];
        const int want = resident ? n2 : QCK_DM_MAX_TILE_BITS;
        if (sw.n_tile != want || sw.op_begin < 0 || sw.op_end < sw.op_begin)
            QCK_FAIL(h, QCK_ERR_INVALID_ARG, "sweep %d: tile of %d bits, ops [%d, %d)", s, sw.n_tile, sw.op_begin,
                     sw.op_end);
        for (int k = 0; k < sw.n_tile; ++k)
            if ((k < 5 && sw.pos[k] != k) || sw.pos[k] < 0 || sw.pos[k] >= n2 || (k && sw.pos[k] <= sw.pos[k - 1]))
                QCK_FAIL(h, QCK_ERR_INVALID_ARG, "sweep %d: tile positions must ascend from 0..4", s);
    }
    const size_t rho_bytes = (size_t)16 << n2;
    if (!resident && (!d_work || work_bytes < rho_bytes))
        QCK_FAIL(h, QCK_ERR_NOMEM, "the work buffer (%zu bytes) holds no density matrix of %d qubits (%zu bytes)",
                 work_bytes, n, rho_bytes);
    if (label_end == label_begin) return QCK_OK;
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    DmRows R;
    const bool unfolded = d_rows && plan->fold_bits > 0;    // without a fold the rows are d_out's and d_rows is unused
    R.rows = unfolded ? d_rows : d_out;
    R.row_stride = unfolded ? (1ll << plan->n_cols) : out_row_stride;
    R.row_label0 = unfolded ? label_begin : 0;
    const long long n_rows = label_end - label_begin;
    DmRows Z = R;
    Z.rows = R.rows + (label_begin - R.row_label0) * R.row_stride;
    dm_zero_kernel<<<(unsigned)std::min<long long>((n_rows << plan->n_cols) / 256 + 1, (long long)h->sm_count * 16),
                     256, 0, st>>>(Z, n_rows, plan->n_cols);
    QCK_CHECK_LAUNCH(h);
    const int64_t ib = plan->item_begin[label_begin], ie = plan->item_begin[label_end];
    const DmItem* items = (const DmItem*)plan->d_items;
    const double2* mats = (const double2*)plan->d_mats;
    DmQcol Q;
    for (int q = 0; q < QCK_DM_MAX_QUBITS; ++q) Q.v[q] = plan->qcol[q];
    if (ie > ib && resident) {
        const size_t smem = ((size_t)16 << n2) + 256 * 16;
        QCK_CUDA(h, cudaFuncSetAttribute(dm_resident_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const long long grid = std::min<long long>(ie - ib, (long long)h->sm_count * (smem <= 40 * 1024 ? 4 : 2));
        const qck_dm_sweep& sw = plan->sweeps[0];
        dm_resident_kernel<<<(unsigned)grid, DM_THREADS, smem, st>>>(plan->d_ops + DM_OP_INTS * sw.op_begin,
                                                                     sw.op_end - sw.op_begin, mats, items + ib,
                                                                     ie - ib, n, R, Q);
        QCK_CHECK_LAUNCH(h);
    } else if (ie > ib) {
        const size_t smem = ((size_t)16 << QCK_DM_MAX_TILE_BITS) + 256 * 16;
        QCK_CUDA(h, cudaFuncSetAttribute(dm_sweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const long long batch_max = (long long)std::min<size_t>(work_bytes / rho_bytes, (size_t)1 << 20);
        const int n_rest = n2 - QCK_DM_MAX_TILE_BITS;
        const long long per_launch = std::max<long long>(1, std::min<long long>(batch_max, INT32_MAX >> n_rest));
        const int blocks_per_item = (int)std::min<long long>(((1ll << n) + 255) / 256, 1024);
        for (int64_t i0 = ib; i0 < ie; i0 += per_launch) {
            const long long nb = std::min<long long>(per_launch, ie - i0);
            for (int s = 0; s < plan->n_sweeps; ++s) {
                const qck_dm_sweep& sw = plan->sweeps[s];
                DmTile T;
                memset(&T, 0, sizeof(T));
                T.n_tile = sw.n_tile;
                unsigned long long in_tile = 0;
                for (int k = 0; k < sw.n_tile; ++k) {
                    T.pos[k] = sw.pos[k];
                    in_tile |= 1ull << sw.pos[k];
                }
                for (int b = 0; b < n2; ++b)
                    if (!((in_tile >> b) & 1ull)) T.rest[T.n_rest++] = b;
                dm_sweep_kernel<<<(unsigned)(nb << n_rest), DM_THREADS, smem, st>>>(
                    plan->d_ops, sw.op_begin, sw.op_end, mats, items + i0, (double2*)d_work, n2, T, s == 0);
                QCK_CHECK_LAUNCH(h);
            }
            dm_diag_kernel<<<(unsigned)(nb * blocks_per_item), 256, 0, st>>>(items + i0, (const double2*)d_work, n,
                                                                               R, Q, blocks_per_item);
            QCK_CHECK_LAUNCH(h);
        }
    }
    DmRadix D;
    D.n_digits = plan->n_digits;
    for (int d = 0; d < QCK_MAX_DIGITS; ++d) D.radix[d] = d < plan->n_digits ? plan->radix[d] : 1;
    dm_finish_kernel<<<(unsigned)n_rows, 256, 0, st>>>(R, label_begin, plan->n_cols, plan->d_ro_mask, plan->d_ro, D,
                                                       plan->fold_bits, d_out, out_row_stride);
    QCK_CHECK_LAUNCH(h);
    return QCK_OK;
}

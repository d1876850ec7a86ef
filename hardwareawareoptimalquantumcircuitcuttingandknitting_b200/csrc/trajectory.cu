// Noisy shots by quantum trajectories (qck_sim_trajectories; the definition is in qck.h, the host lowering in
// trajectory.py, the numpy restatement in tests/trajectory_reference.py).
//
// One CTA runs one trajectory at a time and grid-strides over the (label, shot) pairs.  psi (2^n complex128) lives in
// shared memory when n <= 13, else in the CTA's slot of the work buffer.  A stochastic op is one reduction pass (the
// op's 2x2 / 4x4 reduced density matrix, a fixed warp-butterfly then warp-order sum) and one apply pass; thread 0
// picks the Kraus operator and keeps the trajectory's column.  The block size depends on n only, so every sum, and
// with it every bit of a trajectory, is the same whatever the grid, the label range or the launch.
#include "qck_common.cuh"

#define TJ_MAX_THREADS 512
#define TJ_RED 16                  // reduced-density-matrix values per warp: 4 diagonal reals + 6 complex pairs

struct TjLabel {
    unsigned long long digits;
    uint32_t qmask, ro_mask;
};
static_assert(sizeof(TjLabel) == 16, "qck_traj label record layout");

struct TjParams {
    const int* ops;
    const int* vars;
    const double2* mats;
    const TjLabel* labels;
    const double* ro;
    int n, n_ops, n_cols, n_digits, fold_bits, term_uidx;
    uint32_t ro_cols;
    int qcol[QCK_DM_MAX_QUBITS];
    long long label_begin, n_traj, shots;
    unsigned long long seed;
    uint32_t stream_id;
    double* out;
    long long out_stride;
    long long* shot_list;
    double2* work;
};

// uniform j of one trajectory: Philox call j >> 1 at counter (shot, label, stream id, j >> 1), half j & 1
struct TjRng {
    uint32_t shot, label, sid, k0, k1;
    int call;
    uint32_t w[4];
    __device__ double uniform(int j) {
        if ((j >> 1) != call) {
            call = j >> 1;
            philox4x32_10(shot, label, sid, (uint32_t)call, k0, k1, w);
        }
        const int h = j & 1;
        return qck_uniform(w[2 * h], w[2 * h + 1]);
    }
};

__host__ __device__ __forceinline__ int tj_threads(int n) {
    return n <= 8 ? 32 : min(TJ_MAX_THREADS, 1 << (n - 3));
}

__device__ __forceinline__ double2 tj_cmul(double2 a, double2 b) {
    return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ double2 tj_cmac(double2 acc, double2 a, double2 b) {
    acc.x = fma(a.x, b.x, acc.x);
    acc.x = fma(-a.y, b.y, acc.x);
    acc.y = fma(a.x, b.y, acc.y);
    acc.y = fma(a.y, b.x, acc.y);
    return acc;
}

// psi <- m psi on the op's qubits (m: d x d in shared memory, row-major [out][in], index bit 0 = q0)
__device__ __forceinline__ void tj_apply(double2* psi, int n, int nq, int q0, int q1, const double2* m) {
    if (nq == 1) {
        const double2 m00 = m[0], m01 = m[1], m10 = m[2], m11 = m[3];
        for (uint32_t g = threadIdx.x; g < (1u << (n - 1)); g += blockDim.x) {
            const uint32_t i0 = insert_zero(g, q0), i1 = i0 | (1u << q0);
            const double2 a = psi[i0], b = psi[i1];
            psi[i0] = tj_cmac(tj_cmul(m00, a), m01, b);
            psi[i1] = tj_cmac(tj_cmul(m10, a), m11, b);
        }
        return;
    }
    const int s0 = min(q0, q1), s1 = max(q0, q1);
    for (uint32_t g = threadIdx.x; g < (1u << (n - 2)); g += blockDim.x) {
        const uint32_t base = insert_zero(insert_zero(g, s0), s1);
        uint32_t idx[4];
        double2 v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            idx[j] = base | ((uint32_t)(j & 1) << q0) | ((uint32_t)(j >> 1) << q1);
            v[j] = psi[idx[j]];
        }
#pragma unroll
        for (int o = 0; o < 4; ++o) {
            double2 acc = tj_cmul(m[4 * o], v[0]);
#pragma unroll
            for (int j = 1; j < 4; ++j) acc = tj_cmac(acc, m[4 * o + j], v[j]);
            psi[idx[o]] = acc;
        }
    }
}

// acc += the reduced-density-matrix terms of amplitudes v[0..d): diagonal |v_a|^2 at [a], then for the pairs a < b
// in order (0,1) (0,2) (0,3) (1,2) (1,3) (2,3): v_a conj(v_b) at [d + 2p], [d + 2p + 1]
template <int D>
__device__ __forceinline__ void tj_rho_terms(const double2* v, double* acc) {
#pragma unroll
    for (int a = 0; a < D; ++a) acc[a] += v[a].x * v[a].x + v[a].y * v[a].y;
    int p = 0;
#pragma unroll
    for (int a = 0; a < D; ++a)
#pragma unroll
        for (int b = a + 1; b < D; ++b, ++p) {
            acc[D + 2 * p] += v[a].x * v[b].x + v[a].y * v[b].y;
            acc[D + 2 * p + 1] += v[a].y * v[b].x - v[a].x * v[b].y;
        }
}

// per-warp partial sums of the op's reduced density matrix -> red[warp][0..TJ_RED)
__device__ __forceinline__ void tj_reduce(const double2* psi, int n, int nq, int q0, int q1, double* red) {
    double acc[TJ_RED];
#pragma unroll
    for (int e = 0; e < TJ_RED; ++e) acc[e] = 0.0;
    if (nq == 1) {
        for (uint32_t g = threadIdx.x; g < (1u << (n - 1)); g += blockDim.x) {
            const uint32_t i0 = insert_zero(g, q0);
            const double2 v[2] = {psi[i0], psi[i0 | (1u << q0)]};
            tj_rho_terms<2>(v, acc);
        }
    } else {
        const int s0 = min(q0, q1), s1 = max(q0, q1);
        for (uint32_t g = threadIdx.x; g < (1u << (n - 2)); g += blockDim.x) {
            const uint32_t base = insert_zero(insert_zero(g, s0), s1);
            double2 v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = psi[base | ((uint32_t)(j & 1) << q0) | ((uint32_t)(j >> 1) << q1)];
            tj_rho_terms<4>(v, acc);
        }
    }
    const int nv = nq == 1 ? 4 : TJ_RED;
#pragma unroll
    for (int e = 0; e < TJ_RED; ++e)
        if (e < nv) acc[e] = warp_sum(acc[e]);
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int e = 0; e < TJ_RED; ++e)
            if (e < nv) red[(threadIdx.x >> 5) * TJ_RED + e] = acc[e];
    }
}

// Re Tr(M rho) from the packed rho of tj_rho_terms (M Hermitian, d x d row-major)
__device__ __forceinline__ double tj_expect(const double2* M, const double* r, int d) {
    double p = 0.0;
    for (int a = 0; a < d; ++a) p += M[a * d + a].x * r[a];
    int q = 0;
    for (int a = 0; a < d; ++a)
        for (int b = a + 1; b < d; ++b, ++q) {
            const double2 m = M[a * d + b];
            p += 2.0 * (m.x * r[d + 2 * q] + m.y * r[d + 2 * q + 1]);
        }
    return fmax(p, 0.0);
}

// Inverse CDF over v[0..cnt) starting from the cumulative `base`: the first i with target < base + v[0] + .. + v[i]
// (sequential sums); base becomes the sum before it.  When rounding leaves no such i, the last entry with mass.
template <typename F>
__device__ __forceinline__ int tj_pick(F v, int cnt, double& base, double target) {
    double acc = base, last_base = base;
    int last = 0;
    for (int i = 0; i < cnt; ++i) {
        const double x = v(i), nb = acc + x;
        if (target < nb) {
            base = acc;
            return i;
        }
        if (x > 0.0) last = i, last_base = acc;
        acc = nb;
    }
    base = last_base;
    return last;
}

template <bool SMEM>
__global__ void __launch_bounds__(TJ_MAX_THREADS) tj_kernel(const __grid_constant__ TjParams P) {
    extern __shared__ double2 tj_smem[];
    __shared__ double2 mat_s[16];
    __shared__ double rsum[TJ_RED];
    const int n = P.n, T = blockDim.x, warps = T >> 5;
    const uint32_t N = 1u << n;
    double2* psi = SMEM ? tj_smem : P.work + ((size_t)blockIdx.x << n);
    double* part = reinterpret_cast<double*>(SMEM ? tj_smem + N : tj_smem);    // [T]
    double* red = part + T;              // [warps][TJ_RED], and the 32 lane sums of the terminal sample
    const int row_bits = P.n_cols - P.n_digits;
    for (long long tr = blockIdx.x; tr < P.n_traj; tr += gridDim.x) {
        const long long li = tr / P.shots, shot = tr - li * P.shots, label = P.label_begin + li;
        const TjLabel L = P.labels[label];
        TjRng rng{(uint32_t)shot, (uint32_t)label, P.stream_id, (uint32_t)P.seed, (uint32_t)(P.seed >> 32), -1, {}};
        uint32_t c = 0;                                  // the trajectory's column (kept by thread 0)
        __syncthreads();                                 // the previous trajectory is done with psi and part
        for (uint32_t i = threadIdx.x; i < N; i += T) psi[i] = make_double2(i == 0 ? 1.0 : 0.0, 0.0);
        for (int k = 0; k < P.n_ops; ++k) {
            const int* r = P.ops + QCK_TRAJ_OP_INTS * k;
            const int nq = r[0], q0 = r[1], q1 = r[2], dig = r[3];
            const int v = dig >= 0 ? (int)((L.digits >> (4 * dig)) & 15ull) : 0;
            const int nk = P.vars[2 * (r[6] + v)];
            if (nk == 0) continue;
            const int d = 1 << nq, dd = d * d;
            const double2* K = P.mats + P.vars[2 * (r[6] + v) + 1];
            __syncthreads();                             // the previous op is done with psi and mat_s
            if (nk == 1) {
                if (threadIdx.x < dd) mat_s[threadIdx.x] = K[threadIdx.x];
            } else {
                tj_reduce(psi, n, nq, q0, q1, red);
                __syncthreads();
                if (threadIdx.x < (nq == 1 ? 4 : TJ_RED)) {      // the values tj_reduce wrote
                    double s = 0.0;
                    for (int w = 0; w < warps; ++w) s += red[w * TJ_RED + threadIdx.x];
                    rsum[threadIdx.x] = s;
                }
                __syncthreads();
                if (threadIdx.x == 0) {
                    double tot = 0.0;
                    for (int j = 0; j < nk; ++j) tot += tj_expect(K + (2 * j + 1) * dd, rsum, d);
                    double base = 0.0;
                    const int j = tj_pick([&](int i) { return tj_expect(K + (2 * i + 1) * dd, rsum, d); }, nk, base,
                                          rng.uniform(r[5]) * tot);
                    const double s = 1.0 / sqrt(tj_expect(K + (2 * j + 1) * dd, rsum, d));
                    for (int e = 0; e < dd; ++e) mat_s[e] = make_double2(K[2 * j * dd + e].x * s, K[2 * j * dd + e].y * s);
                    if (r[4] >= 0) c |= (uint32_t)j << r[4];
                }
            }
            __syncthreads();
            tj_apply(psi, n, nq, q0, q1, mat_s);
        }
        if (L.qmask) {                                   // terminal sample: inverse CDF of |psi|^2 in index order
            __syncthreads();
            const uint32_t chunk = N >= (uint32_t)T ? N / T : 1u, first = threadIdx.x * chunk;
            double s = 0.0;
            if (first < N)
                for (uint32_t i = 0; i < chunk; ++i) {
                    const double2 a = psi[first + i];
                    s += a.x * a.x + a.y * a.y;
                }
            part[threadIdx.x] = s;
            __syncthreads();
            const int G = T >> 5;                        // partials per lane of warp 0
            if (threadIdx.x < 32) {
                double w = 0.0;
                for (int i = 0; i < G; ++i) w += part[threadIdx.x * G + i];
                red[threadIdx.x] = w;
                __syncwarp();
                if (threadIdx.x == 0) {
                    double tot = 0.0;
                    for (int l = 0; l < 32; ++l) tot += red[l];
                    const double target = rng.uniform(P.term_uidx) * tot;
                    double base = 0.0;
                    const int l = tj_pick([&](int i) { return red[i]; }, 32, base, target);
                    const int t = l * G + tj_pick([&](int i) { return part[l * G + i]; }, G, base, target);
                    const uint32_t idx = t * chunk + tj_pick([&](int i) {
                        const double2 a = psi[t * chunk + i];
                        return a.x * a.x + a.y * a.y;
                    }, (int)min(chunk, N - min(N, (uint32_t)t * chunk)), base, target);
                    for (int q = 0; q < n; ++q)
                        if ((L.qmask >> q) & 1u) c |= ((idx >> q) & 1u) << P.qcol[q];
                }
            }
        }
        if (threadIdx.x == 0) {
            for (int j = 0; j < P.n_cols; ++j) {
                if (!((L.ro_mask >> j) & 1u)) continue;
                const double u = rng.uniform(P.term_uidx + 1 + __popc(P.ro_cols & ((1u << j) - 1u)));
                const int v = j >= row_bits ? (int)((L.digits >> (4 * (j - row_bits))) & 15ull) : 0;
                const uint32_t m = (c >> j) & 1u;
                const uint32_t o = u < P.ro[4 * (QCK_MAX_VARIANTS * j + v) + 2 + m] ? 1u : 0u;
                c = (c & ~(1u << j)) | (o << j);
            }
            if (P.shot_list) P.shot_list[tr] = c;
            if (P.out) {
                const int xb = P.n_cols - P.fold_bits;
                const long long one = (__popc(c >> xb) & 1) ? -1 : 1;
                atomicAdd(reinterpret_cast<unsigned long long*>(P.out + label * P.out_stride) + (c & ((1u << xb) - 1u)),
                          (unsigned long long)one);
            }
        }
    }
}

// the count rows: int64 zeros before the trajectories, count / shots after them
__global__ void tj_zero_kernel(double* out, long long label_begin, long long n_rows, long long stride, int xb) {
    const long long total = n_rows << xb;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x)
        reinterpret_cast<long long*>(out)[(label_begin + (i >> xb)) * stride + (i & ((1ll << xb) - 1))] = 0;
}
__global__ void tj_finish_kernel(double* out, long long label_begin, long long n_rows, long long stride, int xb,
                                 long long shots) {
    const long long total = n_rows << xb;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        double* p = out + (label_begin + (i >> xb)) * stride + (i & ((1ll << xb) - 1));
        *p = (double)*reinterpret_cast<long long*>(p) / (double)shots;
    }
}

QCK_API int qck_sim_trajectories(qck_handle* h, const qck_traj_plan* plan, int64_t label_begin, int64_t label_end,
                                 int64_t shots, uint64_t seed, uint32_t stream_id, double* d_out,
                                 int64_t out_row_stride, int64_t* d_shot_list, void* d_work, size_t work_bytes,
                                 qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    if (!plan || (!d_out && !d_shot_list) || !plan->d_ops || !plan->d_vars || !plan->d_mats || !plan->d_labels ||
        !plan->d_ro)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "NULL argument");
    const int n = plan->n_qubits;
    if (n < 1 || n > QCK_DM_MAX_QUBITS)
        QCK_FAIL(h, QCK_ERR_UNSUPPORTED, "n_qubits=%d: trajectories take 1 to %d qubits", n, QCK_DM_MAX_QUBITS);
    if (plan->n_ops < 0) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_ops=%d", plan->n_ops);
    if (plan->n_cols < 0 || plan->n_cols > 30 || plan->fold_bits < 0 || plan->fold_bits > plan->n_cols)
        QCK_FAIL(h, QCK_ERR_UNSUPPORTED, "row of 2^%d columns (fold %d) out of range", plan->n_cols, plan->fold_bits);
    if (plan->n_digits < 0 || plan->n_digits > QCK_MAX_DIGITS || plan->n_digits > plan->n_cols)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_digits=%d out of range", plan->n_digits);
    if (plan->term_uidx < 0) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "term_uidx=%d", plan->term_uidx);
    for (int q = 0; q < n; ++q)
        if (plan->qcol[q] >= plan->n_cols) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "qcol[%d]=%d out of range", q, plan->qcol[q]);
    if (label_begin < 0 || label_begin > label_end || label_end > plan->n_labels || label_end > (1ll << 32))
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "label range [%lld, %lld) outside [0, %lld)", (long long)label_begin,
                 (long long)label_end, (long long)plan->n_labels);
    if (shots < 1 || shots > INT32_MAX)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "shots=%lld: need 1 <= shots < 2^31", (long long)shots);
    if (d_out && out_row_stride < (1ll << (plan->n_cols - plan->fold_bits)) && label_end - label_begin > 1)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "output row stride shorter than a row");
    const bool smem_regime = n <= QCK_TRAJ_SMEM_MAX_QUBITS;
    const size_t slot_bytes = (size_t)16 << n;
    if (!smem_regime && (!d_work || work_bytes < slot_bytes))
        QCK_FAIL(h, QCK_ERR_NOMEM, "the work buffer (%zu bytes) holds no state of %d qubits (%zu bytes)", work_bytes,
                 n, slot_bytes);
    const long long n_rows = label_end - label_begin, n_traj = n_rows * shots;
    if (n_traj == 0) return QCK_OK;
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    const int xb = plan->n_cols - plan->fold_bits;
    const int zgrid = (int)std::min<long long>((n_rows << xb) / 256 + 1, (long long)h->sm_count * 8);
    if (d_out) {
        tj_zero_kernel<<<zgrid, 256, 0, st>>>(d_out, label_begin, n_rows, out_row_stride, xb);
        QCK_CHECK_LAUNCH(h);
    }
    TjParams P;
    memset(&P, 0, sizeof(P));
    P.ops = plan->d_ops;
    P.vars = plan->d_vars;
    P.mats = (const double2*)plan->d_mats;
    P.labels = (const TjLabel*)plan->d_labels;
    P.ro = plan->d_ro;
    P.n = n;
    P.n_ops = plan->n_ops;
    P.n_cols = plan->n_cols;
    P.n_digits = plan->n_digits;
    P.fold_bits = plan->fold_bits;
    P.term_uidx = plan->term_uidx;
    P.ro_cols = plan->ro_cols;
    for (int q = 0; q < QCK_DM_MAX_QUBITS; ++q) P.qcol[q] = q < n ? plan->qcol[q] : -1;
    P.label_begin = label_begin;
    P.n_traj = n_traj;
    P.shots = shots;
    P.seed = seed;
    P.stream_id = stream_id;
    P.out = d_out;
    P.out_stride = out_row_stride;
    P.shot_list = (long long*)d_shot_list;
    P.work = (double2*)d_work;
    const int T = tj_threads(n);
    const size_t scratch = (size_t)8 * T + (size_t)8 * std::max(32, TJ_RED * (T / 32));
    if (smem_regime) {
        const size_t smem = ((size_t)16 << n) + scratch;
        QCK_CUDA(h, cudaFuncSetAttribute(tj_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 0;
        QCK_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tj_kernel<true>, T, smem));
        const long long grid = std::min<long long>(n_traj, (long long)h->sm_count * std::max(per_sm, 1));
        tj_kernel<true><<<(unsigned)grid, T, smem, st>>>(P);
    } else {
        const long long grid = std::min<long long>(n_traj, (long long)(work_bytes / slot_bytes));
        tj_kernel<false><<<(unsigned)grid, T, scratch, st>>>(P);
    }
    QCK_CHECK_LAUNCH(h);
    if (d_out) {
        tj_finish_kernel<<<zgrid, 256, 0, st>>>(d_out, label_begin, n_rows, out_row_stride, xb, shots);
        QCK_CHECK_LAUNCH(h);
    }
    return QCK_OK;
}

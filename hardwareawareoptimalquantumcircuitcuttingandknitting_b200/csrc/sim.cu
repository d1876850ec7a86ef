// Batched statevector simulation of fragment instances (sm_100a).
//
// Replaces the reference's per-instance circuit construction and Aer run
// (third_party/qvm/qvm/virtual_circuit.py:183-213, run.py:36-58).  One CTA owns one
// tile of one instance: the tile (2^n_tile complex128 amplitudes) lives in shared
// memory while a run of gates that only touch tile-local qubits is applied.
//   * on-chip regime  (n_state <= 13): one sweep, the whole state is the tile, HBM is
//     touched only by the output row;
//   * streaming regime (n_state  > 13): the state lives in HBM/L2, every sweep is one
//     coalesced read + one coalesced write of the state (tiles always contain the low
//     qubits so that a tile is made of >= 256-byte contiguous runs).
// Measurements whose qubit lives on are CX gates onto ancilla bits (deferred
// measurement); the epilogue folds |amp|^2 into the instance's output row with the
// (-1)^bit weights of the knit rules.
#include "qck_common.cuh"

#include <cuda.h>  // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint)
#include <stdlib.h>

#include <memory>

struct PlanDev {
    int n_state;
    const qck_op* ops;
    const double* mats;
    int n_digits;
    int radix[QCK_MAX_DIGITS];
    int n_out_bits;
    int out_pos[QCK_MAX_OUT_BITS];
    int out_ident;  // out_pos[j] == j for j < out_ident: those row bits map straight to state bits
    int n_stage;    // capacity (records) of the shared-memory program stage of this launch
    unsigned long long sum_mask, sign_mask;
};

struct SweepDev {
    int n_tile;
    int op_begin, op_end;
    int n_low;  // pos[i] == i for i < n_low (contiguous low run)
    int init;   // 1: synthesise |0..0> instead of reading
    int has_x;  // the op range holds tile-resolved ops (QCK_OP_U1X / QCK_OP_PHASE)
    int pos[QCK_MAX_TILE_QUBITS + 2];
};

__device__ __forceinline__ double2 cmul(double2 a, double2 b) {
    return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ double2 cfma(double2 a, double2 b, double2 c) {  // a*b + c
    return make_double2(fma(a.x, b.x, fma(-a.y, b.y, c.x)), fma(a.x, b.y, fma(a.y, b.x, c.y)));
}

__device__ __forceinline__ void decode_digits(const PlanDev& plan, int label, int* digits) {
    int rem = label;
    for (int k = plan.n_digits - 1; k >= 0; --k) {
        int r = plan.radix[k];
        digits[k] = rem % r;
        rem /= r;
    }
}

// Shared-memory layout: amplitude i lives at slot swz(i).  The XOR folds index bits 3-5 into
// bits 0-2 so that eight lanes that differ in *any* three of those six bits hit eight different
// 16-byte bank groups: cluster passes whose register qubits are the low qubits (lane stride
// 128 B) stay conflict-free.  The permutation stays inside 128-byte lines.
__device__ __forceinline__ uint32_t swz(uint32_t i) { return i ^ ((i >> 3) & 7u); }

// ---- register-tiled gate application: a[k], k in [0, 8), bit j of k = cluster qubit j
template <int J>
__device__ __forceinline__ void reg_u1(double2 (&a)[8], double2 m00, double2 m01, double2 m10, double2 m11) {
#pragma unroll
    for (int k = 0; k < 8; ++k)
        if (!(k & (1 << J))) {
            const double2 x = a[k], y = a[k | (1 << J)];
            a[k] = cfma(m01, y, cmul(m00, x));
            a[k | (1 << J)] = cfma(m11, y, cmul(m10, x));
        }
}
template <int J>
__device__ __forceinline__ void reg_diag(double2 (&a)[8], double2 d0, double2 d1) {
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = cmul((k & (1 << J)) ? d1 : d0, a[k]);
}
template <int J0, int J1>
__device__ __forceinline__ void reg_cx(double2 (&a)[8]) {
#pragma unroll
    for (int k = 0; k < 8; ++k)
        if ((k & (1 << J0)) && !(k & (1 << J1))) {
            const double2 t = a[k];
            a[k] = a[k | (1 << J1)];
            a[k | (1 << J1)] = t;
        }
}
template <int J0, int J1>
__device__ __forceinline__ void reg_cz(double2 (&a)[8]) {
#pragma unroll
    for (int k = 0; k < 8; ++k)
        if ((k & (1 << J0)) && (k & (1 << J1))) a[k] = make_double2(-a[k].x, -a[k].y);
}
template <int J0, int J1>
__device__ __forceinline__ void reg_u2(double2 (&a)[8], const double2* m) {
#pragma unroll
    for (int k = 0; k < 8; ++k)
        if (!(k & ((1 << J0) | (1 << J1)))) {
            const double2 x[4] = {a[k], a[k | (1 << J0)], a[k | (1 << J1)], a[k | (1 << J0) | (1 << J1)]};
            double2 r[4];
#pragma unroll
            for (int row = 0; row < 4; ++row) {
                double2 acc = cmul(m[row * 4], x[0]);
#pragma unroll
                for (int c = 1; c < 4; ++c) acc = cfma(m[row * 4 + c], x[c], acc);
                r[row] = acc;
            }
            a[k] = r[0];
            a[k | (1 << J0)] = r[1];
            a[k | (1 << J1)] = r[2];
            a[k | (1 << J0) | (1 << J1)] = r[3];
        }
}

#define QCK_PAIR_DISPATCH(FN, ...)                                     \
    switch (q0 * 3 + q1) {                                             \
        case 1: FN<0, 1>(__VA_ARGS__); break;                          \
        case 2: FN<0, 2>(__VA_ARGS__); break;                          \
        case 3: FN<1, 0>(__VA_ARGS__); break;                          \
        case 5: FN<1, 2>(__VA_ARGS__); break;                          \
        case 6: FN<2, 0>(__VA_ARGS__); break;                          \
        default: FN<2, 1>(__VA_ARGS__); break;                         \
    }

// ---- program staging --------------------------------------------------------------------------
// Op records and the (label-digit-resolved) 2x2 matrices of a chunk of the program are staged in
// shared memory once per CTA, so that per-op fetches are broadcast LDS instead of two dependent
// global loads (op record -> matrix), which dominated the run time of small instances.
struct StagedOp {
    int4 w0, w1;     // the qck_op words; w0.w = resolved matrix offset
    double2 m[16];   // U1: m[0..3]; U2: the 4x4 matrix, row major
};
#define QCK_STAGE_OPS 96
#define QCK_MAX_CLUSTER_OPS 32

// Which threads cooperate on a tile.  WholeCta: every thread of the block, __syncthreads().
// ConsumerWarps<N>: threads [32, 32 + N) of a warp-specialised block (warp 0 drives TMA), named
// barrier 1 - the producer warp never takes part in it.
// CTA barrier for the gate passes.  A pass over fewer items than a warp has lanes (16 quads of a 6-qubit
// tile) leaves the warp diverged in front of the barrier; __syncwarp() makes the reconvergence explicit.
// NOTE (observed on sm_100a, nvcc 12.9): no pass may leave through an early `return` that skips its
// closing barrier, even a warp-uniform one - with the passes inlined into the op loop the lanes that had
// skipped the previous pass's loop then ran ahead of their own warp, and the next pass's results were
// overwritten by the lagging lanes' stores (plain sweep kernel, 64-amplitude tiles).  Every pass therefore
// ends in exactly one barrier on every path.
__device__ __forceinline__ void cta_sync() {
    __syncwarp();
    __syncthreads();
}
struct WholeCta {
    __device__ static __forceinline__ int tid() { return threadIdx.x; }
    __device__ static __forceinline__ int nth() { return blockDim.x; }
    __device__ static __forceinline__ void sync() { cta_sync(); }
};
// TAG only makes the instantiations of the gate passes distinct per kernel: a pass shared by several kernel
// instantiations is no longer inlined into them (measured: 13.3 -> 14.9 ms on the syc-32 d1 expansion sweep).
template <int N, int TAG = 0>
struct ConsumerWarps {
    __device__ static __forceinline__ int tid() { return (int)threadIdx.x - 32; }
    __device__ static __forceinline__ int nth() { return N; }
    // small tiles leave lanes of a warp diverged in front of the barrier (fewer groups than lanes): bar.sync
    // (= barrier.sync.aligned) would be undefined there, so reconverge first and use the unaligned form
    __device__ static __forceinline__ void sync() {
        __syncwarp();
        asm volatile("barrier.sync 1, %0;" ::"n"(N) : "memory");
    }
};

// `perm` (may be NULL) renames tile-local qubits: the TMA sweep kernel lays a tile out as
// [low run | main run | scattered bits], not in ascending state-bit order.  Cluster members
// address their cluster's qubits by rank (reserved == 1) and are left alone; the header's
// positions are renamed (they may then be out of order, run_cluster sorts them).
template <class P>
__device__ __forceinline__ void stage_ops(StagedOp* so, const qck_op* __restrict__ ops, int c0, int n,
                                          const double* __restrict__ mats, const int* digits,
                                          const int* perm = nullptr) {
    for (int i = P::tid(); i < n; i += P::nth()) {
        int4 w0 = __ldg(reinterpret_cast<const int4*>(ops + c0 + i));
        int4 w1 = __ldg(reinterpret_cast<const int4*>(ops + c0 + i) + 1);
        if (w0.x == QCK_OP_U1 || w0.x == QCK_OP_U2) {
            if (w1.x >= 0) w0.w += digits[w1.x] * w1.y;
            const double2* m = reinterpret_cast<const double2*>(mats + w0.w);
            const int n_m = w0.x == QCK_OP_U1 ? 4 : 16;
            for (int e = 0; e < n_m; ++e) so[i].m[e] = __ldg(m + e);
        } else if (w0.x == QCK_OP_TERM) {  // the variants a tile picks from (resolve_tile)
            const double2* m = reinterpret_cast<const double2*>(mats + w0.w);
            for (int e = 0; e < w1.y && e < 16; ++e) so[i].m[e] = __ldg(m + e);
        }
        if (perm) {
            if (w0.x == QCK_OP_CLUSTER) {
                w0.w = perm[w0.w];
                w1.x = perm[w1.x];
                w1.y = perm[w1.y];
            } else if (w0.x == QCK_OP_U1X) {
                w0.y = perm[w0.y];
            } else if (w1.w == 0) {
                w0.y = perm[w0.y];
                if (w0.x != QCK_OP_U1) w0.z = perm[w0.z];
            }
        }
        so[i].w0 = w0;
        so[i].w1 = w1;
    }
}

// Tile-resolved ops: the bits of the tile's base address select, per term, one of the staged variants;
// the header receives the product (U1X: 2x2 matrix in m[0..3]; PHASE: scalar in m[0]).  One thread per
// header; the terms stay intact, so every tile resolves afresh.
template <class P>
__device__ __forceinline__ void resolve_tile(StagedOp* so, int n, unsigned long long base) {
    for (int i = P::tid(); i < n; i += P::nth()) {
        const int kind = so[i].w0.x;
        if ((kind == QCK_OP_U1X || kind == QCK_OP_PHASE) && i + so[i].w0.z >= n) continue;  // terms not staged
        if (kind == QCK_OP_U1X) {
            const int n_terms = so[i].w0.z;
            double2 m00 = make_double2(1.0, 0.0), m01 = make_double2(0.0, 0.0), m10 = m01, m11 = m00;
            for (int t = 1; t <= n_terms; ++t) {
                const StagedOp& tm = so[i + t];
                const double2* v = tm.m + 4 * (int)((base >> tm.w0.y) & 1ull);
                const double2 a = v[0], b = v[1], c = v[2], d = v[3];  // [[a b] [c d]] * M
                const double2 n00 = cfma(b, m10, cmul(a, m00)), n01 = cfma(b, m11, cmul(a, m01));
                const double2 n10 = cfma(d, m10, cmul(c, m00)), n11 = cfma(d, m11, cmul(c, m01));
                m00 = n00; m01 = n01; m10 = n10; m11 = n11;
            }
            so[i].m[0] = m00; so[i].m[1] = m01; so[i].m[2] = m10; so[i].m[3] = m11;
        } else if (kind == QCK_OP_PHASE) {
            const int n_terms = so[i].w0.z;
            double2 sc = make_double2(1.0, 0.0);
            for (int t = 1; t <= n_terms; ++t) {
                const StagedOp& tm = so[i + t];
                int idx = (int)((base >> tm.w0.y) & 1ull);
                if (tm.w0.z >= 0) idx |= (int)((base >> tm.w0.z) & 1ull) << 1;
                sc = cmul(tm.m[idx], sc);
            }
            so[i].m[0] = sc;
        }
    }
}

// Whole-tile scalar (QCK_OP_PHASE after resolve_tile).
template <class P>
__device__ void run_phase(double2* s, int T, double2 sc) {
    if (!(sc.x == 1.0 && sc.y == 0.0)) {  // uniform
        const uint32_t n = 1u << T;
        for (uint32_t j = P::tid(); j < n; j += P::nth()) s[j] = cmul(sc, s[j]);
    }
    P::sync();
}

// One cluster: header so[h], members so[h+1 .. h+n].  Every thread owns groups of 8 amplitudes
// (the 3 cluster bits enumerated) and applies all member ops in registers.
template <class P>
__device__ void run_cluster(double2* s, int T, const StagedOp* so, int h, const double* __restrict__ mats) {
    const int4 h0 = so[h].w0, h1 = so[h].w1;
    const int n_ops = h0.y, p0 = h0.w, p1 = h1.x, p2 = h1.y;
    int nl = h1.z;
    if (nl <= 0 || nl > T) nl = T;
    const uint32_t n_groups = 1u << (nl - 3);
    const uint32_t b0 = 1u << p0, b1 = 1u << p1, b2 = 1u << p2;
    // ascending order for the zero insertion (renamed positions may be out of order)
    const int s0 = min(p0, min(p1, p2)), s2 = max(p0, max(p1, p2)), s1 = p0 + p1 + p2 - s0 - s2;
    for (uint32_t g = P::tid(); g < n_groups; g += P::nth()) {
        const uint32_t base = insert_zero(insert_zero(insert_zero(g, s0), s1), s2);
        double2 a[8];
#pragma unroll
        for (int k = 0; k < 8; ++k)
            a[k] = s[swz(base | ((k & 1) ? b0 : 0u) | ((k & 2) ? b1 : 0u) | ((k & 4) ? b2 : 0u))];
        for (int i = h + 1; i <= h + n_ops; ++i) {
            const int4 w0 = so[i].w0;
            const int kind = w0.x, q0 = w0.y, q1 = w0.z;
            if (kind == QCK_OP_U1) {
                const double2 m00 = so[i].m[0], m01 = so[i].m[1], m10 = so[i].m[2], m11 = so[i].m[3];
                if (m01.x == 0.0 && m01.y == 0.0 && m10.x == 0.0 && m10.y == 0.0) {
                    if (m00.x == 1.0 && m00.y == 0.0 && m11.x == 1.0 && m11.y == 0.0) continue;
                    if (q0 == 0) reg_diag<0>(a, m00, m11);
                    else if (q0 == 1) reg_diag<1>(a, m00, m11);
                    else reg_diag<2>(a, m00, m11);
                } else {
                    if (q0 == 0) reg_u1<0>(a, m00, m01, m10, m11);
                    else if (q0 == 1) reg_u1<1>(a, m00, m01, m10, m11);
                    else reg_u1<2>(a, m00, m01, m10, m11);
                }
            } else if (kind == QCK_OP_CX) {
                QCK_PAIR_DISPATCH(reg_cx, a)
            } else if (kind == QCK_OP_CZ) {
                QCK_PAIR_DISPATCH(reg_cz, a)
            } else {
                const double2* m = so[i].m;
                QCK_PAIR_DISPATCH(reg_u2, a, m)
            }
        }
#pragma unroll
        for (int k = 0; k < 8; ++k)
            s[swz(base | ((k & 1) ? b0 : 0u) | ((k & 2) ? b1 : 0u) | ((k & 4) ? b2 : 0u))] = a[k];
    }
    P::sync();
}

// One un-clustered op (states with fewer than 3 live bits, or clustering disabled).
template <class P>
__device__ void run_single(double2* s, int T, const StagedOp& op, const double* __restrict__ mats) {
    const int tid = P::tid(), nth = P::nth();
    const int kind = op.w0.x, q0 = op.w0.y, q1 = op.w0.z;
    int nl = op.w1.z;
    if (nl <= 0 || nl > T) nl = T;
    if (kind == QCK_OP_U1 || kind == QCK_OP_U1X) {
        const double2 m00 = op.m[0], m01 = op.m[1], m10 = op.m[2], m11 = op.m[3];
        const uint32_t n = 1u << (nl - 1);
        if (m01.x == 0.0 && m01.y == 0.0 && m10.x == 0.0 && m10.y == 0.0) {
            // identity (uniform): nothing to do, but the pass still ends in its barrier (see cta_sync)
            const bool ident = m00.x == 1.0 && m00.y == 0.0 && m11.x == 1.0 && m11.y == 0.0;
            for (uint32_t p = ident ? n : tid; p < n; p += nth) {
                const uint32_t i0 = insert_zero(p, q0), i1 = i0 | (1u << q0);
                s[swz(i0)] = cmul(m00, s[swz(i0)]);
                s[swz(i1)] = cmul(m11, s[swz(i1)]);
            }
        } else {
            for (uint32_t p = tid; p < n; p += nth) {
                const uint32_t i0 = insert_zero(p, q0), i1 = i0 | (1u << q0);
                const double2 a0 = s[swz(i0)], a1 = s[swz(i1)];
                s[swz(i0)] = cfma(m01, a1, cmul(m00, a0));
                s[swz(i1)] = cfma(m11, a1, cmul(m10, a0));
            }
        }
    } else {
        const int lo = q0 < q1 ? q0 : q1, hi = q0 < q1 ? q1 : q0;
        const uint32_t n = 1u << (nl - 2);
        const uint32_t b0 = 1u << q0, b1 = 1u << q1;
        if (kind == QCK_OP_CX) {
            for (uint32_t p = tid; p < n; p += nth) {
                const uint32_t base = insert_zero(insert_zero(p, lo), hi) | b0;  // control set
                const double2 a = s[swz(base)], b = s[swz(base | b1)];
                s[swz(base)] = b;
                s[swz(base | b1)] = a;
            }
        } else if (kind == QCK_OP_CZ) {
            for (uint32_t p = tid; p < n; p += nth) {
                const uint32_t idx = insert_zero(insert_zero(p, lo), hi) | b0 | b1;
                const double2 a = s[swz(idx)];
                s[swz(idx)] = make_double2(-a.x, -a.y);
            }
        } else {  // QCK_OP_U2: generic 4x4, row/col index = bit(q0) + 2 bit(q1)
            // The matrix lives in registers for all of this thread's quads: 64 FP64 instructions per
            // 4 amplitudes plus 4 LDS + 4 STS.  Index math: insert_zero and swz are bitwise-linear, so
            // for p = tid + k * nth (nth a power of two) slot(p) = slot(tid) ^ slot(k * nth): the
            // per-thread part is computed once per op, the per-k part is warp-uniform.
            double2 m[16];
#pragma unroll
            for (int e = 0; e < 16; ++e) m[e] = op.m[e];
            const uint32_t x1 = swz(b0), x2 = swz(b1), x3 = x1 ^ x2;
            bool diag = true;  // uniform: cz / cp / rzz and their fusions with one-qubit phases
#pragma unroll
            for (int e = 0; e < 16; ++e)
                if (e % 5 != 0) diag = diag && m[e].x == 0.0 && m[e].y == 0.0;
            if (diag) {  // 4 complex multiplications per quad instead of 16, entries equal to 1 skipped
                const bool t0 = !(m[0].x == 1.0 && m[0].y == 0.0), t1 = !(m[5].x == 1.0 && m[5].y == 0.0);
                const bool t2 = !(m[10].x == 1.0 && m[10].y == 0.0), t3 = !(m[15].x == 1.0 && m[15].y == 0.0);
                for (uint32_t p = tid; p < n; p += nth) {
                    const uint32_t i0 = swz(insert_zero(insert_zero(p, lo), hi));
                    if (t0) s[i0] = cmul(m[0], s[i0]);
                    if (t1) s[i0 ^ x1] = cmul(m[5], s[i0 ^ x1]);
                    if (t2) s[i0 ^ x2] = cmul(m[10], s[i0 ^ x2]);
                    if (t3) s[i0 ^ x3] = cmul(m[15], s[i0 ^ x3]);
                }
            } else if ((nth & (nth - 1)) == 0) {
                const uint32_t st = swz(insert_zero(insert_zero((uint32_t)tid, lo), hi));
                if ((uint32_t)tid < n) {
#pragma unroll 2
                    for (uint32_t pk = 0; pk < n; pk += nth) {
                        const uint32_t i0 = st ^ swz(insert_zero(insert_zero(pk, lo), hi));
                        const uint32_t i1 = i0 ^ x1, i2 = i0 ^ x2, i3 = i0 ^ x3;
                        const double2 a0 = s[i0], a1 = s[i1], a2 = s[i2], a3 = s[i3];
                        s[i0] = cfma(m[3], a3, cfma(m[2], a2, cfma(m[1], a1, cmul(m[0], a0))));
                        s[i1] = cfma(m[7], a3, cfma(m[6], a2, cfma(m[5], a1, cmul(m[4], a0))));
                        s[i2] = cfma(m[11], a3, cfma(m[10], a2, cfma(m[9], a1, cmul(m[8], a0))));
                        s[i3] = cfma(m[15], a3, cfma(m[14], a2, cfma(m[13], a1, cmul(m[12], a0))));
                    }
                }
            } else {
                for (uint32_t p = tid; p < n; p += nth) {
                    const uint32_t i0 = swz(insert_zero(insert_zero(p, lo), hi));
                    const uint32_t i1 = i0 ^ x1, i2 = i0 ^ x2, i3 = i0 ^ x3;
                    const double2 a0 = s[i0], a1 = s[i1], a2 = s[i2], a3 = s[i3];
                    s[i0] = cfma(m[3], a3, cfma(m[2], a2, cfma(m[1], a1, cmul(m[0], a0))));
                    s[i1] = cfma(m[7], a3, cfma(m[6], a2, cfma(m[5], a1, cmul(m[4], a0))));
                    s[i2] = cfma(m[11], a3, cfma(m[10], a2, cfma(m[9], a1, cmul(m[8], a0))));
                    s[i3] = cfma(m[15], a3, cfma(m[14], a2, cfma(m[13], a1, cmul(m[12], a0))));
                }
            }
        }
    }
    P::sync();
}

// Apply ops[begin, end) to the tile `s` (2^T amplitudes in shared memory).  All threads of the
// CTA call this with identical arguments; the state is synchronised on return.
template <class P, bool CLUSTERS = true>
__device__ void apply_ops(double2* s, int T, StagedOp* so, int n_stage, const qck_op* __restrict__ ops, int begin,
                          int end, const double* __restrict__ mats, const int* digits, bool prestaged,
                          bool resolve = false, unsigned long long base = 0ull, const int* perm = nullptr) {
    int c0 = begin;
    while (c0 < end) {
        const int n = (end - c0) < n_stage ? (end - c0) : n_stage;
        if (!(prestaged && c0 == begin)) {  // the caller may have staged the first chunk already
            stage_ops<P>(so, ops, c0, n, mats, digits, perm);
            P::sync();
        }
        if (resolve) {  // headers whose terms were cut off by the chunk are resolved with the next chunk
            resolve_tile<P>(so, n, base);
            P::sync();
        }
        int i = 0;
        while (i < n) {
            const int kind_i = so[i].w0.x;
            if (CLUSTERS && kind_i == QCK_OP_CLUSTER) {
                const int members = so[i].w0.y;
                if (i + members >= n && c0 + n < end) break;  // cluster continues past the staged chunk
                run_cluster<P>(s, T, so, i, mats);
                i += 1 + members;
            } else if (kind_i == QCK_OP_U1X || kind_i == QCK_OP_PHASE) {
                const int terms = so[i].w0.z;
                if (i + terms >= n && c0 + n < end) break;  // terms continue past the staged chunk
                if (kind_i == QCK_OP_U1X) run_single<P>(s, T, so[i], mats);
                else run_phase<P>(s, T, so[i].m[0]);
                i += 1 + terms;
            } else {
                run_single<P>(s, T, so[i], mats);
                ++i;
            }
        }
        c0 += i;
        P::sync();  // everyone is done with so[] before it is restaged
    }
}

// |amp|^2 folded into the output row (deterministic order, no atomics): one thread per
// output entry walks the summed-out bits with the masked-increment trick.
template <typename LoadAmp>
__device__ __forceinline__ double fold_entry(const PlanDev& plan, uint64_t o, LoadAmp load) {
    uint64_t base = o & ((1ull << plan.out_ident) - 1ull);
    for (int j = plan.out_ident; j < plan.n_out_bits; ++j) {
        if ((o >> j) & 1ull) {
            if (plan.out_pos[j] < 0) return 0.0;  // that bit is never written in this pattern
            base |= 1ull << plan.out_pos[j];
        }
    }
    const uint64_t sm = plan.sum_mask, sg = plan.sign_mask;
    double acc = 0.0;
    uint64_t sub = 0;
    do {
        double2 a = load(base | sub);
        double p = fma(a.x, a.x, a.y * a.y);
        acc += (__popcll(sub & sg) & 1) ? -p : p;
        sub = (sub - sm) & sm;
    } while (sub != 0);
    return acc;
}

// ------------------------------------------------------------------ on-chip regime
extern __shared__ __align__(16) unsigned char smem_raw[];

// Label-independent prefix of an on-chip program (qck_sweep flag QCK_SWEEP_SHARED): run ONCE, the state is left
// in global memory (`snap`, the shared-memory image as it is) and every instance starts from it instead of |0>.
__global__ void __launch_bounds__(256) sim_onchip_prefix_kernel(PlanDev plan, int op_begin, int op_end,
                                                                double2* __restrict__ snap) {
    double2* s = reinterpret_cast<double2*>(smem_raw);
    StagedOp* so = reinterpret_cast<StagedOp*>(smem_raw + ((size_t)16 << plan.n_state));
    __shared__ int digits[QCK_MAX_DIGITS];
    if (threadIdx.x < QCK_MAX_DIGITS) digits[threadIdx.x] = 0;  // no op of a shared prefix selects by digit
    const uint32_t n_amp = 1u << plan.n_state;
    cta_sync();
    {
        const int n0 = (op_end - op_begin) < plan.n_stage ? (op_end - op_begin) : plan.n_stage;
        stage_ops<WholeCta>(so, plan.ops, op_begin, n0, plan.mats, digits);
    }
    for (uint32_t i = threadIdx.x; i < n_amp; i += blockDim.x) s[i] = make_double2(i == 0 ? 1.0 : 0.0, 0.0);
    cta_sync();
    apply_ops<WholeCta>(s, plan.n_state, so, plan.n_stage, plan.ops, op_begin, op_end, plan.mats, digits, true);
    for (uint32_t i = threadIdx.x; i < n_amp; i += blockDim.x) snap[i] = s[i];
}

__global__ void __launch_bounds__(256) sim_onchip_kernel(PlanDev plan, int op_begin, int op_end,
                                                         const int32_t* __restrict__ labels,
                                                         double* __restrict__ out, long long row_stride,
                                                         const double2* __restrict__ init) {
    double2* s = reinterpret_cast<double2*>(smem_raw);
    StagedOp* so = reinterpret_cast<StagedOp*>(smem_raw + ((size_t)16 << plan.n_state));
    __shared__ int digits[QCK_MAX_DIGITS];
    const int label = labels[blockIdx.x];
    if (threadIdx.x == 0) decode_digits(plan, label, digits);
    const uint32_t n_amp = 1u << plan.n_state;
    cta_sync();  // digits visible
    {
        const int n0 = (op_end - op_begin) < plan.n_stage ? (op_end - op_begin) : plan.n_stage;
        stage_ops<WholeCta>(so, plan.ops, op_begin, n0, plan.mats, digits);  // global loads overlap the state init
    }
    if (init) {
        for (uint32_t i = threadIdx.x; i < n_amp; i += blockDim.x) s[i] = __ldg(init + i);
    } else {
        for (uint32_t i = threadIdx.x; i < n_amp; i += blockDim.x) s[i] = make_double2(i == 0 ? 1.0 : 0.0, 0.0);  // swz(0) == 0
    }
    cta_sync();
    apply_ops<WholeCta>(s, plan.n_state, so, plan.n_stage, plan.ops, op_begin, op_end, plan.mats, digits, true);
    const uint64_t n_out = 1ull << plan.n_out_bits;
    double* row = out + (long long)label * row_stride;
    for (uint64_t o = threadIdx.x; o < n_out; o += blockDim.x)
        row[o] = fold_entry(plan, o, [&](uint64_t idx) { return s[swz((uint32_t)idx)]; });
}

// Grouped form: one launch covers several programs (measurement patterns) of the same state size.
// The per-program parts travel in the kernel parameters (CUDA >= 12.1 allows 32 KB of them), the CTA
// looks up its program from its block index.  Replaces one launch per pattern (64 per step at
// hwe-16-d5) by one per state size.
#define QCK_GROUP_MAX 24
struct PlanVarDev {
    int op_begin, op_end;
    int n_out_bits, out_ident;
    signed char out_pos[QCK_MAX_OUT_BITS];
    unsigned long long sum_mask, sign_mask;
    const int32_t* labels;
    const double2* init;  // state after the shared prefix (sim_onchip_prefix_kernel), or nullptr: start from |0>
    int cta_begin, n_stage_unused;
};
struct GroupDev {
    int n_state, n_vars, n_stage, n_digits;
    const qck_op* ops;
    const double* mats;
    int radix[QCK_MAX_DIGITS];
    PlanVarDev var[QCK_GROUP_MAX];
};

__global__ void __launch_bounds__(256) sim_onchip_group_kernel(const __grid_constant__ GroupDev G,
                                                               double* __restrict__ out, long long row_stride) {
    double2* s = reinterpret_cast<double2*>(smem_raw);
    StagedOp* so = reinterpret_cast<StagedOp*>(smem_raw + ((size_t)16 << G.n_state));
    __shared__ int digits[QCK_MAX_DIGITS];
    __shared__ PlanDev plan;
    int v = 0;
    while (v + 1 < G.n_vars && (int)blockIdx.x >= G.var[v + 1].cta_begin) ++v;  // uniform
    const PlanVarDev& pv = G.var[v];
    const int label = __ldg(pv.labels + ((int)blockIdx.x - pv.cta_begin));
    if (threadIdx.x == 0) {
        plan.n_state = G.n_state;
        plan.ops = G.ops;
        plan.mats = G.mats;
        plan.n_digits = G.n_digits;
        for (int k = 0; k < QCK_MAX_DIGITS; ++k) plan.radix[k] = G.radix[k];
        plan.n_out_bits = pv.n_out_bits;
        plan.out_ident = pv.out_ident;
        for (int j = 0; j < QCK_MAX_OUT_BITS; ++j) plan.out_pos[j] = pv.out_pos[j];
        plan.sum_mask = pv.sum_mask;
        plan.sign_mask = pv.sign_mask;
        plan.n_stage = G.n_stage;
        decode_digits(plan, label, digits);
    }
    cta_sync();
    {
        const int n0 = (pv.op_end - pv.op_begin) < G.n_stage ? (pv.op_end - pv.op_begin) : G.n_stage;
        stage_ops<WholeCta>(so, G.ops, pv.op_begin, n0, G.mats, digits);
    }
    const uint32_t n_amp = 1u << G.n_state;
    if (pv.init) {
        for (uint32_t i = threadIdx.x; i < n_amp; i += blockDim.x) s[i] = __ldg(pv.init + i);
    } else {
        for (uint32_t i = threadIdx.x; i < n_amp; i += blockDim.x) s[i] = make_double2(i == 0 ? 1.0 : 0.0, 0.0);  // swz(0) == 0
    }
    cta_sync();
    apply_ops<WholeCta>(s, G.n_state, so, G.n_stage, G.ops, pv.op_begin, pv.op_end, G.mats, digits, true);
    const uint64_t n_out = 1ull << plan.n_out_bits;
    double* row = out + (long long)label * row_stride;
    for (uint64_t o = threadIdx.x; o < n_out; o += blockDim.x)
        row[o] = fold_entry(plan, o, [&](uint64_t idx) { return s[swz((uint32_t)idx)]; });
}

#include "sim_warp_kernel.inc"
#include "sim_tree_kernel.inc"

// ------------------------------------------------------------------ streaming regime
__global__ void __launch_bounds__(256) sim_sweep_kernel(PlanDev plan, SweepDev sw,
                                                        const int32_t* __restrict__ labels, int inst_base,
                                                        double2* __restrict__ work,
                                                        unsigned long long state_stride) {
    const int T = sw.n_tile, c = sw.n_low, n_hi = T - c;
    double2* s = reinterpret_cast<double2*>(smem_raw);
    unsigned long long* hi_off = reinterpret_cast<unsigned long long*>(smem_raw + ((size_t)16 << T));
    StagedOp* so = reinterpret_cast<StagedOp*>(smem_raw + ((size_t)16 << T) + ((((size_t)8 << n_hi) + 15) & ~(size_t)15));
    __shared__ int digits[QCK_MAX_DIGITS];
    const int label = labels[inst_base + blockIdx.y];
    if (threadIdx.x == 0) decode_digits(plan, label, digits);
    // offsets of the non-contiguous tile bits
    for (uint32_t j = threadIdx.x; j < (1u << n_hi); j += blockDim.x) {
        unsigned long long off = 0;
        for (int b = 0; b < n_hi; ++b)
            if ((j >> b) & 1u) off |= 1ull << sw.pos[c + b];
        hi_off[j] = off;
    }
    // base address of this tile: spread the tile index over the non-tile bit positions
    unsigned long long base = blockIdx.x;
    for (int j = 0; j < T; ++j) base = insert_zero64(base, sw.pos[j]);
    double2* st = work + (unsigned long long)blockIdx.y * state_stride;
    cta_sync();
    const uint32_t n_amp = 1u << T, low_mask = (1u << c) - 1u;
    if (sw.init) {
        for (uint32_t j = threadIdx.x; j < n_amp; j += blockDim.x)
            s[j] = make_double2((j == 0 && base == 0) ? 1.0 : 0.0, 0.0);  // swz(0) == 0
    } else {
        // cp.async (LDGSTS): every thread has all of its 16-byte loads in flight at once, the
        // data goes straight to shared memory (L1 bypassed)
        // j = tid + k * 256: the low 8 bits (hence the swizzle term and, for c <= 8, the low-run
        // offset) are per-thread constants; only the hi_off index advances with k
        const uint32_t s_base = (uint32_t)__cvta_generic_to_shared(s);
        const uint32_t xr = (threadIdx.x >> 3) & 7u;
        for (uint32_t j = threadIdx.x; j < n_amp; j += blockDim.x) {
            const double2* src = st + (base | hi_off[j >> c] | (j & low_mask));
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s_base + ((j ^ xr) << 4)), "l"(src) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    {   // stage the program while the tile is in flight
        const int n0 = (sw.op_end - sw.op_begin) < plan.n_stage ? (sw.op_end - sw.op_begin) : plan.n_stage;
        stage_ops<WholeCta>(so, plan.ops, sw.op_begin, n0, plan.mats, digits);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    cta_sync();
    apply_ops<WholeCta>(s, T, so, plan.n_stage, plan.ops, sw.op_begin, sw.op_end, plan.mats, digits, true, sw.has_x != 0,
                        base);
    {
        const uint32_t xr = (threadIdx.x >> 3) & 7u;  // blockDim.x == 256: bits 3-5 of j never change
#pragma unroll 4
        for (uint32_t j = threadIdx.x; j < n_amp; j += blockDim.x)
            __stcs(st + (base | hi_off[j >> c] | (j & low_mask)), s[j ^ xr]);
    }
}

// ------------------------------------------------------------------ streaming regime, TMA pipeline
// Persistent, warp-specialised form of the sweep (one CTA per SM):
//   warp 0 (one elected lane)  TMA producer: cp.async.bulk.tensor loads of the next tiles into a ring of
//                              TMA_STAGES shared-memory stages (mbarrier complete_tx), and the bulk-tensor
//                              STORES of finished tiles (bulk groups); a stage is reloaded once the store
//                              that read it has drained (cp.async.bulk.wait_group.read);
//   warps 1..                  apply the sweep's gates to the resident tile in place.
// HBM therefore stays busy in both directions while the FP64 pipe works.  The state is described to the
// TMA unit as a 5-d tensor of doubles [16 | low run | gap | main run | rest]; SWIZZLE_128B yields exactly
// the swz() shared-memory layout the gate passes expect.  Tile bits outside the low and main run
// ("scattered") are enumerated as separate boxes.
//
// Live-qubit tracking: a qubit no earlier sweep has had in its tile is still |0>, so amplitudes with such
// a bit set are known zeros.  Sweeps visit only tiles whose fixed bits are live, load only the live part
// of a tile (the rest is zero-filled in shared memory) and store the whole tile; memory outside the live
// region is never read before it is written.  The last sweep of a plan also writes the dead tiles (zeros)
// so that the buffer is complete for the epilogue.  A depth-1 circuit thereby costs about one write of
// the state instead of a read and a write per sweep.
#define TMA_STAGES 3
#define TMA_CONSUMERS 256
#define TMA_MAX_BOXES 128
#define TMA_TILE_DONE 0
#define TMA_TILE_LIVE 1
#define TMA_TILE_DEAD 2

struct TmaSweepDev {
    int n_tile, op_begin, op_end, n_state;
    int init;                 // nothing is live yet: no loads, tile 0 starts as |0..0>
    int has_x;                // the op range holds tile-resolved ops
    int fold_direct;          // last sweep of a plan whose output row is the whole register: store |amp|^2
    int lowc, h, k;           // low run [0, lowc), main run [h, h + k) (state bit positions)
    int n_load, n_store;      // boxes per tile
    unsigned load_bytes;      // bytes per load box
    int zf_shift;             // log2(amplitudes per load box)
    unsigned zf_mask;         // load-box index bits that belong to non-live tile bits: those boxes are zero-filled
    int n_enum_bits;          // work index = (instance << n_enum_bits) | tile number
    int n_local;              // state bits below this index a shard; the bits above are the RANK owning it
    unsigned long long fixed_base;   // bits of every tile base of this launch (sharded runs: rank / owner bits)
    unsigned long long enum_mask;    // state-bit positions the tile number is spread over
    unsigned long long live_before;  // state bits that are live when this sweep starts
    int perm[16];             // ascending tile-local bit -> position in the shared-memory layout
    unsigned long long ld_off[TMA_MAX_BOXES], st_off[TMA_MAX_BOXES];  // amplitude offset of each box in the state
    unsigned ld_slot[TMA_MAX_BOXES], st_slot[TMA_MAX_BOXES];          // first amplitude slot of each box in the stage
};

struct TmaTileDesc {
    unsigned long long base;
    int inst, flags;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* b, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* b, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
// A wait that cannot be satisfied (a faulted TMA operation never completes its transaction bytes) must
// not hang the GPU: after ~2 s the kernel reports which barrier it was and traps.
__device__ __noinline__ void mbar_timeout(int who, unsigned long long tile, int stage, int step) {
    printf("qck: sim_sweep_tma_kernel: %s stuck on tile %llu (stage %d, block %d, consumer step %d)\n",
           who ? "consumer" : "producer", tile, stage, (int)blockIdx.x, step);
    __trap();
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity, int who, unsigned long long tile, int stage,
                                          const volatile int* step) {
    uint32_t ok;
    long long t0 = 0;
    for (uint32_t spins = 0;; ++spins) {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
            : "=r"(ok)
            : "r"(smem_u32(b)), "r"(parity)
            : "memory");
        if (ok) return;
        if ((spins & 1023u) == 1023u) {
            const long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > (who ? 4000000000ll : 6000000000ll) && (threadIdx.x & 31) == 0) mbar_timeout(who, tile, stage, *step);
        }
    }
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* map, uint64_t* bar, int c2, int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(0), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* map, uint32_t src, int c2, int c3, int c4) {
    asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %2, %3, %4, %5}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(map)),
                 "r"(src), "r"(0), "r"(c2), "r"(c3), "r"(c4)
                 : "memory");
}

// One store / load tensor map per shard of the state (a single-GPU run has one shard): in a sharded run the
// rank bits of a box select the PEER buffer it lives in - the TMA unit moves it over NVLink.
#ifndef TMA_MAX_SHARDS
#define TMA_MAX_SHARDS 8
#endif
struct TmaShardMaps {
    CUtensorMap st, ld;
};
struct TmaMaps {  // the maps one tile uses sit next to each other (store, load of shard 0, probabilities)
    TmaShardMaps sh0;
    CUtensorMap pr;
    TmaShardMaps peer[TMA_MAX_SHARDS - 1];  // shards 1 ..
    __host__ __device__ const CUtensorMap* st(int r) const { return r == 0 ? &sh0.st : &peer[r - 1].st; }
    __host__ __device__ const CUtensorMap* ld(int r) const { return r == 0 ? &sh0.ld : &peer[r - 1].ld; }
    __host__ CUtensorMap* st_mut(int r) { return r == 0 ? &sh0.st : &peer[r - 1].st; }
    __host__ CUtensorMap* ld_mut(int r) { return r == 0 ? &sh0.ld : &peer[r - 1].ld; }
};

// WIDE: every lane of the producer warp issues boxes (tiles of many small boxes: 32 boxes of 2 KiB issued by one
// lane took as long as the gate passes); the narrow instantiation keeps the whole producer on one lane, which
// is 12 % faster when a tile is a few large boxes (measured: syc-32 d1, 13.3 vs 15.1 ms).
// SHARDED: the rank bits of a box pick its tensor map at run time; with a single shard the map addresses
// stay compile-time constants of the parameter space (a run-time map address cost the single-GPU
// expansion sweep 13 %: 13.3 -> 15.1 ms).
// The four variants are PLAIN kernels generated from one body (sim_tma_kernel.inc), not template instantiations:
// as instantiations of one template the narrow single-shard kernel ran 12 % slower (14.9 vs 13.3 ms, syc-32 d1).
#define QCK_TMA_KERNEL_NAME sim_sweep_tma_kernel
#define QCK_TMA_WIDE false
#define QCK_TMA_SHARDED false
#include "sim_tma_kernel.inc"
#undef QCK_TMA_KERNEL_NAME
#undef QCK_TMA_WIDE
#undef QCK_TMA_SHARDED
#define QCK_TMA_KERNEL_NAME sim_sweep_tma_wide_kernel
#define QCK_TMA_WIDE true
#define QCK_TMA_SHARDED false
#include "sim_tma_kernel.inc"
#undef QCK_TMA_KERNEL_NAME
#undef QCK_TMA_WIDE
#undef QCK_TMA_SHARDED
#define QCK_TMA_KERNEL_NAME sim_sweep_tma_sharded_kernel
#define QCK_TMA_WIDE false
#define QCK_TMA_SHARDED true
#include "sim_tma_kernel.inc"
#undef QCK_TMA_KERNEL_NAME
#undef QCK_TMA_WIDE
#undef QCK_TMA_SHARDED
#define QCK_TMA_KERNEL_NAME sim_sweep_tma_sharded_wide_kernel
#define QCK_TMA_WIDE true
#define QCK_TMA_SHARDED true
#include "sim_tma_kernel.inc"
#undef QCK_TMA_KERNEL_NAME
#undef QCK_TMA_WIDE
#undef QCK_TMA_SHARDED

__global__ void __launch_bounds__(256) fold_probs_kernel(PlanDev plan, const int32_t* __restrict__ labels,
                                                         int inst_base, const double2* __restrict__ work,
                                                         unsigned long long state_stride,
                                                         double* __restrict__ out, long long row_stride) {
    const int label = labels[inst_base + blockIdx.y];
    const double2* st = work + (unsigned long long)blockIdx.y * state_stride;
    double* row = out + (long long)label * row_stride;
    const uint64_t n_out = 1ull << plan.n_out_bits;
    for (uint64_t o = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; o < n_out;
         o += (uint64_t)gridDim.x * blockDim.x)
        row[o] = fold_entry(plan, o, [&](uint64_t idx) { return __ldcs(st + idx); });
}

// ------------------------------------------------------------------ host side
static int validate_plan(qck_handle* h, const qck_sim_plan* plan) {
    if (!plan) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "plan is NULL");
    if (plan->n_state_qubits < 1 || plan->n_state_qubits > 40)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_state_qubits=%d out of range [1,40]", plan->n_state_qubits);
    if (plan->n_sweeps < 1 || !plan->sweeps) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "plan has no sweeps");
    if (plan->n_digits < 0 || plan->n_digits > QCK_MAX_DIGITS)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_digits=%d out of range", plan->n_digits);
    if (plan->n_out_bits < 0 || plan->n_out_bits > QCK_MAX_OUT_BITS)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "n_out_bits=%d out of range", plan->n_out_bits);
    for (int k = 0; k < plan->n_digits; ++k)
        if (plan->radix[k] < 1) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "radix[%d]=%d", k, plan->radix[k]);
    for (int j = 0; j < plan->n_out_bits; ++j)
        if (plan->out_pos[j] >= plan->n_state_qubits)
            QCK_FAIL(h, QCK_ERR_INVALID_ARG, "out_pos[%d]=%d >= n_state_qubits", j, plan->out_pos[j]);
    for (int i = 0; i < plan->n_sweeps; ++i) {
        const qck_sweep& sw = plan->sweeps[i];
        if (sw.n_tile < 1 || sw.n_tile > QCK_MAX_TILE_QUBITS || sw.n_tile > plan->n_state_qubits)
            QCK_FAIL(h, QCK_ERR_INVALID_ARG, "sweep %d: n_tile=%d invalid", i, sw.n_tile);
        for (int j = 0; j < sw.n_tile; ++j) {
            if (sw.pos[j] < 0 || sw.pos[j] >= plan->n_state_qubits || (j > 0 && sw.pos[j] <= sw.pos[j - 1]))
                QCK_FAIL(h, QCK_ERR_INVALID_ARG, "sweep %d: tile positions must be ascending and < n_state", i);
        }
        if (sw.op_begin < 0 || sw.op_end < sw.op_begin)
            QCK_FAIL(h, QCK_ERR_INVALID_ARG, "sweep %d: bad op range", i);
    }
    if ((plan->n_sweeps > 0 && plan->sweeps[0].op_end > plan->sweeps[0].op_begin) && (!plan->d_ops || !plan->d_mats))
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "plan has ops but d_ops/d_mats is NULL");
    return QCK_OK;
}

static PlanDev to_dev(const qck_sim_plan* plan) {
    PlanDev d;
    memset(&d, 0, sizeof(d));
    d.n_state = plan->n_state_qubits;
    d.ops = plan->d_ops;
    d.mats = plan->d_mats;
    d.n_digits = plan->n_digits;
    for (int k = 0; k < QCK_MAX_DIGITS; ++k) d.radix[k] = k < plan->n_digits ? plan->radix[k] : 1;
    d.n_out_bits = plan->n_out_bits;
    for (int j = 0; j < QCK_MAX_OUT_BITS; ++j) d.out_pos[j] = j < plan->n_out_bits ? plan->out_pos[j] : -1;
    d.out_ident = 0;
    while (d.out_ident < plan->n_out_bits && plan->out_pos[d.out_ident] == d.out_ident) ++d.out_ident;
    d.sum_mask = plan->sum_mask;
    d.sign_mask = plan->sign_mask;
    return d;
}

static SweepDev sweep_dev(const qck_sweep& sw, bool init) {
    SweepDev s;
    memset(&s, 0, sizeof(s));
    s.n_tile = sw.n_tile;
    s.op_begin = sw.op_begin;
    s.op_end = sw.op_end;
    s.init = init ? 1 : 0;
    s.has_x = sw.flags & 1;
    int c = 0;
    while (c < sw.n_tile && sw.pos[c] == c) ++c;
    s.n_low = c;
    for (int j = 0; j < sw.n_tile; ++j) s.pos[j] = sw.pos[j];
    return s;
}

// records to stage for an op range: everything when it fits, else the largest chunk (a cluster of
// up to QCK_MAX_CLUSTER_OPS members + header must fit)
static int stage_records(int n_ops) {
    int n = n_ops < QCK_STAGE_OPS ? n_ops : QCK_STAGE_OPS;
    return n < 1 ? 1 : n;
}

// On-chip: the whole state is one tile.  Two such sweeps with QCK_SWEEP_SHARED on the first = a label-independent
// prefix (run once per plan, sim_onchip_prefix_kernel) followed by the per-instance rest.
static bool has_shared_prefix(const qck_sim_plan* plan) {
    return plan->n_sweeps == 2 && plan->sweeps[0].n_tile == plan->n_state_qubits &&
           plan->sweeps[1].n_tile == plan->n_state_qubits && (plan->sweeps[0].flags & QCK_SWEEP_SHARED);
}
// Register-resident plans (one warp per instance): one sweep flagged QCK_SWEEP_WARP whose tile is the
// fragment's own qubits; the state bits above them are branch outcomes.
static bool is_warp_plan(const qck_sim_plan* plan) {
    return plan->n_sweeps == 1 && (plan->sweeps[0].flags & QCK_SWEEP_WARP);
}
static int warp_base(const qck_sim_plan* plan) { return (plan->sweeps[0].flags >> 8) & 0xff; }
static bool is_onchip(const qck_sim_plan* plan) {
    if (is_warp_plan(plan)) return false;
    return (plan->n_sweeps == 1 && plan->sweeps[0].n_tile == plan->n_state_qubits) || has_shared_prefix(plan);
}

// Runs the shared prefix of an on-chip plan into `snap` (16 << n_state bytes) on `st`.
static int launch_prefix(qck_handle* h, const qck_sim_plan* plan, double2* snap, cudaStream_t st) {
    PlanDev pd = to_dev(plan);
    const qck_sweep& sw = plan->sweeps[0];
    const int N = plan->n_state_qubits;
    pd.n_stage = stage_records(sw.op_end - sw.op_begin);
    size_t smem = ((size_t)16 << N) + sizeof(StagedOp) * pd.n_stage;
    if ((int)smem + 2048 > h->max_smem_optin)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "on-chip plan with %d qubits does not fit shared memory", N);
    int threads = 1 << (N > 3 ? N - 3 : 0);
    if (threads < 32) threads = 32;
    if (threads > 256) threads = 256;
    sim_onchip_prefix_kernel<<<1, threads, smem, st>>>(pd, sw.op_begin, sw.op_end, snap);
    QCK_CHECK_LAUNCH(h);
    return QCK_OK;
}

// ---- TMA sweep: host-side description of one sweep ------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tensor_map_encoder() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

struct TmaShard {  // sharded run: this process holds the amplitudes whose bits >= n_local equal `rank`
    int n_local, rank;
};

struct TmaLaunch {
    TmaSweepDev sd;
    TmaMaps maps;
    unsigned long long n_work;
    size_t smem;
    int n_stage;
};

// records the op stage of the TMA kernel holds: everything when it fits next to the tile ring, else as
// many as fit (the kernel then restages chunks per tile; a header and its members / terms need <= 33)
static int tma_stage_records(int n_tile, int n_ops, int max_smem_optin) {
    const long long room = (long long)max_smem_optin - 512 - 1024 - (long long)TMA_STAGES * ((long long)16 << n_tile);
    long long cap = room / (long long)sizeof(StagedOp);
    if (const char* env = getenv("QCK_TMA_STAGE_CAP")) {  // test knob: force the chunked path
        const long long v = atoll(env);
        if (v >= 48 && v < cap) cap = v;
    }
    if (cap > n_ops) cap = n_ops;
    return (int)(cap < 1 ? 1 : cap);
}
static size_t tma_smem_bytes(int n_tile, int n_records) {
    return 1024 + (size_t)TMA_STAGES * ((size_t)16 << n_tile) + sizeof(StagedOp) * (size_t)(n_records < 1 ? 1 : n_records);
}

// Can this sweep run on the TMA kernel?  (pure host logic, no CUDA calls: unit-testable)
// Fills everything but the tensor maps.  live_before: state bits some earlier sweep had in its tile.
static bool tma_describe(const qck_sim_plan* plan, int i, unsigned long long live_before, bool last, int batch,
                         int max_smem_optin, TmaLaunch& L, const TmaShard* shard = nullptr, bool skip_dead = false) {
    const qck_sweep& sw = plan->sweeps[i];
    const int T = sw.n_tile, N = plan->n_state_qubits;
    const int n_loc = shard ? shard->n_local : N;  // bits a single buffer indexes
    const int n_ops = sw.op_end - sw.op_begin;
    if (T < 3 || T > 13 || n_loc > 35 || n_loc < T || N - n_loc > 3) return false;
    if (shard && batch != 1) return false;
    if (sw.flags & 2) return false;  // register clusters: the TMA kernel carries no cluster code (plain kernel)
    const int n_records = tma_stage_records(T, n_ops, max_smem_optin);
    if (n_records < n_ops && n_records < 48) return false;  // no room for a useful op stage
    int c = 0;
    while (c < T && sw.pos[c] == c) ++c;
    int lowc = c < 11 ? c : 11;
    if (live_before) {  // the low run is loaded as one box: all of it must be live
        int lp = 0;
        while (lp < lowc && ((live_before >> lp) & 1ull)) ++lp;
        lowc = lp;
    }
    if (lowc < 3) return false;
    TmaSweepDev& d = L.sd;
    memset(&d, 0, sizeof(d));
    d.n_tile = T;
    d.op_begin = sw.op_begin;
    d.op_end = sw.op_end;
    d.n_state = N;
    d.init = live_before == 0ull;
    d.has_x = sw.flags & 1;
    d.lowc = lowc;
    d.live_before = live_before;
    // main run: the longest run of consecutive positions among the remaining tile bits (<= 8 bits: box
    // extents are capped at 256), preferring a live one on ties
    int best_b = -1, best_len = 0;
    bool best_live = false;
    for (int j = lowc; j < T;) {
        if (sw.pos[j] >= n_loc) {  // a rank bit: its two values live in different buffers, never inside a box
            ++j;
            continue;
        }
        int e = j;
        while (e + 1 < T && sw.pos[e + 1] == sw.pos[e] + 1 && e + 1 - j < 8 && sw.pos[e + 1] < n_loc) ++e;
        bool live = true;
        for (int q = j; q <= e; ++q) live = live && ((live_before >> sw.pos[q]) & 1ull);
        const int len = e - j + 1;
        if (len > best_len || (len == best_len && live && !best_live)) {
            best_b = j;
            best_len = len;
            best_live = live;
        }
        j = e + 1;
    }
    d.k = best_len;
    d.h = best_len ? sw.pos[best_b] : lowc;
    // shared-memory bit order: low run, main run, scattered bits (ascending)
    int local_pos[16];  // state position of each layout bit
    int n_local = 0;
    for (int j = 0; j < lowc; ++j) {
        d.perm[j] = n_local;
        local_pos[n_local++] = sw.pos[j];
    }
    for (int j = best_b; j >= 0 && j < best_b + best_len; ++j) {
        d.perm[j] = n_local;
        local_pos[n_local++] = sw.pos[j];
    }
    for (int j = lowc; j < T; ++j) {
        if (best_len && j >= best_b && j < best_b + best_len) continue;
        d.perm[j] = n_local;
        local_pos[n_local++] = sw.pos[j];
    }
    const int n_scat = T - lowc - best_len;
    // stores: one box [low | main] per combination of the scattered bits
    if (n_scat > 7) return false;
    d.n_store = 1 << n_scat;
    for (int i2 = 0; i2 < d.n_store; ++i2) {
        unsigned long long off = 0;
        for (int b2 = 0; b2 < n_scat; ++b2)
            if ((i2 >> b2) & 1) off |= 1ull << local_pos[lowc + best_len + b2];
        d.st_off[i2] = off;
        d.st_slot[i2] = (unsigned)i2 << (lowc + best_len);
    }
    // loads: the box covers [low | main] when the whole main run is live, else the low run only; one
    // box per combination of the LIVE layout bits above the box, the others stay zero
    const bool box_main = best_live || best_len == 0;
    const int box_bits = box_main ? lowc + best_len : lowc;
    d.zf_shift = box_bits;
    d.load_bytes = 16u << box_bits;
    unsigned live_hi = 0, dead_hi = 0;  // over layout bits >= box_bits, shifted down
    for (int b2 = box_bits; b2 < T; ++b2) {
        if ((live_before >> local_pos[b2]) & 1ull) live_hi |= 1u << (b2 - box_bits);
        else dead_hi |= 1u << (b2 - box_bits);
    }
    d.zf_mask = dead_hi;
    if (d.init) {
        d.n_load = 0;
    } else {
        const int n_live_hi = __builtin_popcount(live_hi);
        if (n_live_hi > 7) return false;
        d.n_load = 1 << n_live_hi;
        for (int i2 = 0; i2 < d.n_load; ++i2) {
            const unsigned hi = (unsigned)soft_pdep((uint64_t)i2, (uint64_t)live_hi);
            unsigned long long off = 0;
            for (int b2 = box_bits; b2 < T; ++b2)
                if ((hi >> (b2 - box_bits)) & 1u) off |= 1ull << local_pos[b2];
            d.ld_off[i2] = off;
            d.ld_slot[i2] = hi << box_bits;
        }
    }
    // work list: tiles whose fixed bits are live (the last sweep also visits - and zero-fills - the others)
    unsigned long long tile_mask = 0;
    for (int j = 0; j < T; ++j) tile_mask |= 1ull << sw.pos[j];
    const unsigned long long all = N >= 64 ? ~0ull : ((1ull << N) - 1ull);
    d.n_local = n_loc;
    // (skip_dead: the caller has zero-filled the dead region itself - zero_dead_kernel - so the last sweep visits
    // the live tiles only, like every other sweep)
    d.enum_mask = ((last && !skip_dead) ? all : live_before) & ~tile_mask;
    if (shard) {
        // Which rank works on which tile: the rank bits OUTSIDE the tile are the rank's own (its shard); for
        // every rank bit INSIDE the tile (the tile spans the buffers of two ranks) one of the highest non-tile
        // local positions - a live one when there is one - is pinned to the rank's bit instead, so that every
        // tile has exactly one owner and the owners share the live tiles evenly.
        const unsigned long long rank_mask = all & ~((1ull << n_loc) - 1ull);
        unsigned long long fixed = ((unsigned long long)shard->rank << n_loc) & ~tile_mask, owner_mask = 0;
        for (int b = n_loc; b < N; ++b) {
            if (!((tile_mask >> b) & 1ull)) continue;
            int pick = -1;
            for (int pass = 0; pass < 2 && pick < 0; ++pass)  // first pass: live positions only
                for (int p = n_loc - 1; p >= 0 && pick < 0; --p)
                    if (!((tile_mask >> p) & 1ull) && !((owner_mask >> p) & 1ull) && (pass == 1 || ((live_before >> p) & 1ull)))
                        pick = p;
            if (pick < 0) return false;
            owner_mask |= 1ull << pick;
            fixed |= (unsigned long long)((shard->rank >> (b - n_loc)) & 1) << pick;
        }
        d.fixed_base = fixed;
        d.enum_mask &= ~rank_mask & ~owner_mask;
    }
    d.n_enum_bits = __builtin_popcountll(d.enum_mask);
    L.n_work = (unsigned long long)batch << d.n_enum_bits;
    if (shard && !last && (d.fixed_base & ~live_before)) L.n_work = 0;  // every tile of this rank is still all zero
    L.smem = tma_smem_bytes(T, n_records);
    L.n_stage = n_records;
    // extents the tensor map can describe
    if (((unsigned long long)batch << (n_loc - d.h - d.k)) > 0xffffffffull) return false;
    return true;
}

static int tma_encode(qck_handle* h, const TmaSweepDev& d, int batch, double2* work, bool box_main, CUtensorMap* out) {
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc) QCK_FAIL(h, QCK_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    const int N = d.n_local, top = d.h + d.k;
    cuuint64_t dims[5] = {16ull, 1ull << (d.lowc - 3), 1ull << (d.h - d.lowc), 1ull << d.k,
                          (cuuint64_t)batch << (N - top)};
    cuuint64_t strides[4] = {128ull, 16ull << d.lowc, 16ull << d.h, 16ull << top};
    cuuint32_t box[5] = {16u, 1u << (d.lowc - 3), 1u, box_main ? (1u << d.k) : 1u, 1u};
    cuuint32_t estr[5] = {1u, 1u, 1u, 1u, 1u};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 5, (void*)work, dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        QCK_FAIL(h, QCK_ERR_CUDA,
                 "cuTensorMapEncodeTiled failed (%d): dims {16,%llu,%llu,%llu,%llu} box {16,%u,1,%u,1} lowc=%d h=%d k=%d", (int)r,
                 (unsigned long long)dims[1], (unsigned long long)dims[2], (unsigned long long)dims[3],
                 (unsigned long long)dims[4], box[1], box[3], d.lowc, d.h, d.k);
    return QCK_OK;
}

// Output row as a tensor of doubles with the geometry of the state map (8 doubles = 8 amplitudes per inner
// row, no swizzle): the fused fold stores |amp|^2 of a finished tile straight into the row.
static int tma_encode_probs(qck_handle* h, const TmaSweepDev& d, double* row, CUtensorMap* out) {
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc) QCK_FAIL(h, QCK_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    const int N = d.n_state, top = d.h + d.k;
    cuuint64_t dims[5] = {8ull, 1ull << (d.lowc - 3), 1ull << (d.h - d.lowc), 1ull << d.k, 1ull << (N - top)};
    cuuint64_t strides[4] = {64ull, 8ull << d.lowc, 8ull << d.h, 8ull << top};
    cuuint32_t box[5] = {8u, 1u << (d.lowc - 3), 1u, 1u << d.k, 1u};
    cuuint32_t estr[5] = {1u, 1u, 1u, 1u, 1u};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 5, (void*)row, dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        QCK_FAIL(h, QCK_ERR_CUDA, "cuTensorMapEncodeTiled (probabilities) failed (%d): lowc=%d h=%d k=%d", (int)r, d.lowc, d.h, d.k);
    return QCK_OK;
}

// Exposed for the host-logic tests (no GPU needed): describe sweep `i` of `plan` the way the TMA kernel
// would run it.  Returns 1 and fills the arrays when the sweep is eligible, else 0.
extern "C" int qck_debug_tma_describe(const qck_sim_plan* plan, int sweep, uint64_t live_before, int last,
                                              int batch, int n_local, int rank,
                                              int32_t* geom /*[8]: lowc,h,k,n_load,n_store,zf_shift,zf_mask,n_enum_bits*/,
                                              int32_t* perm /*[16]*/, uint64_t* ld_off, uint32_t* ld_slot, uint64_t* st_off,
                                              uint32_t* st_slot, uint64_t* enum_mask, uint64_t* n_work, uint64_t* fixed_base) {
    static TmaLaunch L;  // large: keep it off the stack; debug entry point, not re-entrant
    if (!plan || sweep < 0 || sweep >= plan->n_sweeps) return 0;
    TmaShard sh = {n_local, rank};
    if (!tma_describe(plan, sweep, live_before, last != 0, batch, 232448, L, n_local > 0 ? &sh : nullptr)) return 0;
    const TmaSweepDev& d = L.sd;
    const int32_t g[8] = {d.lowc, d.h, d.k, d.n_load, d.n_store, d.zf_shift, (int32_t)d.zf_mask, d.n_enum_bits};
    for (int j = 0; j < 8; ++j) geom[j] = g[j];
    for (int j = 0; j < 16; ++j) perm[j] = d.perm[j];
    for (int j = 0; j < d.n_load; ++j) {
        ld_off[j] = d.ld_off[j];
        ld_slot[j] = d.ld_slot[j];
    }
    for (int j = 0; j < d.n_store; ++j) {
        st_off[j] = d.st_off[j];
        st_slot[j] = d.st_slot[j];
    }
    *enum_mask = d.enum_mask;
    *n_work = L.n_work;
    if (fixed_base) *fixed_base = d.fixed_base;
    return 1;
}

static int tma_mode();

// Exact HBM traffic of the sweeps of `plan` for `batch` instances (host arithmetic only): what the TMA
// path loads and stores with live-qubit tracking, or - when a sweep is not eligible for it - the plain
// kernel's read + write of the whole state per sweep.
extern "C" int qck_sim_plan_traffic(const qck_sim_plan* plan, int batch, int fold_fused, uint64_t* bytes_loaded,
                                    uint64_t* bytes_stored, int* uses_tma) {
    if (!plan || !plan->sweeps || batch < 1 || !bytes_loaded || !bytes_stored) return QCK_ERR_INVALID_ARG;
    std::unique_ptr<TmaLaunch> L(new TmaLaunch);
    bool tma = tma_mode() != 0;
    unsigned long long live = 0, ld = 0, st = 0;
    for (int i = 0; i < plan->n_sweeps && tma; ++i) {
        tma = tma_describe(plan, i, live, i == plan->n_sweeps - 1, batch, 232448, *L);
        if (!tma) break;
        const TmaSweepDev& d = L->sd;
        // live tiles: the tile number is spread over enum_mask; a tile is live iff its bits outside the live set are 0
        const unsigned long long live_tiles = (unsigned long long)batch << __builtin_popcountll(d.enum_mask & live);
        ld += live_tiles * (unsigned long long)d.n_load * d.load_bytes;
        // the fused fold stores 8-byte probabilities instead of 16-byte amplitudes in the last sweep
        st += L->n_work * ((unsigned long long)((fold_fused && i == plan->n_sweeps - 1) ? 8 : 16) << d.n_tile);
        for (int j = 0; j < plan->sweeps[i].n_tile; ++j) live |= 1ull << plan->sweeps[i].pos[j];
    }
    if (!tma) {
        const unsigned long long full = ((unsigned long long)16 << plan->n_state_qubits) * (unsigned long long)batch;
        ld = full * (unsigned long long)(plan->n_sweeps - 1);
        st = full * (unsigned long long)plan->n_sweeps;
    }
    *bytes_loaded = ld;
    *bytes_stored = st;
    if (uses_tma) *uses_tma = tma ? 1 : 0;
    return QCK_OK;
}

static bool fold_fusion_enabled() {  // QCK_FOLD_FUSION=0: always run the separate fold pass (tuning / test knob)
    const char* env = getenv("QCK_FOLD_FUSION");
    return env ? atoi(env) != 0 : true;
}

static int tma_mode() {  // QCK_SIM_TMA: 0 = never, 1 = when eligible (default)
    const char* env = getenv("QCK_SIM_TMA");
    return env ? atoi(env) : 1;
}

// fold_row != NULL: the caller wants the probabilities of the single instance in fold_row instead of the
// final state (only honoured - *folded = true - when the plan runs on the TMA kernels).
// Zero-fill of the DEAD region of a state / probability row: the indices with a bit set that no sweep ever had
// in a tile (that qubit is still |0>).  The last sweep used to write those tiles itself - zero-filling a
// shared-memory stage and TMA-storing it, tile by tile, through the full producer / consumer hand-shake: for a
// shallow circuit that is almost the whole buffer (uncut syc-32 d1: 2^23 of 2^32 amplitudes are ever non-zero)
// and ran at 0.46 of the HBM peak.  A plain streaming store kernel does it at memset speed, before the sweeps.
// One warp per run of 2^c contiguous elements (c = contiguous low live bits).
__global__ void __launch_bounds__(256) zero_dead_kernel(unsigned char* __restrict__ base, unsigned long long inst_stride_bytes,
                                                        int n_bits, unsigned long long live_after, int c, int log_es) {
    const unsigned long long n_runs = 1ull << (n_bits - c);
    const unsigned long long run_bytes = (1ull << c) << log_es;
    const int lane = threadIdx.x & 31;
    const unsigned long long n_warps = (unsigned long long)gridDim.x * (blockDim.x >> 5);
    unsigned char* inst = base + (unsigned long long)blockIdx.y * inst_stride_bytes;
    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
    for (unsigned long long r = (unsigned long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < n_runs; r += n_warps) {
        if (((r << c) & ~live_after) == 0ull) continue;  // a live run: the sweeps write it
        uint4* dst = reinterpret_cast<uint4*>(inst + r * run_bytes);
        for (unsigned long long o = lane; o < run_bytes / 16ull; o += 32) __stcs(dst + o, z);
    }
}

static int zero_dead_region(qck_handle* h, void* base, unsigned long long inst_stride_bytes, int batch, int n_bits,
                            unsigned long long live_after, int log_es, cudaStream_t st) {
    int c = 0;
    while (c < n_bits && ((live_after >> c) & 1ull)) ++c;
    if (c >= n_bits) return QCK_OK;  // nothing dead
    if (((1ull << c) << log_es) < 512ull) c = 0;  // (tiles always hold qubits 0-4: runs are >= 256 bytes; be safe)
    unsigned long long runs = 1ull << (n_bits - c);
    unsigned long long grid = (runs + 7) / 8;
    if (grid > (unsigned long long)h->sm_count * 16) grid = (unsigned long long)h->sm_count * 16;
    zero_dead_kernel<<<dim3((unsigned)grid, (unsigned)batch), 256, 0, st>>>(reinterpret_cast<unsigned char*>(base), inst_stride_bytes,
                                                                           n_bits, live_after, c, log_es);
    QCK_CHECK_LAUNCH(h);
    return QCK_OK;
}

static int run_sweeps(qck_handle* h, const qck_sim_plan* plan, const PlanDev& pd, const int32_t* d_labels,
                      int inst_base, int batch, double2* work, unsigned long long state_stride,
                      cudaStream_t st, double* fold_row = nullptr, bool* folded = nullptr) {
    if (folded) *folded = false;
    // The TMA kernels track live qubits, i.e. they leave memory outside the live region unwritten between
    // sweeps: a plan runs either entirely on them or entirely on the plain kernel.
    bool use_tma = tma_mode() != 0 && state_stride == (1ull << plan->n_state_qubits) && tensor_map_encoder() != nullptr;
    std::unique_ptr<TmaLaunch> L(use_tma ? new TmaLaunch : nullptr);  // ~5 KB of kernel parameters: off the stack
    if (use_tma) {
        unsigned long long live = 0;
        for (int i = 0; i < plan->n_sweeps && use_tma; ++i) {
            use_tma = tma_describe(plan, i, live, i == plan->n_sweeps - 1, batch, h->max_smem_optin, *L);
            for (int j = 0; j < plan->sweeps[i].n_tile; ++j) live |= 1ull << plan->sweeps[i].pos[j];
        }
    }
    if (use_tma) {
        unsigned long long live = 0;
        // The dead region is zero-filled by a streaming kernel up front; the last sweep then visits the live tiles
        // only.  (The sharded sweeps instead have their last sweep write the dead tiles: skip_dead = false.)
        bool prezero = true;
        {
            unsigned long long live_after = 0;
            for (int i = 0; i < plan->n_sweeps; ++i)
                for (int j = 0; j < plan->sweeps[i].n_tile; ++j) live_after |= 1ull << plan->sweeps[i].pos[j];
            const unsigned long long all = plan->n_state_qubits >= 64 ? ~0ull : ((1ull << plan->n_state_qubits) - 1ull);
            if ((live_after & all) == all) prezero = false;  // nothing is dead
            if (prezero) {
                const bool to_row = fold_row && batch == 1;
                int rc = zero_dead_region(h, to_row ? (void*)fold_row : (void*)work, state_stride * 16ull, to_row ? 1 : batch,
                                          plan->n_state_qubits, live_after, to_row ? 3 : 4, st);
                if (rc) return rc;
            }
        }
        // Tile scheduling: static round robin.  Pulling tiles from a counter measured 1-2 % faster on
        // compute-heavy sweeps but 13 % slower on the write-only expansion sweep of syc-32 d1 (15.1 vs
        // 13.4 ms): neighbouring CTAs on neighbouring tiles suit the TMA stores.
        for (int i = 0; i < plan->n_sweeps; ++i) {
            tma_describe(plan, i, live, i == plan->n_sweeps - 1, batch, h->max_smem_optin, *L, nullptr, prezero);
            for (int j = 0; j < plan->sweeps[i].n_tile; ++j) live |= 1ull << plan->sweeps[i].pos[j];
            int rc = tma_encode(h, L->sd, batch, work, true, &L->maps.sh0.st);
            if (rc) return rc;
            const bool box_main = L->sd.zf_shift == L->sd.lowc + L->sd.k;
            rc = tma_encode(h, L->sd, batch, work, box_main, &L->maps.sh0.ld);
            if (rc) return rc;
            L->maps.pr = L->maps.sh0.st;
            if (fold_row && batch == 1 && i == plan->n_sweeps - 1) {
                rc = tma_encode_probs(h, L->sd, fold_row, &L->maps.pr);
                if (rc) return rc;
                L->sd.fold_direct = 1;
                if (folded) *folded = true;
            }
            PlanDev pdl = pd;
            pdl.n_stage = L->n_stage;
            unsigned long long grid = L->n_work < (unsigned long long)h->sm_count ? L->n_work : (unsigned long long)h->sm_count;
            if (L->sd.n_store >= 16 || L->sd.n_load >= 16)  // measured: 8 boxes of 8 KiB are still faster from one lane
                sim_sweep_tma_wide_kernel<<<(unsigned)grid, TMA_CONSUMERS + 32, L->smem, st>>>(
                    L->maps, L->sd, pdl, d_labels, inst_base, L->n_work);
            else
                sim_sweep_tma_kernel<<<(unsigned)grid, TMA_CONSUMERS + 32, L->smem, st>>>(
                    L->maps, L->sd, pdl, d_labels, inst_base, L->n_work);
            QCK_CHECK_LAUNCH(h);
        }
        return QCK_OK;
    }
    for (int i = 0; i < plan->n_sweeps; ++i) {
        SweepDev sd = sweep_dev(plan->sweeps[i], i == 0);
        if (sd.n_tile - sd.n_low > 10)
            QCK_FAIL(h, QCK_ERR_UNSUPPORTED, "sweep %d: more than 10 non-contiguous tile bits", i);
        PlanDev pdl = pd;
        pdl.n_stage = stage_records(sd.op_end - sd.op_begin);
        const size_t aux = ((((size_t)8 << (sd.n_tile - sd.n_low)) + 15) & ~(size_t)15) + sizeof(StagedOp) * pdl.n_stage;
        size_t smem = ((size_t)16 << sd.n_tile) + aux;
        if ((int)smem + 1024 > h->max_smem_optin)
            QCK_FAIL(h, QCK_ERR_INVALID_ARG, "sweep %d: tile of 2^%d amplitudes does not fit shared memory", i,
                     sd.n_tile);
        unsigned long long tiles = 1ull << (plan->n_state_qubits - sd.n_tile);
        if (tiles > 0x7fffffffull) QCK_FAIL(h, QCK_ERR_UNSUPPORTED, "too many tiles");
        dim3 grid((unsigned)tiles, (unsigned)batch);
        // many tiles: 128 threads, 3 CTAs per SM de-phase load / compute / store (256 threads: 2 phase-locked CTAs);
        // few tiles (L2-resident states): latency bound, use all 256 threads per tile
        const int sweep_threads = tiles * (unsigned long long)batch >= 4ull * h->sm_count ? 128 : 256;
        sim_sweep_kernel<<<grid, sweep_threads, smem, st>>>(pdl, sd, d_labels, inst_base, work, state_stride);
        QCK_CHECK_LAUNCH(h);
    }
    return QCK_OK;
}

static int qck_warp_init(qck_handle* h);
static int qck_tree_init(qck_handle* h);
static int pick_side_stream(qck_handle* h, unsigned* used, cudaStream_t* st);
static int region_fork_call(qck_handle* h, cudaStream_t main_st);
static int warp_single_plan(qck_handle* h, const qck_sim_plan* plan, const int32_t* d_labels, int64_t n_instances,
                            double* d_out, int64_t out_row_stride, cudaStream_t st);

extern "C" int qck_sim_fragments(qck_handle* h, const qck_sim_plan* plan, const int32_t* d_labels,
                                 int64_t n_instances, double* d_out, int64_t out_row_stride, void* d_work,
                                 size_t work_bytes, qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    int rc = validate_plan(h, plan);
    if (rc) return rc;
    if (n_instances == 0) return QCK_OK;
    if (n_instances < 0 || !d_labels || !d_out) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "bad instance list / output");
    if (out_row_stride < (1ll << plan->n_out_bits))
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "out_row_stride smaller than the row (2^%d)", plan->n_out_bits);
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (is_warp_plan(plan)) return warp_single_plan(h, plan, d_labels, n_instances, d_out, out_row_stride, st);
    PlanDev pd = to_dev(plan);
    if (is_onchip(plan)) {
        const int N = plan->n_state_qubits;
        const qck_sweep& sw0 = plan->sweeps[0];
        pd.n_stage = stage_records(sw0.op_end - sw0.op_begin);
        size_t smem = ((size_t)16 << N) + sizeof(StagedOp) * pd.n_stage;
        if ((int)smem + 1024 > h->max_smem_optin)
            QCK_FAIL(h, QCK_ERR_INVALID_ARG, "on-chip plan with %d qubits does not fit shared memory", N);
        int threads = 1 << (N > 3 ? N - 3 : 0);  // one thread per group of 8 amplitudes
        if (threads < 32) threads = 32;
        if (threads > 256) threads = 256;
        const bool shared = has_shared_prefix(plan);
        const qck_sweep& sw = plan->sweeps[shared ? 1 : 0];
        const double2* init = nullptr;
        if (shared) {
            if (!d_work || work_bytes < ((size_t)16 << N))
                QCK_FAIL(h, QCK_ERR_INVALID_ARG, "a plan with a shared prefix needs %zu bytes of work space, got %zu",
                         (size_t)16 << N, work_bytes);
            rc = launch_prefix(h, plan, (double2*)d_work, st);
            if (rc) return rc;
            init = (const double2*)d_work;
            const int st1 = stage_records(sw.op_end - sw.op_begin);
            if (st1 > pd.n_stage) pd.n_stage = st1;
            smem = ((size_t)16 << N) + sizeof(StagedOp) * pd.n_stage;
        }
        for (int64_t done = 0; done < n_instances;) {
            int64_t batch = n_instances - done;
            if (batch > (1ll << 30)) batch = 1ll << 30;
            sim_onchip_kernel<<<(unsigned)batch, threads, smem, st>>>(pd, sw.op_begin, sw.op_end, d_labels + done,
                                                                       d_out, (long long)out_row_stride, init);
            QCK_CHECK_LAUNCH(h);
            done += batch;
        }
        return QCK_OK;
    }
    // streaming regime
    const unsigned long long state_amps = 1ull << plan->n_state_qubits;
    const size_t state_bytes = (size_t)state_amps * 16;
    if (!d_work || work_bytes < state_bytes)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "streaming regime needs >= %zu bytes of work space, got %zu", state_bytes,
                 work_bytes);
    int64_t cap = (int64_t)(work_bytes / state_bytes);
    if (cap > 65535) cap = 65535;
    for (int64_t done = 0; done < n_instances;) {
        int batch = (int)((n_instances - done) < cap ? (n_instances - done) : cap);
        // The output row is the whole register (uncut circuit, every qubit measured into its own clbit, one
        // instance): the last sweep stores |amp|^2 straight into the row - no final state, no fold pass.
        const bool direct = plan->n_digits == 0 && n_instances == 1 && pd.out_ident == plan->n_out_bits &&
                            plan->n_out_bits == plan->n_state_qubits && plan->sum_mask == 0 && plan->sign_mask == 0 &&
                            fold_fusion_enabled();
        bool folded = false;
        rc = run_sweeps(h, plan, pd, d_labels, (int)done, batch, (double2*)d_work, state_amps, st,
                        direct ? d_out : nullptr, &folded);  // one instance without digits: label 0, row 0
        if (rc) return rc;
        if (folded) {
            done += batch;
            continue;
        }
        unsigned long long n_out = 1ull << plan->n_out_bits;
        unsigned gx = (unsigned)((n_out + 255) / 256 < 148ull * 16 ? (n_out + 255) / 256 : 148ull * 16);
        fold_probs_kernel<<<dim3(gx, batch), 256, 0, st>>>(pd, d_labels, (int)done, (const double2*)d_work,
                                                             state_amps, d_out, (long long)out_row_stride);
        QCK_CHECK_LAUNCH(h);
        done += batch;
    }
    return QCK_OK;
}

// Opt-in shared-memory limits are per-function process state: set them ONCE to the device maximum
// (at handle creation) - setting them per launch races between host threads.
int qck_sim_init(qck_handle* h) {
    QCK_CUDA(h, qck_allow_max_smem(sim_onchip_kernel, h->max_smem_optin));
    QCK_CUDA(h, qck_allow_max_smem(sim_onchip_prefix_kernel, h->max_smem_optin));
    QCK_CUDA(h, qck_allow_max_smem(sim_onchip_group_kernel, h->max_smem_optin));
    QCK_CUDA(h, qck_allow_max_smem(sim_sweep_kernel, h->max_smem_optin));
    QCK_CUDA(h, qck_allow_max_smem(sim_sweep_tma_kernel, h->max_smem_optin));
    QCK_CUDA(h, qck_allow_max_smem(sim_sweep_tma_wide_kernel, h->max_smem_optin));
    QCK_CUDA(h, qck_allow_max_smem(sim_sweep_tma_sharded_kernel, h->max_smem_optin));
    QCK_CUDA(h, qck_allow_max_smem(sim_sweep_tma_sharded_wide_kernel, h->max_smem_optin));
    int rc = qck_warp_init(h);
    return rc ? rc : qck_tree_init(h);
}

typedef void (*WarpKernelFn)(const WarpGroupDev, double*, long long);
static WarpKernelFn warp_kernel(int log_r) {
    switch (log_r) {
        case 0: return sim_warp_kernel<0>;
        case 1: return sim_warp_kernel<1>;
        case 2: return sim_warp_kernel<2>;
        case 3: return sim_warp_kernel<3>;
        case 4: return sim_warp_kernel<4>;
        default: return sim_warp_kernel<5>;
    }
}

static int qck_warp_init(qck_handle* h) {
    for (int r = 0; r <= 5; ++r) {
        const int smem = QCK_WARP_PER_CTA * ((32 << (r + 5)) + (int)sizeof(WarpStagedOp) * QCK_WARP_STAGE);
        QCK_CUDA(h, cudaFuncSetAttribute(warp_kernel(r), cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        int occ = 0;
        QCK_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, warp_kernel(r), 32 * QCK_WARP_PER_CTA, smem));
        h->warp_occ[r] = occ < 1 ? 1 : occ;
    }
    return QCK_OK;
}

#define WARP_DFS_LEVELS 2  // outcome levels one warp walks itself; the levels above are split over warps

// A group of register-resident plans (same fragment qubit count) = one launch.  warp_group_layout fills the
// kernel parameters and says how much scratch the launch needs ([global stash | partial rows | counters]);
// warp_group_launch binds the scratch and launches.
struct WarpGroupHost {
    WarpGroupDev G;
    int log_r;
    long long ctas;
    size_t stash_bytes, part_bytes, cnt_bytes;
};

static int warp_group_layout(qck_handle* h, const qck_sim_plan* plans, const int* idx, int n,
                             const int32_t* const* d_labels, const int64_t* n_instances, int64_t out_row_stride,
                             WarpGroupHost* W) {
    WarpGroupDev& G = W->G;
    memset(W, 0, sizeof(*W));
    const qck_sim_plan& p0 = plans[idx[0]];
    G.n_base = warp_base(&p0);
    G.n_vars = n;
    G.n_digits = p0.n_digits;
    G.ops = p0.d_ops;
    G.mats = p0.d_mats;
    long long div = 1;
    for (int k = QCK_MAX_DIGITS - 1; k >= 0; --k) {
        G.radix[k] = k < p0.n_digits ? p0.radix[k] : 1;
        G.div[k] = (int)div;
        if (k < p0.n_digits) div *= p0.radix[k];
        if (div > 0x7fffffffll) QCK_FAIL(h, QCK_ERR_UNSUPPORTED, "fragment label space exceeds 2^31");
    }
    long long items = 0, parts = 0, cnts = 0;
    int max_walk = 0;
    for (int i = 0; i < n; ++i) {
        const qck_sim_plan& p = plans[idx[i]];
        if (p.d_ops != p0.d_ops || p.d_mats != p0.d_mats || p.n_digits != p0.n_digits || warp_base(&p) != G.n_base)
            QCK_FAIL(h, QCK_ERR_INVALID_ARG, "plans of one batch must share the program blob and the label radices");
        if (out_row_stride < (1ll << p.n_out_bits))
            QCK_FAIL(h, QCK_ERR_INVALID_ARG, "out_row_stride smaller than the row (2^%d)", p.n_out_bits);
        const int n_anc = p.n_state_qubits - G.n_base;
        if (n_anc < 0 || n_anc > QCK_WARP_MAX_DEPTH || G.n_base < 1 || G.n_base > 10 || p.n_out_bits > 30 ||
            p.sweeps[0].op_end - p.sweeps[0].op_begin > 60000)
            QCK_FAIL(h, QCK_ERR_INVALID_ARG, "register-resident plan out of range (%d qubits, %d branch points)",
                     G.n_base, n_anc);
        // the leaves are signed by every sign_mask bit and all of them are added: a sign on an unsummed bit, or an
        // outcome bit that is neither a row bit nor summed, would give other rows than the shared-memory kernels
        unsigned long long row_bits = 0;
        for (int j = 0; j < p.n_out_bits; ++j)
            if (p.out_pos[j] >= 0) row_bits |= 1ull << p.out_pos[j];
        if (p.sign_mask & ~p.sum_mask)
            QCK_FAIL(h, QCK_ERR_INVALID_ARG, "register-resident plan: sign_mask bits outside sum_mask");
        for (int a = G.n_base; a < p.n_state_qubits; ++a)
            if (!(((p.sum_mask | row_bits) >> a) & 1ull))
                QCK_FAIL(h, QCK_ERR_INVALID_ARG, "register-resident plan: outcome bit %d is neither a row bit nor summed", a);
        WarpVarDev& v = G.var[i];
        v.op_begin = p.sweeps[0].op_begin;
        v.op_end = p.sweeps[0].op_end;
        v.n_out_bits = p.n_out_bits;
        v.n_anc = n_anc;
        int n_free = 0;
        v.mode = QCK_WARP_MODE_ACC;
        for (int j = 0; j < QCK_MAX_OUT_BITS; ++j) {
            v.out_pos[j] = (signed char)(j < p.n_out_bits ? p.out_pos[j] : -1);
            if (j < p.n_out_bits && p.out_pos[j] >= G.n_base) v.mode = QCK_WARP_MODE_RMW;  // an outcome is a column bit
            if (j < p.n_out_bits && p.out_pos[j] >= 0 && p.out_pos[j] < G.n_base) ++n_free;
        }
        v.sum_mask = p.sum_mask;
        v.sign_mask = p.sign_mask;
        v.labels = d_labels[idx[i]];
        v.split_bits = (v.mode == QCK_WARP_MODE_ACC && n_anc > WARP_DFS_LEVELS) ? n_anc - WARP_DFS_LEVELS : 0;
        const int walk = n_anc - v.split_bits;
        if (walk > max_walk) max_walk = walk;
        v.item_begin = (int)items;
        items += n_instances[idx[i]] << v.split_bits;
        v.cnt_off = (int)cnts;
        v.part_off = parts;
        if (v.split_bits > 0) {
            cnts += n_instances[idx[i]];
            parts += (n_instances[idx[i]] << v.split_bits) << n_free;
        }
        if (items > 0x7fffffffll || cnts > 0x7fffffffll) QCK_FAIL(h, QCK_ERR_UNSUPPORTED, "too many instances in one group");
    }
    G.total = (int)items;
    W->log_r = G.n_base > 5 ? G.n_base - 5 : 0;
    W->ctas = (items + QCK_WARP_PER_CTA - 1) / QCK_WARP_PER_CTA;
    const long long cap = (long long)h->sm_count * h->warp_occ[W->log_r];
    if (W->ctas > cap) W->ctas = cap;
    W->stash_bytes = max_walk > QCK_WARP_SMEM_LEVELS
                         ? (size_t)W->ctas * QCK_WARP_PER_CTA * QCK_WARP_MAX_DEPTH * (32u << W->log_r) * sizeof(double2)
                         : 0;
    W->part_bytes = ((size_t)parts * sizeof(double) + 255) & ~(size_t)255;
    W->cnt_bytes = ((size_t)cnts * sizeof(unsigned) + 255) & ~(size_t)255;
    return QCK_OK;
}

// scratch layout of the handle: [counters of every group (zero between launches) | stash + partial rows ...]
static int warp_groups_run(qck_handle* h, WarpGroupHost* W, int n_groups, cudaStream_t* streams, double* d_out,
                           int64_t out_row_stride) {
    const int cs = h->region ? (int)(h->region_calls++ % QCK_SIDE_STREAMS) : 0;  // scratch slot of this call
    size_t cnt_total = 0, rest_total = 0;
    for (int g = 0; g < n_groups; ++g) {
        cnt_total += W[g].cnt_bytes;
        rest_total += W[g].stash_bytes + W[g].part_bytes;
    }
    const size_t need = cnt_total + rest_total;
    if (need > h->warp_stash_bytes[cs]) {  // grows only; synchronous, first use of a larger shape only
        if (h->warp_stash[cs]) QCK_CUDA(h, cudaFree(h->warp_stash[cs]));
        h->warp_stash[cs] = nullptr;
        h->warp_stash_bytes[cs] = 0;
        const size_t want = need + (need >> 2);
        cudaError_t e = cudaMalloc(&h->warp_stash[cs], want);
        if (e != cudaSuccess) QCK_FAIL(h, QCK_ERR_NOMEM, "cudaMalloc(%zu bytes of branch scratch): %s", want, cudaGetErrorString(e));
        h->warp_stash_bytes[cs] = want;
        h->warp_cnt_bytes[cs] = 0;
    }
    if (cnt_total > h->warp_cnt_bytes[cs]) {  // the counter region grew over bytes that held other data: zero it once
        QCK_CUDA(h, cudaMemset(h->warp_stash[cs], 0, cnt_total));
        h->warp_cnt_bytes[cs] = cnt_total;
    }
    char* cnt_ptr = reinterpret_cast<char*>(h->warp_stash[cs]);
    char* rest_ptr = cnt_ptr + h->warp_cnt_bytes[cs];
    if (h->warp_cnt_bytes[cs] + rest_total > h->warp_stash_bytes[cs]) {  // counters once needed more than now: regrow
        QCK_CUDA(h, cudaFree(h->warp_stash[cs]));
        h->warp_stash[cs] = nullptr;
        const size_t want = h->warp_cnt_bytes[cs] + rest_total + (rest_total >> 2);
        cudaError_t e = cudaMalloc(&h->warp_stash[cs], want);
        if (e != cudaSuccess) QCK_FAIL(h, QCK_ERR_NOMEM, "cudaMalloc(%zu bytes of branch scratch): %s", want, cudaGetErrorString(e));
        h->warp_stash_bytes[cs] = want;
        QCK_CUDA(h, cudaMemset(h->warp_stash[cs], 0, h->warp_cnt_bytes[cs]));
        cnt_ptr = reinterpret_cast<char*>(h->warp_stash[cs]);
        rest_ptr = cnt_ptr + h->warp_cnt_bytes[cs];
    }
    for (int g = 0; g < n_groups; ++g) {
        WarpGroupDev& G = W[g].G;
        G.cnt = reinterpret_cast<unsigned*>(cnt_ptr);
        cnt_ptr += W[g].cnt_bytes;
        G.stash = W[g].stash_bytes ? reinterpret_cast<double2*>(rest_ptr) : nullptr;
        rest_ptr += W[g].stash_bytes;
        G.part = reinterpret_cast<double*>(rest_ptr);
        rest_ptr += W[g].part_bytes;
        const int smem = QCK_WARP_PER_CTA * ((32 << (W[g].log_r + 5)) + (int)sizeof(WarpStagedOp) * QCK_WARP_STAGE);
        warp_kernel(W[g].log_r)<<<(unsigned)W[g].ctas, 32 * QCK_WARP_PER_CTA, smem, streams[g]>>>(
            G, d_out, (long long)out_row_stride);
        QCK_CHECK_LAUNCH(h);
    }
    return QCK_OK;
}

// ---- tree-walk simulation ----------------------------------------------------------------------
typedef void (*TreeKernelFn)(const TreeDev, int, int, long long, const double2*, double2*, double*);
static TreeKernelFn tree_kernel(int log_r) {
    switch (log_r) {
        case 0: return sim_tree_level_kernel<0>;
        case 1: return sim_tree_level_kernel<1>;
        case 2: return sim_tree_level_kernel<2>;
        case 3: return sim_tree_level_kernel<3>;
        case 4: return sim_tree_level_kernel<4>;
        default: return sim_tree_level_kernel<5>;
    }
}
static int tree_smem(int log_r) {
    return QCK_WARP_PER_CTA * ((8 << (log_r + 5)) + (int)sizeof(WarpStagedOp) * QCK_WARP_STAGE + 16 * 64);
}

static int qck_tree_init(qck_handle* h) {
    for (int r = 0; r <= 5; ++r) {
        QCK_CUDA(h, cudaFuncSetAttribute(tree_kernel(r), cudaFuncAttributeMaxDynamicSharedMemorySize, tree_smem(r)));
        int occ = 0;
        QCK_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, tree_kernel(r), 32 * QCK_WARP_PER_CTA, tree_smem(r)));
        h->tree_occ[r] = occ < 1 ? 1 : occ;
    }
    return QCK_OK;
}

// nodes per level (n[l] = nodes BEFORE branching op l; n[n_levels] = leaves); false when out of range
static bool tree_counts(const qck_sim_tree_plan* p, long long* n) {
    if (!p || p->n_levels < 1 || p->n_levels > QCK_TREE_MAX_LEVELS || p->n_base < 1 || p->n_base > 10) return false;
    n[0] = 1;
    for (int l = 0; l < p->n_levels; ++l) {
        const int b = p->level[l].n_choices;
        if (b < 1 || b > QCK_TREE_MAX_CHOICES) return false;
        n[l + 1] = n[l] * b;
        if (n[l + 1] > 0x7fffffffll) return false;  // node indices are 32-bit on the device
    }
    return true;
}
static void tree_layout(const qck_sim_tree_plan* p, const long long* n, size_t* state_bytes, size_t* part_bytes) {
    long long max_inner = 0;
    for (int l = 1; l < p->n_levels; ++l)
        if (n[l] > max_inner) max_inner = n[l];
    const int nq = p->n_base > 5 ? p->n_base : 5;
    *state_bytes = (((size_t)max_inner * sizeof(double2)) << nq) + 256;
    *part_bytes = (((size_t)n[p->n_levels] * sizeof(double)) << p->n_free) + 256;
}

extern "C" size_t qck_sim_tree_work_bytes(const qck_sim_tree_plan* plan) {
    long long n[QCK_TREE_MAX_LEVELS + 1];
    if (!tree_counts(plan, n)) return 0;
    size_t sb, pb;
    tree_layout(plan, n, &sb, &pb);
    return 2 * sb + pb;
}

#define TREE_FUSE_ITEMS 300  // items of the last level fused into the first launch of qck_sim_tree

extern "C" int qck_sim_tree(qck_handle* h, const qck_sim_tree_plan* plan, int64_t label_begin, int64_t label_end,
                            double* d_out, int64_t out_row_stride, void* d_work, size_t work_bytes,
                            qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    long long n[QCK_TREE_MAX_LEVELS + 1];
    if (!tree_counts(plan, n)) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "tree plan out of range");
    if (!d_out || !plan->d_ops || !plan->d_mats || label_begin < 0 || label_end < label_begin)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "bad tree arguments");
    if (plan->n_out_bits < 0 || plan->n_out_bits > 20 || plan->n_free < 0 || plan->n_free > plan->n_out_bits ||
        plan->n_free > plan->n_base || out_row_stride < (1ll << plan->n_out_bits) || plan->n_digits > QCK_MAX_DIGITS)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "bad tree row layout");
    if (label_end == label_begin) return QCK_OK;
    size_t sb, pb;
    tree_layout(plan, n, &sb, &pb);
    if (!d_work || work_bytes < 2 * sb + pb)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "tree simulation needs %zu bytes of work space, got %zu", 2 * sb + pb, work_bytes);
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (h->region) {  // the levels are dependent launches: the whole call goes on ONE side stream of the region
        int rc = region_fork_call(h, st);
        if (rc) return rc;
        rc = pick_side_stream(h, &h->region_used, &st);
        if (rc) return rc;
    }
    std::unique_ptr<TreeDev> T(new TreeDev);
    memset(T.get(), 0, sizeof(TreeDev));
    T->n_base = plan->n_base;
    T->n_levels = plan->n_levels;
    T->n_digits = plan->n_digits;
    T->n_out_bits = plan->n_out_bits;
    T->seg0_begin = plan->seg0_begin;
    T->seg0_end = plan->seg0_end;
    T->n_free = plan->n_free;
    memcpy(T->free_bit, plan->free_bit, sizeof(T->free_bit));
    memcpy(T->free_pos, plan->free_pos, sizeof(T->free_pos));
    T->base_sum = plan->base_sum;
    T->ops = plan->d_ops;
    T->mats = plan->d_mats;
    long long div = 1, total = 1;
    for (int k = QCK_MAX_DIGITS - 1; k >= 0; --k) {
        T->radix[k] = k < plan->n_digits ? plan->radix[k] : 1;
        T->div[k] = (int)div;
        if (k < plan->n_digits) div *= plan->radix[k];
        if (div > 0x7fffffffll) QCK_FAIL(h, QCK_ERR_UNSUPPORTED, "fragment label space exceeds 2^31");
    }
    total = div;
    if (label_end > total) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "label range exceeds the %lld labels of the fragment", total);
    for (int l = 0; l < plan->n_levels; ++l) {
        T->level[l] = plan->level[l];
        const qck_tree_level& L = plan->level[l];
        if (L.qubit < 0 || L.qubit >= plan->n_base || (L.kind != QCK_TREE_MMEAS && (L.digit < 0 || L.digit >= plan->n_digits)))
            QCK_FAIL(h, QCK_ERR_INVALID_ARG, "tree level %d: bad qubit / digit", l);
    }
    // refusals of the combine: checked before anything is launched
    int n_fork_max = 0;
    long long n_rep_labels = 1, n_eq_max = 1;
    for (int l = 0; l < plan->n_levels; ++l) {
        const qck_tree_level& L = plan->level[l];
        if (L.kind == QCK_TREE_MMEAS) continue;
        n_fork_max += L.kind == QCK_TREE_SLOT;
        int reps = 0, biggest = 1;
        for (int v = 0; v < 8; ++v) {
            if (L.first_choice[v] < 0) continue;
            ++reps;
            int cls = 0;
            for (int d = 0; d < plan->radix[L.digit]; ++d) cls += (int)((L.canon >> (4 * d)) & 15u) == v;
            if (cls > biggest) biggest = cls;
        }
        n_rep_labels *= reps;
        n_eq_max *= biggest;
    }
    if (n_fork_max > 8) QCK_FAIL(h, QCK_ERR_UNSUPPORTED, "more than 8 measuring slots whose qubit lives on");
    if (n_eq_max > 256) QCK_FAIL(h, QCK_ERR_UNSUPPORTED, "more than 256 labels share one representative");
    const int log_r = plan->n_base > 5 ? plan->n_base - 5 : 0;
    double2* sbuf[2] = {reinterpret_cast<double2*>(d_work), reinterpret_cast<double2*>((char*)d_work + sb)};
    double* part = reinterpret_cast<double*>((char*)d_work + 2 * sb);
    const long long cap = (long long)h->sm_count * h->tree_occ[log_r];
    // the first levels in ONE launch (every warp replays its item's path from the root) while the last fused
    // level has at most TREE_FUSE_ITEMS items.  Measured:
    // hwe-16 d5 0.1735 -> 0.1689 ms, syc-16 d5 0.119 -> 0.113 ms per step with levels 0-2 (216 items) fused; fusing
    // on to 1 296 items (one wave of warps) gives the gain back - a level is bound by its chain of gates, not by
    // its launch, and the replay makes the chain longer.
    long long fuse_cap = TREE_FUSE_ITEMS;
    if (fuse_cap > cap * QCK_WARP_PER_CTA) fuse_cap = cap * QCK_WARP_PER_CTA;
    int fused_to = 0;
    while (fused_to + 1 < plan->n_levels && n[fused_to + 2] <= fuse_cap) ++fused_to;
    for (int l = fused_to; l < plan->n_levels; ++l) {
        const long long items = n[l + 1];
        long long ctas = (items + QCK_WARP_PER_CTA - 1) / QCK_WARP_PER_CTA;
        if (ctas > cap) ctas = cap;
        const int first = l == fused_to ? 0 : l;
        tree_kernel(log_r)<<<(unsigned)ctas, 32 * QCK_WARP_PER_CTA, tree_smem(log_r), st>>>(
            *T, first, l, items, sbuf[(l + 1) & 1], sbuf[l & 1], part);
        QCK_CHECK_LAUNCH(h);
    }
    unsigned long long cg = ((unsigned long long)n_rep_labels + QCK_TREE_COMBINE_WARPS - 1) / QCK_TREE_COMBINE_WARPS;
    if (cg > (unsigned long long)h->sm_count * 8) cg = (unsigned long long)h->sm_count * 8;
    sim_tree_combine_kernel<<<(unsigned)cg, 32 * QCK_TREE_COMBINE_WARPS, 0, st>>>(
        *T, n_rep_labels, label_begin, label_end, part, d_out, (long long)out_row_stride);
    QCK_CHECK_LAUNCH(h);
    return QCK_OK;
}

static int warp_single_plan(qck_handle* h, const qck_sim_plan* plan, const int32_t* d_labels, int64_t n_instances,
                            double* d_out, int64_t out_row_stride, cudaStream_t st) {
    const int one = 0;
    const int32_t* labs[1] = {d_labels};
    const int64_t cnt[1] = {n_instances};
    std::unique_ptr<WarpGroupHost> W(new WarpGroupHost);
    int rc = warp_group_layout(h, plan, &one, 1, labs, cnt, out_row_stride, W.get());
    if (rc) return rc;
    return warp_groups_run(h, W.get(), 1, &st, d_out, out_row_stride);
}

static int ensure_side_streams(qck_handle* h) {
    if (h->side_ready) return QCK_OK;
    for (int i = 0; i < QCK_SIDE_STREAMS; ++i) {
        QCK_CUDA(h, cudaStreamCreateWithFlags(&h->side[i], cudaStreamNonBlocking));
        QCK_CUDA(h, cudaEventCreateWithFlags(&h->side_done[i], cudaEventDisableTiming));
    }
    QCK_CUDA(h, cudaEventCreateWithFlags(&h->fork, cudaEventDisableTiming));
    h->side_ready = 1;
    return QCK_OK;
}

static int launch_group(qck_handle* h, const qck_sim_plan* plans, const int* idx, int n, const int32_t* const* d_labels,
                        const int64_t* n_instances, double* d_out, int64_t out_row_stride, cudaStream_t st,
                        char* d_work, size_t work_bytes, size_t* work_used) {
    GroupDev G;
    memset(&G, 0, sizeof(G));
    const qck_sim_plan& p0 = plans[idx[0]];
    G.n_state = p0.n_state_qubits;
    G.n_vars = n;
    G.n_digits = p0.n_digits;
    G.ops = p0.d_ops;
    G.mats = p0.d_mats;
    for (int k = 0; k < QCK_MAX_DIGITS; ++k) G.radix[k] = k < p0.n_digits ? p0.radix[k] : 1;
    long long ctas = 0;
    int max_ops = 1;
    for (int i = 0; i < n; ++i) {
        const qck_sim_plan& p = plans[idx[i]];
        if (p.d_ops != p0.d_ops || p.d_mats != p0.d_mats || p.n_digits != p0.n_digits)
            QCK_FAIL(h, QCK_ERR_INVALID_ARG, "plans of one batch must share the program blob and the label radices");
        if (out_row_stride < (1ll << p.n_out_bits))
            QCK_FAIL(h, QCK_ERR_INVALID_ARG, "out_row_stride smaller than the row (2^%d)", p.n_out_bits);
        PlanDev pd = to_dev(&p);
        PlanVarDev& v = G.var[i];
        v.op_begin = p.sweeps[0].op_begin;
        v.op_end = p.sweeps[0].op_end;
        v.init = nullptr;
        if (has_shared_prefix(&p)) {  // prefix once (same stream, so ordered before the group launch), then the rest
            const size_t need = (size_t)16 << p.n_state_qubits;
            if (!d_work || *work_used + need > work_bytes)
                QCK_FAIL(h, QCK_ERR_INVALID_ARG,
                         "plans with a shared prefix need 16 << n_state bytes of work space each (%zu of %zu used)",
                         *work_used, work_bytes);
            double2* snap = reinterpret_cast<double2*>(d_work + *work_used);
            *work_used += need;
            int rc = launch_prefix(h, &p, snap, st);
            if (rc) return rc;
            v.init = snap;
            v.op_begin = p.sweeps[1].op_begin;
            v.op_end = p.sweeps[1].op_end;
        }
        v.n_out_bits = pd.n_out_bits;
        v.out_ident = pd.out_ident;
        for (int j = 0; j < QCK_MAX_OUT_BITS; ++j) v.out_pos[j] = (signed char)pd.out_pos[j];
        v.sum_mask = pd.sum_mask;
        v.sign_mask = pd.sign_mask;
        v.labels = d_labels[idx[i]];
        v.cta_begin = (int)ctas;
        ctas += n_instances[idx[i]];
        if (v.op_end - v.op_begin > max_ops) max_ops = v.op_end - v.op_begin;
    }
    if (ctas > 0x7fffffffll) QCK_FAIL(h, QCK_ERR_UNSUPPORTED, "too many instances in one group");
    G.n_stage = stage_records(max_ops);
    const int N = G.n_state;
    size_t smem = ((size_t)16 << N) + sizeof(StagedOp) * G.n_stage;
    if ((int)smem + 2048 > h->max_smem_optin)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "on-chip plan with %d qubits does not fit shared memory", N);
    int threads = 1 << (N > 3 ? N - 3 : 0);
    if (threads < 32) threads = 32;
    if (threads > 256) threads = 256;
    sim_onchip_group_kernel<<<(unsigned)ctas, threads, smem, st>>>(G, d_out, (long long)out_row_stride);
    QCK_CHECK_LAUNCH(h);
    return QCK_OK;
}

// Region: several qck_sim_fragments_batch calls (the fragments of one cut circuit) whose launches should
// OVERLAP on the device.  Between begin and end every call puts its launches on the handle's side streams
// (rotating, so that consecutive calls land on different ones) and does not join; end joins them all into
// `stream`.  One region per handle at a time; outputs and work buffers of the calls must not alias.
extern "C" int qck_sim_region_begin(qck_handle* h, qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    if (h->region) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "qck_sim_region_begin: a region is already open on this handle");
    DeviceGuard guard(h->device);
    int rc = ensure_side_streams(h);
    if (rc) return rc;
    QCK_CUDA(h, cudaEventRecord(h->fork, (cudaStream_t)stream));
    h->region = 1;
    h->region_used = 0;
    h->region_forked = 0;
    h->region_calls = 0;
    return QCK_OK;
}

extern "C" int qck_sim_region_end(qck_handle* h, qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    if (!h->region) return QCK_OK;
    DeviceGuard guard(h->device);
    h->region = 0;
    for (int s = 0; s < QCK_SIDE_STREAMS; ++s) {
        if (!((h->region_used >> s) & 1u)) continue;
        QCK_CUDA(h, cudaEventRecord(h->side_done[s], h->side[s]));
        QCK_CUDA(h, cudaStreamWaitEvent((cudaStream_t)stream, h->side_done[s], 0));
    }
    h->region_used = 0;
    return QCK_OK;
}

// next side stream of a fan-out; *used: the side streams already ordered after the fork point
static int pick_side_stream(qck_handle* h, unsigned* used, cudaStream_t* st) {
    const int slot = (int)(h->side_next++ % QCK_SIDE_STREAMS);
    *st = h->side[slot];
    // inside a region every CALL has its own fork point (region_fork_call): what the caller enqueued on its stream
    // between region_begin and the call - the H2D copy of the program, a memset of the output - is ordered
    // before the call's launches, too
    unsigned* forked = h->region ? &h->region_forked : used;
    if (!((*forked >> slot) & 1u)) {
        QCK_CUDA(h, cudaStreamWaitEvent(*st, h->fork, 0));
        *forked |= 1u << slot;
    }
    *used |= 1u << slot;
    return QCK_OK;
}

// first thing a simulation call does inside a region: a fresh fork point on the caller's stream
static int region_fork_call(qck_handle* h, cudaStream_t main_st) {
    if (!h->region) return QCK_OK;
    QCK_CUDA(h, cudaEventRecord(h->fork, main_st));
    h->region_forked = 0;
    return QCK_OK;
}

extern "C" int qck_sim_fragments_batch(qck_handle* h, int n_plans, const qck_sim_plan* plans,
                                       const int32_t* const* d_labels, const int64_t* n_instances, double* d_out,
                                       int64_t out_row_stride, void* d_work, size_t work_bytes, qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    if (n_plans < 0 || (n_plans > 0 && (!plans || !d_labels || !n_instances || !d_out)))
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "bad plan list");
    for (int i = 0; i < n_plans; ++i) {
        int rc = validate_plan(h, &plans[i]);
        if (rc) return rc;
        if (n_instances[i] < 0 || (n_instances[i] > 0 && !d_labels[i])) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "bad instance list");
    }
    DeviceGuard guard(h->device);
    cudaStream_t main_st = (cudaStream_t)stream;
    // on-chip plans grouped by state size -> one launch per group (chunks of QCK_GROUP_MAX)
    int n_groups = 0;
    for (int N = 1; N <= QCK_MAX_TILE_QUBITS; ++N) {
        int cnt = 0;
        for (int i = 0; i < n_plans; ++i)
            if (n_instances[i] > 0 && is_onchip(&plans[i]) && plans[i].n_state_qubits == N) ++cnt;
        n_groups += (cnt + QCK_GROUP_MAX - 1) / QCK_GROUP_MAX;
    }
    int n_warp_groups = 0;
    for (int N = 1; N <= 10; ++N) {
        int cnt = 0;
        for (int i = 0; i < n_plans; ++i)
            if (n_instances[i] > 0 && is_warp_plan(&plans[i]) && warp_base(&plans[i]) == N) ++cnt;
        n_warp_groups += (cnt + QCK_GROUP_MAX - 1) / QCK_GROUP_MAX;
    }
    n_groups += n_warp_groups;
    const bool region = h->region != 0;
    const bool fan = region || n_groups >= 2;
    unsigned used_local = 0;
    unsigned* used = region ? &h->region_used : &used_local;
    size_t work_used = 0;  // snapshots of shared prefixes: disjoint slices of d_work (groups run concurrently)
    if (fan && !region) {
        int rc = ensure_side_streams(h);
        if (rc) return rc;
        QCK_CUDA(h, cudaEventRecord(h->fork, main_st));
    }
    if (region) {
        int rc = region_fork_call(h, main_st);
        if (rc) return rc;
    }
    for (int N = QCK_MAX_TILE_QUBITS; N >= 1; --N) {  // largest states first: they run longest
        int idx[QCK_GROUP_MAX], cnt = 0;
        for (int i = 0; i <= n_plans; ++i) {
            const bool take = i < n_plans && n_instances[i] > 0 && is_onchip(&plans[i]) && plans[i].n_state_qubits == N;
            if (take) idx[cnt++] = i;
            if (cnt == QCK_GROUP_MAX || (i == n_plans && cnt > 0)) {
                cudaStream_t st = main_st;
                if (fan) {
                    int rc = pick_side_stream(h, used, &st);
                    if (rc) return rc;
                }
                int rc = launch_group(h, plans, idx, cnt, d_labels, n_instances, d_out, out_row_stride, st,
                                      (char*)d_work, work_bytes, &work_used);
                if (rc) return rc;
                cnt = 0;
            }
        }
    }
    // register-resident plans: most branch points first (they run longest), one launch per QCK_GROUP_MAX plans
    if (n_warp_groups > 0) {
        std::unique_ptr<WarpGroupHost[]> W(new WarpGroupHost[n_warp_groups]);
        std::unique_ptr<cudaStream_t[]> wst(new cudaStream_t[n_warp_groups]);
        int g = 0;
        for (int N = 10; N >= 1; --N) {
            int order[1024], n_sel = 0;
            for (int a = QCK_WARP_MAX_DEPTH; a >= 0; --a)
                for (int i = 0; i < n_plans && n_sel < 1024; ++i)
                    if (n_instances[i] > 0 && is_warp_plan(&plans[i]) && warp_base(&plans[i]) == N &&
                        plans[i].n_state_qubits - N == a)
                        order[n_sel++] = i;
            for (int b = 0; b < n_sel; b += QCK_GROUP_MAX) {
                const int cnt = n_sel - b < QCK_GROUP_MAX ? n_sel - b : QCK_GROUP_MAX;
                cudaStream_t st = main_st;
                if (fan) {
                    int rc = pick_side_stream(h, used, &st);
                    if (rc) return rc;
                }
                int rc = warp_group_layout(h, plans, order + b, cnt, d_labels, n_instances, out_row_stride, &W[g]);
                if (rc) return rc;
                wst[g++] = st;
            }
        }
        int rc = warp_groups_run(h, W.get(), g, wst.get(), d_out, out_row_stride);
        if (rc) return rc;
    }
    for (int s = 0; s < QCK_SIDE_STREAMS && !region; ++s) {  // join (a region joins at its end)
        if (!((used_local >> s) & 1u)) continue;
        QCK_CUDA(h, cudaEventRecord(h->side_done[s], h->side[s]));
        QCK_CUDA(h, cudaStreamWaitEvent(main_st, h->side_done[s], 0));
    }
    // streaming plans: one after the other, sharing d_work - on the caller's stream, or inside a region on ONE
    // side stream of their own (the streaming fragments of a cut circuit then overlap each other)
    cudaStream_t stream_st = main_st;
    bool picked = false;
    for (int i = 0; i < n_plans; ++i) {
        if (n_instances[i] <= 0 || is_onchip(&plans[i]) || is_warp_plan(&plans[i])) continue;
        if (region && !picked) {
            int rc = pick_side_stream(h, used, &stream_st);
            if (rc) return rc;
            picked = true;
        }
        int rc = qck_sim_fragments(h, &plans[i], d_labels[i], n_instances[i], d_out, out_row_stride, d_work, work_bytes,
                                   (qck_stream)stream_st);
        if (rc) return rc;
    }
    return QCK_OK;
}

// Instances of a fragment whose label digits select identical variants (several instantiations of a virtual gate
// look the same from one side: virtual_gates.py:62-103 measures Z for both the I and the Z term) have identical
// rows: the caller simulates one representative per class and copies its row to the others.
__global__ void __launch_bounds__(256) rows_broadcast_kernel(double* __restrict__ table, long long row_stride,
                                                             long long row_len, const int32_t* __restrict__ src,
                                                             long long n_rows) {
    for (long long r = blockIdx.x; r < n_rows; r += gridDim.x) {
        const long long from = __ldg(src + r);
        if (from == r) continue;  // uniform per CTA
        const double* a = table + from * row_stride;
        double* b = table + r * row_stride;
        if (((row_stride | row_len) & 1) == 0 && (reinterpret_cast<uintptr_t>(table) & 15) == 0) {
            const double2* a2 = reinterpret_cast<const double2*>(a);
            double2* b2 = reinterpret_cast<double2*>(b);
            for (long long i = threadIdx.x; i < row_len / 2; i += blockDim.x) b2[i] = a2[i];
        } else {
            for (long long i = threadIdx.x; i < row_len; i += blockDim.x) b[i] = a[i];
        }
    }
}

extern "C" int qck_rows_broadcast(qck_handle* h, double* d_table, int64_t row_stride, int64_t row_len,
                                  const int32_t* d_src, int64_t n_rows, qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    if (n_rows == 0) return QCK_OK;
    if (!d_table || !d_src || n_rows < 0 || row_len < 1 || row_stride < row_len)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "bad table / source list");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    long long grid = n_rows < 16ll * h->sm_count ? n_rows : 16ll * h->sm_count;
    rows_broadcast_kernel<<<(unsigned)grid, 256, 0, st>>>(d_table, (long long)row_stride, (long long)row_len, d_src,
                                                           (long long)n_rows);
    QCK_CHECK_LAUNCH(h);
    return QCK_OK;
}

extern "C" int qck_sim_statevector(qck_handle* h, const qck_sim_plan* plan, int32_t label, void* d_state,
                                   size_t state_bytes, qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    int rc = validate_plan(h, plan);
    if (rc) return rc;
    if (is_onchip(plan) && plan->n_state_qubits > 0) {
        // an on-chip plan is also a valid one-sweep streaming plan
    }
    const unsigned long long state_amps = 1ull << plan->n_state_qubits;
    if (!d_state || state_bytes < state_amps * 16)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "state buffer too small: need %llu bytes", state_amps * 16);
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    // the label travels through a one-element device list kept in the handle scratch
    int32_t* d_label = reinterpret_cast<int32_t*>(h->d_partials + h->partials_count - 8);  // reserved tail
    QCK_CUDA(h, cudaMemcpyAsync(d_label, &label, sizeof(int32_t), cudaMemcpyHostToDevice, st));
    PlanDev pd = to_dev(plan);
    return run_sweeps(h, plan, pd, d_label, 0, 1, (double2*)d_state, state_amps, st);
}

// ------------------------------------------------------------------ sharded statevector (several GPUs)
// The state of an uncut circuit too large for one GPU: 2^n_local amplitudes per rank, the top bits of the
// amplitude index are the rank.  Every rank runs the same sweeps on the tiles it owns; a sweep whose tile
// contains rank bits loads / stores the peer halves of its tiles straight from / to the peers' buffers with
// TMA (mapped through CUDA IPC, NVLink): the exchange IS the sweep, there is no separate all-to-all.  The
// caller synchronises the ranks between sweeps (qck.h).
extern "C" int qck_sim_sweeps_sharded(qck_handle* h, const qck_sim_plan* plan, int sweep_begin, int sweep_end, int rank,
                                      int world, void* const* d_shards, size_t shard_bytes, qck_stream stream) {
    if (!h) return QCK_ERR_INVALID_ARG;
    int rc = validate_plan(h, plan);
    if (rc) return rc;
    int g = 0;
    while ((1 << g) < world) ++g;
    if (world < 1 || world > TMA_MAX_SHARDS || (1 << g) != world || rank < 0 || rank >= world || !d_shards)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "world=%d must be a power of two <= %d, 0 <= rank < world", world, TMA_MAX_SHARDS);
    const int n_local = plan->n_state_qubits - g;
    if (plan->n_digits != 0) QCK_FAIL(h, QCK_ERR_UNSUPPORTED, "sharded runs simulate one uncut circuit (no label digits)");
    if (n_local < 14 || shard_bytes < ((size_t)16 << n_local))
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "shard of 2^%d amplitudes needs %zu bytes, got %zu", n_local, (size_t)16 << n_local,
                 shard_bytes);
    if (sweep_begin < 0 || sweep_end > plan->n_sweeps || sweep_begin > sweep_end)
        QCK_FAIL(h, QCK_ERR_INVALID_ARG, "bad sweep range [%d, %d)", sweep_begin, sweep_end);
    for (int r = 0; r < world; ++r)
        if (!d_shards[r]) QCK_FAIL(h, QCK_ERR_INVALID_ARG, "shard pointer of rank %d is NULL", r);
    if (!tensor_map_encoder()) QCK_FAIL(h, QCK_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    DeviceGuard guard(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    PlanDev pd = to_dev(plan);
    int32_t* d_label = reinterpret_cast<int32_t*>(h->d_partials + h->partials_count - 8);  // reserved tail
    QCK_CUDA(h, cudaMemsetAsync(d_label, 0, sizeof(int32_t), st));
    std::unique_ptr<TmaLaunch> L(new TmaLaunch);
    TmaShard sh = {n_local, rank};
    unsigned long long live = 0;
    for (int i = 0; i < sweep_end; ++i) {
        if (i >= sweep_begin) {
            if (!tma_describe(plan, i, live, i == plan->n_sweeps - 1, 1, h->max_smem_optin, *L, &sh))
                QCK_FAIL(h, QCK_ERR_UNSUPPORTED, "sweep %d cannot run on the TMA kernel (tile layout / op count)", i);
            if (L->n_work > 0) {
                const bool box_main = L->sd.zf_shift == L->sd.lowc + L->sd.k;
                for (int r = 0; r < world; ++r) {
                    rc = tma_encode(h, L->sd, 1, (double2*)d_shards[r], true, L->maps.st_mut(r));
                    if (rc) return rc;
                    rc = tma_encode(h, L->sd, 1, (double2*)d_shards[r], box_main, L->maps.ld_mut(r));
                    if (rc) return rc;
                }
                L->maps.pr = L->maps.sh0.st;
                PlanDev pdl = pd;
                pdl.n_stage = L->n_stage;
                const unsigned long long grid =
                    L->n_work < (unsigned long long)h->sm_count ? L->n_work : (unsigned long long)h->sm_count;
                if (L->sd.n_store >= 16 || L->sd.n_load >= 16)  // measured: 8 boxes of 8 KiB are still faster from one lane
                    sim_sweep_tma_sharded_wide_kernel<<<(unsigned)grid, TMA_CONSUMERS + 32, L->smem, st>>>(
                        L->maps, L->sd, pdl, d_label, 0, L->n_work);
                else
                    sim_sweep_tma_sharded_kernel<<<(unsigned)grid, TMA_CONSUMERS + 32, L->smem, st>>>(
                        L->maps, L->sd, pdl, d_label, 0, L->n_work);
                QCK_CHECK_LAUNCH(h);
            }
        }
        for (int j = 0; j < plan->sweeps[i].n_tile; ++j) live |= 1ull << plan->sweeps[i].pos[j];
    }
    return QCK_OK;
}

// Plain device memory + CUDA IPC for the shards (torch's caching allocator sub-allocates, which IPC cannot
// export directly).
extern "C" int qck_mem_alloc(qck_handle* h, size_t bytes, void** d_ptr) {
    if (!h || !d_ptr) return QCK_ERR_INVALID_ARG;
    DeviceGuard guard(h->device);
    if (cudaMalloc(d_ptr, bytes) != cudaSuccess) {
        cudaGetLastError();
        QCK_FAIL(h, QCK_ERR_NOMEM, "cudaMalloc of %zu bytes failed", bytes);
    }
    return QCK_OK;
}
extern "C" int qck_mem_free(qck_handle* h, void* d_ptr) {
    if (!h) return QCK_ERR_INVALID_ARG;
    DeviceGuard guard(h->device);
    QCK_CUDA(h, cudaFree(d_ptr));
    return QCK_OK;
}
extern "C" int qck_ipc_export(qck_handle* h, void* d_ptr, unsigned char* handle64) {
    if (!h || !d_ptr || !handle64) return QCK_ERR_INVALID_ARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    DeviceGuard guard(h->device);
    cudaIpcMemHandle_t ih;
    QCK_CUDA(h, cudaIpcGetMemHandle(&ih, d_ptr));
    memcpy(handle64, &ih, 64);
    return QCK_OK;
}
extern "C" int qck_ipc_open(qck_handle* h, const unsigned char* handle64, void** d_ptr) {
    if (!h || !handle64 || !d_ptr) return QCK_ERR_INVALID_ARG;
    DeviceGuard guard(h->device);
    cudaIpcMemHandle_t ih;
    memcpy(&ih, handle64, 64);
    QCK_CUDA(h, cudaIpcOpenMemHandle(d_ptr, ih, cudaIpcMemLazyEnablePeerAccess));
    return QCK_OK;
}
extern "C" int qck_ipc_close(qck_handle* h, void* d_ptr) {
    if (!h) return QCK_ERR_INVALID_ARG;
    DeviceGuard guard(h->device);
    QCK_CUDA(h, cudaIpcCloseMemHandle(d_ptr));
    return QCK_OK;
}

/*
 * qck.h - C ABI of libqck.so: B200 (sm_100a) fragment simulation + knitting.
 *
 * Drop-in boundary for the hot path of
 * thangktran/HardwareAwareOptimalQuantumCircuitCuttingAndKnitting, i.e. what
 * third_party/qvm/qvm/run.py:23-71 (run_virtual_circuit) delegates to a Qiskit
 * backend and a multiprocessing.Pool today.  The reference is pure Python, so
 * the binding a maintainer adds is a ctypes stub (see INTEGRATION.md); every
 * entry point below names the reference call site it replaces.
 *
 * Conventions
 *   - plain C, no exceptions, every function returns a qck_status (0 = ok);
 *     qck_last_error_string(h) gives the detail for the last failure on h.
 *   - pointers named d_* are DEVICE pointers owned by the caller (torch on the
 *     Python side); the library allocates only small scratch inside the handle.
 *   - `stream` is a cudaStream_t passed as void* (0 = default stream); all work
 *     is enqueued asynchronously on it; nothing synchronises unless documented.
 *   - one handle per host thread (the reference calls run_virtual_circuit from
 *     several Python threads at once, src/HwAwareCutter/Utilities.py:85-101);
 *     handles share no mutable state.
 *   - bitstring convention: bit i of an output index = classical bit i of the
 *     cut circuit (quasi_distr.py:13-20).  Statevector index bit q = local
 *     qubit q of the fragment (little endian, as Qiskit).
 */
#ifndef QCK_H
#define QCK_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QCK_ABI_VERSION 1

#if defined(__GNUC__)
#define QCK_API __attribute__((visibility("default")))
#else
#define QCK_API
#endif

typedef enum {
    QCK_OK = 0,
    QCK_ERR_INVALID_ARG = 1,   /* -> ValueError on the Python side   */
    QCK_ERR_CUDA = 2,          /* -> RuntimeError                    */
    QCK_ERR_UNSUPPORTED = 3,   /* -> NotImplementedError             */
    QCK_ERR_NOMEM = 4          /* -> MemoryError                     */
} qck_status;

typedef struct qck_handle qck_handle;
typedef void* qck_stream;

QCK_API int qck_abi_version(void);
QCK_API int qck_create(int device, qck_handle** out);
QCK_API int qck_destroy(qck_handle* h);
QCK_API const char* qck_last_error_string(const qck_handle* h);
QCK_API const char* qck_status_string(int status);
/* number of kernels this handle has launched so far (bench.py's gpu_launches) */
QCK_API int64_t qck_launch_count(const qck_handle* h);

/* ------------------------------------------------------------------ fragment simulation
 * Replaces: virt.get_backend(frag).run(instantiations, shots) + get_counts()
 *           (run.py:36-58) together with generate_instantiations /
 *           _instantiate_fragment (virtual_circuit.py:183-213) and
 *           VirtualGateEndpoint.instantiate (virtual_gates.py:134-150):
 * instances are never materialised on the host; each CTA decodes its
 * mixed-radix label and picks the variant matrices itself.
 */
#define QCK_MAX_TILE_QUBITS 14
#define QCK_MAX_DIGITS 16
#define QCK_MAX_OUT_BITS 40

enum {
    QCK_OP_U1 = 0, QCK_OP_CX = 1, QCK_OP_CZ = 2, QCK_OP_U2 = 3, QCK_OP_CLUSTER = 4,
    QCK_OP_U1X = 5, QCK_OP_TERM = 6, QCK_OP_PHASE = 7
};
#define QCK_CLUSTER_QUBITS 3

/* One gate application.  Qubits are TILE-LOCAL bit positions of the sweep the op
 * belongs to.  A measurement whose qubit lives on is a QCK_OP_CX onto a fresh
 * ancilla bit (deferred measurement: the two halves of the state are the two
 * un-normalised branches of SURVEY.md A.2).
 * QCK_OP_CLUSTER is a header: the next q0 ops act only on the QCK_CLUSTER_QUBITS
 * tile positions (mat, sel_digit, sel_stride) = ascending positions p0 < p1 < p2 and
 * address them by their rank 0..2; each thread applies the whole cluster to its 8
 * amplitudes in registers (one shared-memory round trip for several gates).
 *
 * Tile-resolved ops (streaming sweeps only).  A qubit an op is block diagonal in (the control of a
 * cx, both qubits of cz / cp / rzz, the qubit of rz / z / p) need not be in the tile of the sweep: its bit
 * is a constant of the tile and only selects a variant.
 *   QCK_OP_U1X  header: a one-qubit op on tile qubit q0 whose matrix is the ordered product of the
 *               q1 following QCK_OP_TERM records; term j contributes mats[mat + 8 * bit(e0)]
 *               (two 2x2 matrices), e0 = its q0 = a STATE bit position outside the tile.
 *   QCK_OP_PHASE header: a scalar for the whole tile, the product over the q1 following terms of
 *               mats[mat + 2 * (bit(q0) + 2 * bit(q1))] (q1 = -1: one qubit, two scalars).
 *   QCK_OP_TERM sel_stride = number of complex values the record owns (8, 2 or 4).
 * The device resolves them once per tile (sim.cu: resolve_tile). */
typedef struct {
    int32_t kind;        /* QCK_OP_*                                                     */
    int32_t q0, q1;      /* U1: q0.  CX: control q0, target q1.  CZ/U2: q0 (bit0), q1     */
    int32_t mat;         /* offset (in doubles) into the matrix pool; U1: 8, U2: 32       */
    int32_t sel_digit;   /* -1, or the label digit that selects the variant matrix:       */
    int32_t sel_stride;  /*   offset = mat + digit[sel_digit] * sel_stride                */
    int32_t n_live;      /* ops touch only the first 2^n_live amplitudes of the tile      */
    int32_t reserved;    /* 1 when q0/q1 are not tile positions (cluster members: ranks;   */
                         /* TERM / PHASE records: state positions), else 0                */
} qck_op;

/* A sweep = one pass over the state: every CTA stages a 2^n_tile tile (the
 * amplitudes that differ only in the listed bit positions) in shared memory,
 * applies ops[op_begin, op_end) there and writes it back. */
#define QCK_SWEEP_SHARED 4
/* QCK_SWEEP_WARP (bit 3): register-resident plan - ONE sweep whose tile is the n_base = (flags >> 8) & 0xff
 * qubits of the fragment itself (n_base <= 10), ops restricted to QCK_OP_U1 / CX / CZ on state bit positions.
 * One warp simulates one instance with the 2^n_base amplitudes in its registers; a QCK_OP_CX onto a state bit
 * >= n_base is a mid-circuit measurement of q0 whose qubit lives on: the warp walks both outcomes depth first
 * (n_state_qubits - n_base <= 8 of them) instead of widening the state.  out_pos / sum_mask / sign_mask address
 * those outcome bits exactly as they address ancilla bits in the other regimes. */
#define QCK_SWEEP_WARP 8
typedef struct {
    int32_t n_tile;
    int32_t op_begin, op_end;
    int32_t flags;                         /* bit 0: the op range holds QCK_OP_U1X / QCK_OP_PHASE;   */
                                           /* bit 1: it holds QCK_OP_CLUSTER (-> plain sweep kernel) */
                                           /* bit 2 (QCK_SWEEP_SHARED): no op of the range selects by */
                                           /* label digit - on-chip plans only, first of two sweeps:  */
                                           /* run once per plan, every instance starts from its state */
    int32_t pos[QCK_MAX_TILE_QUBITS + 2];  /* ascending state-bit positions of the tile bits */
} qck_sweep;

/* Program of one (fragment, measurement pattern): all instances that share it
 * differ only in the matrices the label digits select. */
typedef struct {
    int32_t n_state_qubits;          /* fragment qubits + branch ancillas                 */
    int32_t n_sweeps;                /* 1 and n_tile == n_state_qubits: on-chip regime     */
    const qck_sweep* sweeps;         /* HOST array                                        */
    const qck_op* d_ops;             /* device                                            */
    const double* d_mats;            /* device, interleaved re/im                         */
    int32_t n_digits;                /* digits of a fragment label, last fastest          */
    int32_t radix[QCK_MAX_DIGITS];
    /* output row: bit j of the row index <- state bit out_pos[j] (-1: the bit is
     * never set, entries with it set are 0).  Bits in sum_mask are summed out,
     * those also in sign_mask with weight (-1)^bit (signed fold of the config
     * bits, SURVEY.md A.3). */
    int32_t n_out_bits;
    int32_t out_pos[QCK_MAX_OUT_BITS];
    uint64_t sum_mask;
    uint64_t sign_mask;
} qck_sim_plan;

/* d_labels[i] = fragment-label index of instance i (row-major over the touched
 * virtual gates, last fastest: virtual_circuit.py:39-48); its row is written at
 * d_out + d_labels[i] * out_row_stride.  d_work: scratch for the streaming
 * regime (>= 16 << n_state_qubits bytes, more = more instances in flight);
 * in the on-chip regime only plans with a QCK_SWEEP_SHARED prefix use it
 * (16 << n_state_qubits bytes per such plan: the state after the prefix). */
QCK_API int qck_sim_fragments(qck_handle* h, const qck_sim_plan* plan, const int32_t* d_labels,
                      int64_t n_instances, double* d_out, int64_t out_row_stride,
                      void* d_work, size_t work_bytes, qck_stream stream);

/* d_table[r][0..row_len) = d_table[d_src[r]][0..row_len) for every row r with d_src[r] != r (sources are rows
 * with d_src[s] == s).  Several instantiations of a virtual gate look the same from one side of the cut
 * (virtual_gates.py:62-103: the I and the Z term both measure Z), so instances whose label digits select
 * identical variants have identical rows: one representative per class is simulated
 * (virtual_circuit.py:39-48 still enumerates all of them) and its row is copied to the others. */
QCK_API int qck_rows_broadcast(qck_handle* h, double* d_table, int64_t row_stride, int64_t row_len,
                               const int32_t* d_src, int64_t n_rows, qck_stream stream);

/* Several programs of one fragment in one call (one per measurement pattern).  On-chip
 * programs are independent small launches: they are fanned out over internal side streams
 * (forked from and joined back into `stream` with events) so that they overlap on the GPU;
 * streaming programs run one after the other on `stream`, sharing d_work. */
QCK_API int qck_sim_fragments_batch(qck_handle* h, int n_plans, const qck_sim_plan* plans,
                                    const int32_t* const* d_labels, const int64_t* n_instances,
                                    double* d_out, int64_t out_row_stride, void* d_work, size_t work_bytes,
                                    qck_stream stream);

/* Overlap the qck_sim_fragments_batch calls of several fragments (their instances are independent:
 * run.py:36-43 submits one job per fragment).  Between begin and end every batch call launches on the handle's
 * side streams and returns without joining; end makes `stream` wait for all of them.  The launches of a call
 * are ordered after everything enqueued on `stream` before THAT call (each call forks anew: a program uploaded
 * or an output zero-filled between begin and the call is seen).  d_out and d_work of the calls inside one
 * region must not alias.  One region per handle at a time. */
QCK_API int qck_sim_region_begin(qck_handle* h, qck_stream stream);
QCK_API int qck_sim_region_end(qck_handle* h, qck_stream stream);

/* ------------------------------------------------------------------ tree-walk simulation (SURVEY.md 8f-4)
 * ALL instances of a fragment of <= 10 qubits (ops: QCK_OP_U1 / CX / CZ) in one call, every shared prefix
 * simulated once.  The program is cut at its BRANCHING OPS - virtual-gate endpoints ("slots",
 * virtual_gates.py:127-150) and mid-circuit measurements of the input circuit - into label-independent
 * segments; level l of the tree = the l-th branching op, a choice = (representative variant of the slot's
 * gate, outcome of its measurement if that variant measures and the qubit lives on).  One launch per level
 * (one warp per parent node x choice, state in registers, states of a level in d_work), then one launch that
 * writes the row of EVERY label in [label_begin, label_end): the sum, in a fixed order, of the partial rows of
 * its outcome leaves (labels whose variants are identical to a representative's read the same leaves).
 * Rows are the signed-folded rows of qck_sim_fragments (config bits folded with (-1)^bit). */
#define QCK_TREE_MAX_LEVELS 24
#define QCK_TREE_MAX_CHOICES 16
enum { QCK_TREE_SLOT = 0,       /* slot whose qubit lives on: a measuring variant forks into two outcomes   */
       QCK_TREE_TERMINAL = 1,   /* slot on a wire that ends there: a measuring variant signs the qubit's bit */
       QCK_TREE_MMEAS = 2 };    /* mid-circuit measurement of the input circuit: the outcome is row bit col_bit */
typedef struct {
    int32_t seg_begin, seg_end;   /* ops AFTER this branching op, up to the next one (indices into d_ops)   */
    int32_t kind, qubit, digit;   /* digit: label digit of the slot's gate (-1: QCK_TREE_MMEAS)              */
    int32_t pre_off, post_off;    /* variant matrices in d_mats (doubles, 8 per variant), -1: all identity   */
    int32_t n_choices, col_bit;
    uint32_t meas_mask;           /* bit v: variant v measures                                               */
    uint32_t canon;               /* 4 bits per variant: its representative (identical pre / meas / post)    */
    uint8_t choice_variant[QCK_TREE_MAX_CHOICES];
    int8_t choice_outcome[QCK_TREE_MAX_CHOICES];   /* -1: no projection; a fork lists outcome 0 then 1       */
    int8_t first_choice[8];                        /* per representative variant: its first choice           */
} qck_tree_level;
typedef struct {
    int32_t n_base, n_levels, n_digits, n_out_bits;
    int32_t seg0_begin, seg0_end; /* ops before the first branching op                                       */
    int32_t n_free;               /* row bits that are fragment qubits: row bit free_bit[r] <- state bit free_pos[r] */
    int8_t free_bit[16], free_pos[16];
    uint64_t base_sum;            /* fragment qubits summed out                                              */
    const qck_op* d_ops;          /* device: ops on STATE bit positions, no label-selected matrices          */
    const double* d_mats;         /* device                                                                  */
    int32_t radix[QCK_MAX_DIGITS];
    qck_tree_level level[QCK_TREE_MAX_LEVELS];
} qck_sim_tree_plan;
QCK_API size_t qck_sim_tree_work_bytes(const qck_sim_tree_plan* plan);
QCK_API int qck_sim_tree(qck_handle* h, const qck_sim_tree_plan* plan, int64_t label_begin, int64_t label_end,
                         double* d_out, int64_t out_row_stride, void* d_work, size_t work_bytes, qck_stream stream);

/* Final statevector of ONE instance in the streaming regime left in d_work
 * (used for the uncut reference run, Utilities.py:39-69). */
QCK_API int qck_sim_statevector(qck_handle* h, const qck_sim_plan* plan, int32_t label,
                        void* d_state, size_t state_bytes, qck_stream stream);

/* Host half of the program compiler (no CUDA call, re-entrant): list-schedules the ops of ONE
 * on-chip sweep (records on tile-local qubits) into register clusters - a QCK_OP_CLUSTER header
 * followed by its members, their qubits renamed to ranks; lone two-qubit ops and ops on fewer than
 * QCK_CLUSTER_QUBITS live bits stay plain.  `out` needs room for 2 * n_ops records.  (compiler.py
 * did this in Python: 64 plans per hwe-16 d5 run made it the largest part of the cold e2e time.) */
QCK_API int qck_host_cluster_ops(const int32_t* ops, int n_ops, int n_tile, int max_cluster_ops,
                                 int32_t* out, int* n_out);

/* Host half of the program compiler, first stage (no CUDA call, re-entrant): a flattened fragment circuit ->
 * the op list the device programs are made of.  Replaces what the reference does per INSTANCE with Qiskit
 * objects (virtual_circuit.py:183-213: copy, splice `instantiate(label[k])`, `.decompose()`): the fragment is
 * lowered once, virtual-gate endpoints become slots whose variant matrices a label digit selects.
 *   instr     [n_instr][6] int32: kind (1 one-qubit gate, 2 two-qubit gate with a matrix, 3 cx, 4 cz, 5 measure,
 *             6 virtual-gate endpoint), qubit 0, qubit 1, clbit, matrix offset (doubles into `pool`), endpoint row;
 *             qubits are indices into the fragment's register, barriers are already dropped
 *   endpoints [n_endpoints][6] int32: virtual-gate index, side, variants, bit mask of the variants that measure,
 *             offsets of the variants' pre- and post-measurement 2x2 matrices (8 doubles each, variant-major)
 *   flags     bit 0: register-resident (warp) programs wanted, bit 1: pair fusion
 * Products of consecutive one-qubit gates, pair fusion (cost model of compiler.py) and the qubit order (finally
 * measured qubits first, by clbit) are done here.  Returns -1 when two terminal measurements write one clbit.
 * The result is read back with qck_host_program_get (sizes first, with buf == NULL; see host_program.cu for the
 * list of items) and released with qck_host_program_free. */
typedef struct qck_host_program qck_host_program;
QCK_API int qck_host_lower(const int32_t* instr, int n_instr, const int32_t* endpoints, int n_endpoints,
                           const double* pool, int64_t pool_len, int n_qubits, int n_clbits, int flags,
                           int warp_max_qubits, int warp_max_depth, qck_host_program** out);
/* Second stage, on the lowered program: planning knobs (compiler.py's constructor arguments and module constants:
 * share_prefix / dedupe 0 off, 1 on, 2 auto), then one of: stage 0 the tree program (returns 1 when the fragment
 * is eligible - register regime, every virtual gate with one endpoint here - else 0), 1 the per-pattern plans
 * (sweep scheduling for streaming states, register clusters for on-chip ones), 2 their host image (the blob the
 * executor uploads + filled qck_sim_plan structs), 3 the canonical label of every label (identical instances).
 * Errors: QCK_ERR_UNSUPPORTED (state > 40 bits, an op that fits no tile, ...), -2 (a clbit written twice). */
QCK_API int qck_host_program_configure(qck_host_program* p, int onchip_max, int stream_tile, int cluster,
                                       int share_prefix, int tree, int dedupe, uint64_t early_bits);
QCK_API int qck_host_program_build(qck_host_program* p, int stage, int fold);
QCK_API void qck_host_program_free(qck_host_program* p);
QCK_API int64_t qck_host_program_get(const qck_host_program* p, int what, void* buf, int64_t cap_bytes);

/* Host-logic probe (no CUDA call, usable without a GPU; not re-entrant): how the TMA sweep kernel
 * would run sweep `sweep` of `plan` when the state bits in `live_before` are live (some earlier
 * sweep had them in its tile; all other qubits are still |0>).  Returns 1 and fills the arrays when
 * the sweep is eligible for the TMA path, else 0.
 *   geom[8]  = { low-run length, main-run start, main-run length, load boxes per tile, store boxes
 *                per tile, log2(amplitudes per load box), mask of load-box index bits that are
 *                zero-filled instead of loaded, number of state bits the tile number is spread over }
 *   perm[16] : ascending tile-local bit -> bit of the shared-memory layout [low | main | scattered]
 *   ld_off / st_off [<= 128]: amplitude offset of each load / store box inside the state,
 *   ld_slot / st_slot: first shared-memory amplitude slot of the box; enum_mask: the state bits a
 *   tile number is spread over; n_work = batch << popcount(enum_mask) tiles are visited. */
QCK_API int qck_debug_tma_describe(const qck_sim_plan* plan, int sweep, uint64_t live_before, int last,
                                   int batch, int n_local, int rank, int32_t* geom, int32_t* perm,
                                   uint64_t* ld_off, uint32_t* ld_slot, uint64_t* st_off,
                                   uint32_t* st_slot, uint64_t* enum_mask, uint64_t* n_work,
                                   uint64_t* fixed_base);
/*   n_local > 0: sharded run (qck_sim_sweeps_sharded) - the state bits >= n_local are the rank that
 *   holds an amplitude; `rank` is the describing rank; *fixed_base = the bits every tile base of that
 *   rank carries (its own rank bits outside the tile, owner bits for rank bits inside it). */

/* ------------------------------------------------------------------ sharded statevector
 * Replaces: the ideal UNCUT run (Utilities.py:39-69) when the state does not fit one GPU: 2^n_local
 * amplitudes per rank (n_local = n_state_qubits - log2(world)), the top bits of the amplitude index
 * are the rank.  qck_sim_sweeps_sharded enqueues sweeps [sweep_begin, sweep_end) of `plan` for THIS
 * rank (one instance, no label digits; the TMA sweep kernel with live-qubit tracking).  d_shards
 * (HOST array of `world` device pointers valid on this device: the own buffer and the peers' buffers
 * mapped with qck_ipc_open) - a sweep whose tile holds rank bits moves the peer halves of its tiles
 * over NVLink with TMA, there is no separate exchange.  The caller must order the ranks: all ranks
 * finish sweep s (e.g. a stream-ordered NCCL all-reduce of one element) before any rank starts
 * sweep s + 1 whenever sweep s or s + 1 has a tile position >= n_local.
 * qck_mem_alloc / qck_ipc_*: plain cudaMalloc memory and CUDA IPC handles (64 bytes) for the shards. */
QCK_API int qck_sim_sweeps_sharded(qck_handle* h, const qck_sim_plan* plan, int sweep_begin, int sweep_end,
                                   int rank, int world, void* const* d_shards, size_t shard_bytes,
                                   qck_stream stream);
QCK_API int qck_mem_alloc(qck_handle* h, size_t bytes, void** d_ptr);
QCK_API int qck_mem_free(qck_handle* h, void* d_ptr);
QCK_API int qck_ipc_export(qck_handle* h, void* d_ptr, unsigned char* handle64);
QCK_API int qck_ipc_open(qck_handle* h, const unsigned char* handle64, void** d_ptr);
QCK_API int qck_ipc_close(qck_handle* h, void* d_ptr);

/* Exact HBM bytes the sweeps of a streaming plan move for `batch` instances (host arithmetic, no
 * CUDA call): the TMA path with live-qubit tracking when every sweep is eligible (*uses_tma = 1),
 * else one read + one write of the whole state per sweep.  fold_fused != 0: the last sweep stores
 * probabilities instead of amplitudes (what qck_sim_fragments does when the output row is the
 * whole register of a single instance).  bench.py's roofline figures use it. */
QCK_API int qck_sim_plan_traffic(const qck_sim_plan* plan, int batch, int fold_fused, uint64_t* bytes_loaded,
                                 uint64_t* bytes_stored, int* uses_tma);

/* ------------------------------------------------------------------ knitting
 * Replaces: VirtualCircuit.knit (virtual_circuit.py:50-68), _merge /
 *           _merge_distrs / QuasiDistr.merge (virtual_circuit.py:150-171,216-228;
 *           quasi_distr.py:55-60) and Virtual*.knit (virtual_gates.py:105-124,
 *           179-194,262-286) in their exact (unpruned) closed form.
 */
#define QCK_MAX_FRAGMENTS 8
#define QCK_MAX_VARIANTS 8

/* running statistics of a produced distribution (all doubles, device memory) */
typedef struct {
    double sum;      /* sum of entries                                   */
    double min;      /* smallest entry                                   */
    double sum_sqrt; /* sum of sqrt(max(entry, 0))                       */
    double nnz;      /* number of entries != 0                           */
} qck_stats;

/* K = 0: out[y - y_begin] = prod_f tables[f][pext(y, masks[f])], y in [y_begin, y_end).
 * d_tables / masks are HOST arrays of n_frag device pointers / bit masks (masks may overlap;
 * every mask bit < n_out_bits).  d_out may be NULL: statistics only -
 * called with the square-rooted tables of the cut fragments AND of a factorised
 * reference distribution this yields the Bhattacharyya sum of the Hellinger
 * fidelity without materialising anything.  d_stats may be NULL. */
QCK_API int qck_knit_outer(qck_handle* h, int n_frag, const double* const* d_tables, const uint64_t* masks,
                   int n_out_bits, uint64_t y_begin, uint64_t y_end, double* d_out,
                   qck_stats* d_stats, qck_stream stream);
/* The same call on a result SHARDED over `world` ranks by output index: the statistics of the slices are combined
 * across the ranks in the kernel's own tail (the last CTA to finish writes them into the peers' mailboxes, see
 * qck_stats_exchange) - no further launch, no collective.  d_mailboxes as for qck_stats_exchange; every rank
 * calls it with a non-empty slice.  world == 1: plain qck_knit_outer. */
QCK_API int qck_knit_outer_exchange(qck_handle* h, int n_frag, const double* const* d_tables, const uint64_t* masks,
                                    int n_out_bits, uint64_t y_begin, uint64_t y_end, double* d_out,
                                    qck_stats* d_stats, int rank, int world, void* const* d_mailboxes,
                                    qck_stream stream);

/* K >= 1: out[y] (+)= sum_{l in [l_begin, l_end)} w(l) prod_f Q_f[lf(l)][pext(y, masks[f])]
 * with l the global label (last virtual gate fastest), w(l) = prod_k coef[k][l_k],
 * lf(l) = sum_k l_k * frag_stride[f][k] (0 when gate k does not touch f).
 * coef: HOST array, n_digits rows of QCK_MAX_VARIANTS doubles.
 * frag_stride: HOST array [n_frag][QCK_MAX_DIGITS]. */
QCK_API int qck_knit_contract(qck_handle* h, int n_frag, const double* const* d_tables, const uint64_t* masks,
                      const int64_t* row_strides, int n_out_bits,
                      int n_digits, const int32_t* radix, const double* coef,
                      const int32_t* frag_stride, int64_t l_begin, int64_t l_end,
                      double* d_out, int accumulate, qck_stream stream);

/* Reference-faithful knit: the same result as VirtualCircuit.knit with
 * QuasiDistr.ACCURACY = accuracy (quasi_distr.py:3,7-10), i.e. |v| <= accuracy is dropped after
 * from_counts, after every merge fold, every split half and every + / - / scalar * of the per-gate
 * formulas, evaluated in the reference's order (virtual_circuit.py:59-68,216-228;
 * virtual_gates.py:105-124,179-194,262-286).  Tables are UNFOLDED fragment tables: row = fragment
 * label, column = pext(key, mask_f) | (config bits of f's gates, in digit order) << popcount(mask_f).
 * gates: HOST array; frag_stride / cfg_bit: HOST [n_frag][QCK_MAX_DIGITS]; measures: HOST
 * [n_frag][QCK_MAX_DIGITS][QCK_MAX_VARIANTS] (does f's instance measure gate k under variant v). */
typedef struct {
    int32_t n_variants;
    int32_t form;         /* 0: 0.5 * signed chain of (r_i0 - r_i1) (move, cz, cx, cy); 1: rzz / cp form */
    int32_t degenerate;   /* form 1: 0 = six variants, 1 = |cos| < 1e-5 (r * sin^2), 2 = |sin| < 1e-5 */
    int32_t reserved;
    double sign[QCK_MAX_VARIANTS];                          /* form 0: +1 / -1 per variant */
    double cos_half, sin_half, cos_half_sq, sin_half_sq;    /* form 1: of m_theta / 2 */
} qck_faithful_gate;

QCK_API int qck_knit_faithful(qck_handle* h, int n_frag, const double* const* d_tables, const uint64_t* masks,
                              const int64_t* row_strides, int n_out_bits, int n_gates,
                              const qck_faithful_gate* gates, const int32_t* frag_stride, const int32_t* cfg_bit,
                              const uint8_t* measures, double accuracy, double* d_out, qck_stream stream);
/* The same evaluation restricted to part `part` of `n_parts` of the output entries (every entry is an independent
 * expression tree): the entries of the other parts are written as +0, so the parts of the ranks ADD up to the full
 * vector (one all-reduce).  With accuracy > 0 the parts split the list of alive entries (entries none of whose
 * fragment columns is pruned away entirely), else the index range. */
QCK_API int qck_knit_faithful_part(qck_handle* h, int n_frag, const double* const* d_tables, const uint64_t* masks,
                                   const int64_t* row_strides, int n_out_bits, int n_gates,
                                   const qck_faithful_gate* gates, const int32_t* frag_stride, const int32_t* cfg_bit,
                                   const uint8_t* measures, double accuracy, double* d_out, int part, int n_parts,
                                   qck_stream stream);

/* ------------------------------------------------------------------ observables from the fragment tables
 * Expectation values, bitstring probabilities and marginals of the knitted (exact, unpruned) quasi-distribution
 * without the dense 2^n_out vector (observables.py).  The knit is linear in every fragment table and the output
 * masks are disjoint, so each quantity factorises over the fragments.  Fixed summation orders: deterministic.
 * No host synchronisation; capturable in a CUDA graph once the handle's scratch holds what the call needs (an
 * eager call of the same shape first).
 *
 * qck_rows_wht: out[r][s] = sum_x in[r][x] * (-1)^popcount(x & s) over 2^m_bits columns, for every row (out of
 *   place; the unnormalised Walsh-Hadamard transform).  Then <Z_S> = sum_l w(l) prod_f W_f[lf(l)][pext(S, mask_f)].
 * qck_rows_marginal: out[r][c] = sum_{x : pext(x, keep_mask) = c} in[r][x]; d_out is dense,
 *   [n_rows][2^popcount(keep_mask)].
 * qck_knit_terms: out[p] = sum_l w(l) prod_f T_f[lf(l)][cols[f][p]] over ALL global labels, w / lf / radix / coef /
 *   frag_stride as for qck_knit_contract (n_digits = 0: one label of weight 1).  d_cols: DEVICE array
 *   [n_frag][n_terms] of column indices (int64).  On Walsh-Hadamard rows it gives expectation values, on the
 *   fragment tables themselves entries of the knitted distribution. */
QCK_API int qck_rows_wht(qck_handle* h, const double* d_in, int64_t n_rows, int64_t row_stride, int m_bits,
                         double* d_out, int64_t out_row_stride, qck_stream stream);
QCK_API int qck_rows_marginal(qck_handle* h, const double* d_in, int64_t n_rows, int64_t row_stride, int m_bits,
                              uint64_t keep_mask, double* d_out, qck_stream stream);
QCK_API int qck_knit_terms(qck_handle* h, int n_frag, const double* const* d_tables, const int64_t* row_strides,
                           int n_digits, const int32_t* radix, const double* coef, const int32_t* frag_stride,
                           int64_t n_terms, const int64_t* d_cols, double* d_out, qck_stream stream);

/* ------------------------------------------------------------------ finite-shot sampling
 * Replaces: backend.run(instantiations, shots) on AerSimulator + QuasiDistr.from_counts (run.py:42,
 * quasi_distr.py:13-20): every instance is sampled `shots` times instead of returning its exact distribution.
 *
 * qck_rows_sample draws, for every row r of an UNFOLDED fragment table (simulate_fragments(fold=False): a row is an
 * instance's joint distribution over its written clbits and config bits, the config bits the top fold_bits column
 * bits), a multinomial of `shots` over its 2^m_bits columns.  Definition (tests/sampling_reference.py restates it):
 *   - sum tree: s_0[x] = v[x], s_{j+1}[i] = s_j[2i] + s_j[2i+1] (doubles, exactly this pairing);
 *   - the root s_m[0] gets `shots`; node (j, i), j >= 1, with count c > 0 gives its left child B(c, p),
 *     p = s_{j-1}[2i] / s_j[i], and its right child the rest; when c = 0, p = 0 or p = 1 there is no draw and no
 *     random number is consumed.  The leaves' counts are the sample;
 *   - B(c, p): ATen's sample_binomial - inversion when c * min(p, 1 - p) < 10, else BTRS (Hormann 1993); for
 *     p > 1/2 it draws c - B(c, 1 - p) with 1 - p rounded to double;
 *   - random numbers: Philox4x32-10, key = (seed mod 2^32, seed >> 32), counter of the t-th Philox call of node
 *     (j, i) of row r = (i mod 2^32, (i >> 32) | j << 16, row_label_begin + r, stream_id << 20 | t).  Call t gives
 *     two uniforms, from (w0, w1) then (w2, w3): x = w_lo | w_hi << 32, u = ((x >> 11) | 1) * 2^-53, which lies in
 *     [2^-53, 1 - 2^-53].  So the counts depend on (seed, stream id, row label, row values) only: not on how rows
 *     are split over calls, ranks or CTAs.  Copies of one instance are separate rows and draw independently.
 * Outputs (either or both):
 *   d_out [n_rows][out_row_stride]: fold_bits = 0: count[x] / shots; fold_bits = f: the signed fold
 *     (sum_c (-1)^popcount(c) count[x | c << (m - f)]) / shots over 2^(m - f) columns, summed in integers - equal,
 *     bit for bit, to folding the counts of the unfolded output.  Padding past the row is not touched.
 *   d_shot_list [n_rows][shots]: the drawn column indices in ascending order (for single wide rows).
 * Entries must be finite and >= 0 and a row total > 0: otherwise bit 0 (an entry) / bit 1 (a total) is OR-ed into
 * *d_status (device); a row whose total is not > 0 gets no shots.  1 <= shots < 2^31, stream_id < 2^12, labels < 2^32.  Rows of
 * <= 2^13 columns: one CTA per row; wider ones: one pass writes the 2^12-column tile sums into the handle's scratch,
 * the descent reads only the tiles that received shots again.  No host synchronisation; capturable once the
 * handle's scratch is sized. */
QCK_API int qck_rows_sample(qck_handle* h, const double* d_in, int64_t n_rows, int64_t row_stride, int m_bits,
                            int64_t shots, uint64_t seed, uint32_t stream_id, int64_t row_label_begin,
                            double* d_out, int64_t out_row_stride, int fold_bits, int64_t* d_shot_list,
                            uint64_t* d_status, qck_stream stream);

/* ------------------------------------------------------------------ density-matrix simulation under noise
 * Replaces: backend.run(instantiations, shots) on a noisy Aer backend (run.py:42) by the exact noisy outcome
 * distribution of every instance (density.py lowers a fragment and a noise model into this plan).
 *
 * rho: 2^(2n) complex128, index r | c << n for rho[r][c].  Op record (int32[12]): {nq, mat_off, sel_digit, branch_bit,
 * p0, p1, p2, p3, s0, s1, s2, s3}: a superoperator (4x4 when nq = 1 on tile positions (p0, p1) = (row bit, column
 * bit); 16x16 when nq = 2 on (p0, p1, p2, p3) = (r0, r1, c0, c1)), s = the same positions ascending.  Its matrix is
 * d_mats + mat_off + msize * (digit * (branch_bit >= 0 ? 2 : 1) + bit), digit = the item's label digit sel_digit
 * (0 when < 0), bit = the item's branch bit branch_bit (0 when < 0), msize = 16 or 256 complex entries.
 * Sweep: ops [op_begin, op_end) on the tile of entries whose bits outside pos[0..n_tile) are fixed; pos ascending,
 * pos[k] = k for k < min(5, n_tile).  n_tile = 2n (one sweep, rho never leaves shared memory) when 2n <= 12, else 12.
 * Item (24 bytes): {uint64 digits (4 bits per digit), int32 label, uint32 branch, uint32 col_base, uint32 qmask};
 * items are sorted by label and item_begin (HOST, n_labels + 1) indexes them.  An item starts from |0><0|, runs
 * every sweep and adds Re rho[i][i] to column col_base | sum_{q in qmask} bit_q(i) << qcol[q] of its label's
 * unfolded row (2^n_cols columns); the items of one label write disjoint columns.  Then every row of
 * [label_begin, label_end) gets, for each column bit j of d_ro_mask[label], the butterfly
 * (u0, u1) -> (R00 u0 + R01 u1, R10 u0 + R11 u1) with R = d_ro[j][v] (R[o][i] = p(recorded o | measured i); v = the
 * label's digit of a configuration column, 0 for a clbit column), and
 * with fold_bits = f > 0 the top f column bits are folded with sign (-1)^bit into d_out.
 * d_out row `label` (absolute, stride out_row_stride) receives the result; d_rows (unused when fold_bits = 0: d_out
 * is used) holds the unfolded rows of the range, row label - label_begin, stride 2^n_cols.  d_work: as many rho as
 * fit when 2n > 12 (at least one, else QCK_ERR_NOMEM before anything is launched); unused otherwise. */
#define QCK_DM_MAX_TILE_BITS 12
#define QCK_DM_MAX_QUBITS 20
typedef struct {
    int32_t n_tile, op_begin, op_end;
    int32_t pos[QCK_DM_MAX_TILE_BITS];
} qck_dm_sweep;
typedef struct {
    int32_t n_qubits, n_sweeps;
    const qck_dm_sweep* sweeps;          /* HOST */
    const int32_t* d_ops;
    const double* d_mats;                /* complex128 pool */
    const void* d_items;
    const int64_t* item_begin;           /* HOST */
    int64_t n_labels;
    const uint32_t* d_ro_mask;
    const double* d_ro;                  /* [n_cols][QCK_MAX_VARIANTS][4] */
    int32_t n_cols, fold_bits;
    int32_t qcol[QCK_DM_MAX_QUBITS];
    int32_t n_digits;                    /* the top n_digits columns are configuration bits */
    int32_t radix[QCK_MAX_DIGITS];       /* label = mixed radix, last digit fastest */
} qck_dm_plan;
QCK_API int qck_sim_density(qck_handle* h, const qck_dm_plan* plan, int64_t label_begin, int64_t label_end,
                            double* d_out, int64_t out_row_stride, double* d_rows, void* d_work, size_t work_bytes,
                            qck_stream stream);

/* ------------------------------------------------------------------ reductions
 * qck_stats_dense: sum / min / nnz of a dense vector (entries |v| <= acc count as absent).
 * qck_hellinger: result[0..2] = sum p, sum q, sum sqrt(p q) over max(.,0) entries; the
 *   fidelity (Utilities.py:224, qiskit hellinger_fidelity) is (r2 / sqrt(r0 r1))^2.
 * qck_npd: QuasiDistr.nearest_probability_distribution (quasi_distr.py:28-43) on a dense
 *   vector, in place; returns beta (sum of the dropped entries) and num (survivors) on the host, so it
 *   synchronises the stream ONCE at the end (qck_npd_async + one 256-byte read-back). */
QCK_API int qck_stats_dense(qck_handle* h, const double* d_p, uint64_t n, double acc, qck_stats* d_stats,
                    qck_stream stream);
QCK_API int qck_hellinger(qck_handle* h, const double* d_p, const double* d_q, uint64_t n, double* d_result3,
                  qck_stream stream);
QCK_API int qck_npd(qck_handle* h, double* d_p, uint64_t n, double acc, double* host_beta, double* host_num,
            qck_stream stream);

/* Cross-rank reduction of a qck_stats (sums added, min min-reduced, in rank order: the same bits on every
 * rank) for results sharded over the GPUs of one box (SURVEY.md 8e: "scalar allreduce for min / sum"), WITHOUT a
 * collective launch: every rank writes its values into every peer's mailbox with NVLink stores and waits for
 * the peers' values in its own.  Setup (once): every rank allocates qck_stats_exchange_mailbox_bytes(world)
 * bytes with qck_mem_alloc, zeroes them (qck_mem_zero), exports them (qck_ipc_export) and opens the peers'
 * (qck_ipc_open); d_mailboxes = HOST array of `world` device pointers in rank order (own + mapped).  Every
 * rank must call it the same number of times; a rank whose peers never arrive traps after ~4 s instead of
 * hanging.  One launch, capturable in a CUDA graph. */
#define QCK_MAX_RANKS 16
QCK_API size_t qck_stats_exchange_mailbox_bytes(int world);
QCK_API int qck_stats_exchange(qck_handle* h, qck_stats* d_stats, int rank, int world, void* const* d_mailboxes,
                       qck_stream stream);
QCK_API int qck_mem_zero(qck_handle* h, void* d_ptr, size_t bytes, qck_stream stream);

/* The same without any host round trip: 8 launches enqueued on `stream` (statistics, <= 5 radix
 * refinement levels of 13 bits each on the ordered integer image of the doubles + one summation pass,
 * apply), each looking at the state the previous one left in the workspace; launches with nothing
 * left to do return at once.  d_ws: qck_npd_workspace_bytes() bytes of device memory, ZEROED once by
 * the caller (NULL: the handle's own - one npd in flight per handle).  After the stream has passed the
 * call the first QCK_NPD_STATE_SLOTS 8-byte slots of the workspace hold (doubles unless noted):
 *   0 sum, 1 min, 2 sum of negative entries, 3 alive entries (|v| > acc), 4 negative entries,
 *   5 status (int64: QCK_NPD_ST_*), 6 / 7 lo / hi (int64 keys: the dropped set is {key <= lo}),
 *   10 / 11 sum / count of the entries with key <= lo, 13 t0, 14 beta / num, 15 beta, 16 num. */
#define QCK_NPD_STATE_SLOTS 32
enum { QCK_NPD_ST_SEARCH = 0, QCK_NPD_ST_IDENTITY = 1, QCK_NPD_ST_SOLVED = 2, QCK_NPD_ST_NEGATIVE_TOTAL = 3,
       QCK_NPD_ST_LOCATED = 4 };
QCK_API size_t qck_npd_workspace_bytes(void);
QCK_API int qck_npd_async(qck_handle* h, double* d_p, uint64_t n, double acc, void* d_ws, qck_stream stream);

/* One stage of the above, for results SHARDED over ranks by output index (SURVEY.md 8e row 4: the ranks
 * exchange scalars and one 128 KiB histogram per level, never the distribution).  Per rank:
 *   QCK_NPD_STATS (fuse_tail = 0)  local statistics -> slots 0-4; the caller reduces them over the ranks
 *                                  (sum, min, sum, sum, sum), writes them back, then
 *   QCK_NPD_PLAN                   identity / error / first key range;
 *   repeat 6 times:
 *   QCK_NPD_LEVEL (fuse_tail = 0)  local histogram of the range: slots 10-11 (doubles) and the bins
 *                                  (2 x 8192 int64 right after the state slots); the caller sum-reduces
 *                                  both over the ranks, then
 *   QCK_NPD_SELECT                 narrows the range or finishes;
 *   QCK_NPD_APPLY                  rewrites the local shard.
 * With fuse_tail = 1 the last CTA of STATS / LEVEL runs PLAN / SELECT itself (single-rank form). */
enum { QCK_NPD_STATS = 0, QCK_NPD_PLAN = 1, QCK_NPD_LEVEL = 2, QCK_NPD_SELECT = 3, QCK_NPD_APPLY = 4 };
#define QCK_NPD_BINS 8192
QCK_API int qck_npd_stage(qck_handle* h, int stage, double* d_p, uint64_t n, double acc, void* d_ws, int fuse_tail,
                  qck_stream stream);

/* Roofline denominators MEASURED_PEAKS.json does not hold (SURVEY.md 8d), measured on this device:
 * out4 = { FP64 FMA TFLOP/s, FP64 tensor-core (DMMA m8n8k4) TFLOP/s, shared-memory load TB/s (LDS.128,
 * whole device), SM count }.  A measurement utility (bench.py records it next to its roofline figures);
 * synchronises the device, ~50 ms. */
QCK_API int qck_measure_peaks(qck_handle* h, double* out4);

/* ------------------------------------------------------------------ dense QuasiDistr algebra
 * Device forms of quasi_distr.py:45-86 on dense vectors of 2^n_bits doubles with
 * the reference's pruning (v = |v| > acc ? v : 0 after every operation).  They
 * back the per-gate operator API VirtualBinaryGate.knit(results, clbit_idx)
 * (virtual_gates.py:39) and the reference-faithful (acc = 1e-5) mode.
 */
QCK_API int qck_qd_prune(qck_handle* h, double* d_v, uint64_t n, double acc, qck_stream stream);
/* out = sqrt(max(v, 0)) (Hellinger building block) */
QCK_API int qck_qd_sqrt(qck_handle* h, const double* d_v, double* d_out, uint64_t n, qck_stream stream);
/* out = prune(a * x + b * y); y may be NULL */
QCK_API int qck_qd_axpby(qck_handle* h, double a, const double* d_x, double b, const double* d_y,
                 double* d_out, uint64_t n, double acc, qck_stream stream);
/* split on bit: lo[i] = v[insert0(i)], hi[i] = v[insert1(i)], each pruned; n = size of v */
QCK_API int qck_qd_split(qck_handle* h, const double* d_v, uint64_t n, int bit, double* d_lo, double* d_hi,
                 double acc, qck_stream stream);
/* merge: out[k] = a[k & mask_a] * b[k & mask_b] pruned (disjoint supports, XOR = OR) */
QCK_API int qck_qd_merge(qck_handle* h, const double* d_a, uint64_t mask_a, const double* d_b, uint64_t mask_b,
                 double* d_out, uint64_t n, double acc, qck_stream stream);
/* one exact knit level: out[i] = sum_r coef0[r] * v_r[insert0(i)] + coef1[r] * v_r[insert1(i)] */
QCK_API int qck_qd_knit_level(qck_handle* h, int n_results, const double* const* d_results, uint64_t n,
                      int bit, const double* coef0, const double* coef1, double* d_out,
                      qck_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* QCK_H */

/*
 * fa_b200.h — C ABI of the B200-native flash-attention engine (libfa_b200.so).
 *
 * This is the drop-in boundary for nothingstopsme/tf_flash_attention: every entry
 * point replaces one member of the reference's C++ launcher template
 *   cuda_launch::FlashAttentionLauncher<T, RefShape, OrderMap, Policy>
 *   (reference: flash_attention/kernel/flash_attention.h:220-260)
 * plus the host helpers the reference's TF OpKernels run before calling it
 *   (flash_attention/kernel/flash_attention_forward.cc:97-140,280-386 and
 *    flash_attention/kernel/flash_attention_backward.cc:181-344).
 * Plain pointers and sizes only; no TensorFlow, PyTorch or CuTe types.
 *
 * Tensors are dense, channel-first, row-major, exactly as TensorFlow hands them
 * to the reference op:   Q [batch, d, q...]  K [batch, d, k...]  V [batch, v_d, k...]
 *                        O [batch, v_d, q...]  l, m [batch, q...]
 * with every leading batch axis (heads included) flattened into `batch` and the
 * 1 or 2 sequence axes flattened row-major (q = prod(q_shape), k = prod(k_shape)).
 *
 * All functions are re-entrant and asynchronous with respect to the host: work is
 * enqueued on `stream` and no host synchronisation happens (like the reference,
 * flash_attention_forward.cc:371-385). The caller owns every buffer, workspace
 * included; the library never allocates device memory.
 */
#ifndef FA_B200_H_
#define FA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* dtype of Q/K/V/O/m and the gradients. `l` is float for FA_F16 and T otherwise
 * (reference: flash_attention.h:181-185, flash_attention_forward.cc:151-153,187-189).
 * FA_BF16 (no reference counterpart) follows the FA_F16 contract exactly: `l` is float, `m` is rounded to bf16 and `l`
 * re-expressed against the rounded `m`, empty rows get o = 0, l = 0, m = bytes 0xFA. */
enum { FA_F16 = 0, FA_F32 = 1, FA_F64 = 2, FA_BF16 = 3 };
/* masking rule (reference policies, flash_attention.h:45-149) */
enum { FA_RULE_FULL = 0, FA_RULE_CAUSAL = 1, FA_RULE_LOCAL = 2 };
/* sync mode (reference: sync_methods.cc:113-117) */
enum { FA_SYNC_NONE_FRONT = 0, FA_SYNC_SCALE_FRONT = 1, FA_SYNC_SCALE_END = 2 };

/* tensor layout of q, k, v, o (and d_o, d_q, d_k, d_v). The reference's ops are channel-first only and expect an
 * einsum either side (README.md:40); channel-last is read and written directly through 4-D TMA descriptors by the
 * 16-bit (fp16 / bf16) tensor-core kernels, which removes those transposes. l, m are [batch, q] in both layouts. */
enum {
  FA_LAYOUT_CHANNEL_FIRST = 0, /* [batch..., channels, sequence...]                          */
  FA_LAYOUT_CHANNEL_LAST = 1   /* [outer, sequence..., heads, channels], batch = outer*heads */
};

/* status codes; 0 = ok. Each FA_EINVAL_* mirrors one reference check. */
enum {
  FA_OK = 0,
  FA_EINVAL_NULL = -1,         /* null problem / pointer                                   */
  FA_EINVAL_DTYPE = -2,        /* dtype not in {f16,f32,f64,bf16} (op "T" attr constraint)  */
  FA_EINVAL_SEQ_DIMS = -3,     /* seq_dims not 1 or 2            (ops exist for 1d/2d only) */
  FA_EINVAL_RULE = -4,         /* rule not in {full,causal,local}                           */
  FA_EINVAL_SYNC_MODE = -5,    /* "Unsupported sync_mode: ..."   forward.cc:275-276         */
  FA_EINVAL_WINDOW = -6,       /* window_size < 1                forward.cc:173 (int >= 1)  */
  FA_EINVAL_STRIDE = -7,       /* log2_stride_size < 0, >= 31 or window<<stride overflows   */
                               /*                                flash_attention.h:90       */
  FA_EINVAL_SHAPE = -8,        /* a dimension < 1, or q/k/orders do not fit int32           */
  FA_EINVAL_WORKSPACE = -9,    /* workspace smaller than fa_workspace_bytes(), or needed and */
                               /* NULL or not 256-byte aligned (host arenas: always)        */
  FA_EINVAL_RANK = -10,        /* fa_check_*_shapes: rank mismatch / rank < seq_dims+2      */
  FA_EINVAL_CHANNEL = -11,     /* fa_check_*_shapes: channel mismatch                       */
  FA_EINVAL_BATCH = -12,       /* fa_check_*_shapes: batch shapes differ                    */
  FA_EINVAL_SEQ_SHAPE = -13,   /* fa_check_*_shapes: sequence shapes differ                 */
  FA_EINVAL_LAYOUT = -14,      /* layout / heads invalid, or channel-last asked of a path that cannot read it */
  FA_ECUDA = -100,             /* a CUDA call failed; fa_last_cuda_error() has the code     */
  FA_ENODEVICE = -101          /* no sm_100 device is current                               */
};

typedef struct fa_problem_t {
  int32_t dtype;            /* FA_F16 | FA_F32 | FA_F64 | FA_BF16                            */
  int32_t seq_dims;         /* 1 or 2                                                        */
  int32_t rule;             /* FA_RULE_*                                                     */
  int32_t window_size;      /* local only, >= 1; attended span per dim = 2*window-1          */
  int32_t log2_stride_size; /* local only, 0..30                                             */
  int32_t is_causal;        /* local only                                                    */
  int32_t sync_mode;        /* FA_SYNC_*                                                     */
  int32_t d;                /* channels of Q and K                                           */
  int32_t v_d;              /* channels of V and O                                           */
  int32_t layout;           /* FA_LAYOUT_*; 0 (channel-first) is the reference's layout      */
  int64_t batch;            /* product of all batch axes (heads included)                    */
  int32_t q_shape[2];       /* TF axis order (outer, inner); 1-D uses q_shape[0]             */
  int32_t k_shape[2];
  /* K/V-ring support (one long sequence sharded over GPUs): this call sees rows
   * [q_index_base, q_index_base + q_shape[0]) of a longer logical sequence whose full
   * length is q_full_len (same for k). All zeros = not sharded (the reference
   * has no such notion; the rule is evaluated on global coordinates). 1-D only. */
  int32_t q_index_base;
  int32_t k_index_base;
  int32_t q_full_len;       /* 0 = q_shape[0]                                                */
  int32_t k_full_len;       /* 0 = k_shape[0]                                                */
  /* 1 = `o`,`l`,`m` already hold a partial result of the same rows (from earlier
   * K/V shards) and this call merges into them online; 0 = overwrite.              */
  int32_t accumulate;
  int32_t heads;            /* FA_LAYOUT_CHANNEL_LAST only: innermost batch axis (>= 1)      */
} fa_problem_t;

/* ---- the hot path ------------------------------------------------------------- */

/* Replaces FlashAttentionLauncher::Forward (flash_attention.h:225-236) together with
 * the four cudaMemsetAsync calls that precede it (flash_attention_forward.cc:352-369):
 * every element of o, l, m is written by the kernels themselves.
 *   o : T  [batch, v_d, q]     l : float (f16, bf16) or T  [batch, q]     m : T [batch, q]
 * Rows with no attended key get o = 0, l = 0, m = bytes 0xFA.. (type_util.h:43-45).
 * `stream` is a cudaStream_t passed as void*. */
int fa_forward(const fa_problem_t* p, const void* q, const void* k, const void* v,
               void* o, void* l, void* m, void* workspace, size_t workspace_bytes, void* stream);

/* Replaces FlashAttentionLauncher::Backward (flash_attention.h:238-249) plus its four
 * memsets (flash_attention_backward.cc:309-323). Inputs o, l, m are the forward outputs.
 *   d_q : T [batch, d, q]    d_k : T [batch, d, k]    d_v : T [batch, v_d, k]       */
int fa_backward(const fa_problem_t* p, const void* q, const void* k, const void* v,
                const void* o, const void* l, const void* m, const void* d_o,
                void* d_q, void* d_k, void* d_v, void* workspace, size_t workspace_bytes,
                void* stream);

/* Device scratch the caller must provide (replaces the reference's allocate_temp of
 * Br_occupancy, flash_attention_forward.cc:330 / flash_attention_backward.cc:283).
 * May be 0. When it is not, the workspace must be 256-byte aligned: fa_forward, fa_backward
 * and fa_backward_accumulate return FA_EINVAL_WORKSPACE before any launch otherwise. */
size_t fa_workspace_bytes(const fa_problem_t* p, int is_backward);

/* Replaces FlashAttentionLauncher::EstimateForwardFlops (flash_attention.h:254-260,
 * flash_attention.cu:2069-2144): the reference's per-(Bc,Br)-block-pair estimate for a
 * device with `shared_mem_bytes` of opt-in shared memory per block (pass 0 to use
 * B200's 232448). Host only; writes *flops. */
int fa_estimate_forward_flops(const fa_problem_t* p, int32_t shared_mem_bytes, float* flops);

/* ---- partial results over disjoint key shards (K/V ring; new, the reference is single-GPU) ----- */

/* Folds the partial result of one key shard (o_part, l_part, m_part exactly as fa_forward wrote
 * them for problem *p) into running accumulators with the online-softmax algebra:
 *   o_acc [batch, v_d, q], l_acc [batch, q], m_acc [batch, q]   float (double for FA_F64);
 * o_acc is unnormalised (sum of exp(s - m_acc) * v). first != 0 initialises the accumulators. */
int fa_partial_merge(const fa_problem_t* p, const void* o_part, const void* l_part, const void* m_part,
                     void* o_acc, void* l_acc, void* m_acc, int first, void* stream);
/* Emits O = o_acc / l_acc, l, m in the reference's output contract (sentinel on empty rows). */
int fa_partial_finalize(const fa_problem_t* p, const void* o_acc, const void* l_acc, const void* m_acc,
                        void* o, void* l, void* m, void* stream);

/* Ring backward: a gradient shard (dQ of the local queries, or the dK / dV that travel with their K/V
 * shard) is the sum of the fa_backward results of every (query chunk, key chunk) block; each call is
 * made with the FINAL l, m, O of the whole sequence, so the blocks simply add.
 *   fa_grad_accumulate: acc[i] = (first ? 0 : acc[i]) + part[i]    acc float (double for FA_F64)
 *   fa_grad_finalize  : out[i] = (dtype) acc[i]                                                  */
int fa_grad_accumulate(int32_t dtype, const void* part, void* acc, int64_t n, int first, void* stream);
/* The same sum for dQ made inside the backward launch: dq_acc [dq_fold, d, q] is a float accumulator that dQ of
 * problem *p is ADDED into (finished values: the softmax scale is applied); batch element pb adds into accumulator
 * element pb % dq_fold (0 = batch: one accumulator element per batch element; batch / 2: the two halves of a
 * [Q_hi; Q_hi] pair launch of the ring fold into the same accumulator). d_k, d_v are written as by fa_backward.
 * Saves the dQ scratch memset, the convert pass, the fp16 / bf16 dQ tensor and its fa_grad_accumulate pass per block.
 * Available where fa_backward_accumulate_supported() says so (fp16 or bf16, channel-first, head_dim 128 with 64 or 128 value
 * channels, lengths multiples of 8: the fused dQ/dK/dV kernel, whose TMA reduce-add then lands in dq_acc directly);
 * FA_EINVAL_SHAPE otherwise, and the caller uses fa_backward + fa_grad_accumulate. Workspace as for fa_backward. */
int fa_backward_accumulate_supported(const fa_problem_t* p, int64_t dq_fold);
int fa_backward_accumulate(const fa_problem_t* p, const void* q, const void* k, const void* v, const void* o,
                           const void* l, const void* m, const void* d_o, void* dq_acc, void* d_k, void* d_v,
                           int64_t dq_fold, void* workspace, size_t workspace_bytes, void* stream);
int fa_grad_finalize(int32_t dtype, const void* acc, void* out, int64_t n, void* stream);

/* Layout adapter for the step either side of the op (no reference counterpart: README.md:40 of the reference assumes an
 * einsum either side of the op that builds the channel-first layout; SURVEY.md section 8, row f3).
 * to_channel_first != 0: x [batch, seq, heads, channels] -> y [batch, heads, channels, seq]; otherwise the inverse. Same dtype codes as fa_problem_t. HBM-bound transpose, asynchronous on `stream`.       */
int fa_layout_transpose(int32_t dtype, const void* x, void* y, int64_t batch, int64_t seq, int32_t heads,
                        int32_t channels, int to_channel_first, void* stream);

/* ---- host-side helpers shared with the kernels (same code, fa_rules.h) ---------- */

/* Number of attended (q,k) pairs per batch element under the bit-exact rule; the unit
 * of the unmasked-FLOP metric: fwd = 2*nnz*(d+v_d)*batch, bwd = 2*nnz*(3d+2v_d)*batch. */
int fa_count_attended(const fa_problem_t* p, int64_t* nnz);

/* Writes the dense attended-index pattern, mask[q*k] (1 = attended), evaluated by the
 * very same inline functions the kernels use. For tests / debugging. */
int fa_pattern_mask(const fa_problem_t* p, uint8_t* mask);

/* The same pattern assembled from the closed-form 32-column masks the tcgen05 kernels build per tile
 * (queries resident: forward / dQ kernels; keys resident: dK/dV kernel). For tests.               */
int fa_pattern_mask_fast(const fa_problem_t* p, int32_t tile, int32_t resident_is_q, uint8_t* mask);

/* Orders of the Q and K entries in the shared power-of-two reference grid
 * (sync_methods.h:56-85); q_order[q], k_order[k], ref_shape[seq_dims] innermost first. */
int fa_orders(const fa_problem_t* p, int32_t* q_order, int32_t* k_order, int32_t* ref_shape);

/* Tile schedule the kernels derive for (q tile of `tile_q` rows) x (k tile of `tile_k`):
 * cls[nq_tiles*nk_tiles] = 0 skip (never loaded), 1 partial (element mask), 2 full. */
int fa_classify_tiles(const fa_problem_t* p, int32_t tile_q, int32_t tile_k, uint8_t* cls);

/* Shape validation exactly as the reference OpKernels do it, on un-flattened TF shapes.
 * Fills batch, d, v_d, q_shape, k_shape of *p (other fields untouched).
 *   forward : flash_attention_forward.cc:97-140      backward: flash_attention_backward.cc:197-258 */
int fa_check_forward_shapes(int32_t seq_dims, int32_t rank_q, const int64_t* q_dims,
                            int32_t rank_k, const int64_t* k_dims,
                            int32_t rank_v, const int64_t* v_dims, fa_problem_t* p);
int fa_check_backward_shapes(int32_t seq_dims, int32_t rank_q, const int64_t* q_dims,
                             int32_t rank_k, const int64_t* k_dims,
                             int32_t rank_v, const int64_t* v_dims,
                             int32_t rank_o, const int64_t* o_dims,
                             int32_t rank_l, const int64_t* l_dims,
                             int32_t rank_m, const int64_t* m_dims,
                             int32_t rank_do, const int64_t* do_dims, fa_problem_t* p);

/* ---- the reference-facing plugin call with HOST buffers -------------------------- */

/* Same contract as fa_forward / fa_backward but every tensor pointer is HOST memory
 * (pinned or pageable). The library stages through the caller-provided device arena
 * `dev_arena` (>= fa_host_arena_bytes, 256-byte aligned, else FA_EINVAL_WORKSPACE), copies
 * in, runs, copies the results back and returns after the stream has drained. Used for the
 * end-to-end number in bench.py. */
size_t fa_host_arena_bytes(const fa_problem_t* p, int is_backward);
int fa_forward_host(const fa_problem_t* p, const void* q, const void* k, const void* v,
                    void* o, void* l, void* m, void* dev_arena, size_t dev_arena_bytes, void* stream);
int fa_backward_host(const fa_problem_t* p, const void* q, const void* k, const void* v,
                     const void* o, const void* l, const void* m, const void* d_o,
                     void* d_q, void* d_k, void* d_v, void* dev_arena, size_t dev_arena_bytes,
                     void* stream);
/* Backward of the forward that fa_forward_host has just run in the SAME arena. The arena must have been sized with
 * fa_host_arena_bytes(p, 1) for that forward call too (the forward and backward layouts share the offsets of Q, K, V,
 * O, l, m) and must not have been written since: those six tensors are taken from the arena and only d_o is uploaded.
 * This is what the reference's host framework does between the forward op and its registered gradient
 * (flash_attention.py:374-390: the gradient receives op.inputs / op.outputs, which TensorFlow keeps on the device). */
int fa_backward_host_resident(const fa_problem_t* p, const void* d_o, void* d_q, void* d_k, void* d_v,
                              void* dev_arena, size_t dev_arena_bytes, void* stream);

/* One training step on host buffers: forward, then the gradient, pipelined over batch chunks so that the uploads of
 * Q, K, V, d_o of the next chunk overlap the kernels of the current one and the downloads of O, l, m, d_q, d_k, d_v of
 * the previous one (both PCIe directions busy for the whole step). Same results as fa_forward_host followed by
 * fa_backward_host. Arena >= fa_step_host_arena_bytes(p); p->accumulate must be 0. Returns after the stream drained. */
size_t fa_step_host_arena_bytes(const fa_problem_t* p);
int fa_forward_backward_host(const fa_problem_t* p, const void* q, const void* k, const void* v, const void* d_o,
                             void* o, void* l, void* m, void* d_q, void* d_k, void* d_v, void* dev_arena,
                             size_t dev_arena_bytes, void* stream);

/* ---- diagnostics ---------------------------------------------------------------- */
const char* fa_strerror(int status);
int fa_last_cuda_error(void);          /* cudaError_t of the last FA_ECUDA on this thread */
/* Which kernel family the last fa_forward/fa_backward in this process dispatched to:
 * 0 none, 1 generic SIMT (FFMA / DFMA), 2 tcgen05 16-bit (fp16 / bf16), 3 tcgen05 fp32 split precision
 * (forward: 3xTF32; backward: three bf16 pieces per operand), 4 fp64 on the FP64 tensor cores (DMMA). */
int fa_last_path(void);
/* The same answer BEFORE the call, host only: which family fa_forward (is_backward = 0) / fa_backward will take for *p
 * given 256-byte-aligned tensors and a workspace of fa_workspace_bytes(). When it is 1 (generic kernels) `reason`
 * (may be NULL) receives why the tensor-core family declines: channel counts, a sequence beyond the 2048 streamed tiles
 * of a CTA's schedule, accumulate, ... Negative = the FA_EINVAL_* the call would return.                          */
int fa_dispatch_path(const fa_problem_t* p, int is_backward, char* reason, size_t reason_len);
/* Number of kernel launches issued by this library in this process since the last reset. */
int64_t fa_launch_count(int reset);
/* Per-kernel device timing for bench.py: when enabled every kernel this library launches is
 * bracketed by CUDA events on the launching stream. fa_kernel_timings() synchronises on them,
 * returns up to max_entries (name, milliseconds) pairs in launch order and clears the list.   */
void fa_kernel_timing(int enable);
int fa_kernel_timings(int max_entries, const char** names, float* ms);
/* Force a kernel family (testing): 0 auto, 1 generic only, 4 fp16 / bf16 backward as the two-kernel
 * (dQ, then dK/dV) variant instead of the fused kernel, 5 fp16 / bf16 head_dim-64 forward with 128-key
 * tiles and one CTA per SM instead of 64-key tiles and two CTAs per SM. Developer A/B values:
 * 7 / 8 / 9 = element-wise kernels of fa_layout_transpose (pairs / singles / quads of halves). */
void fa_set_path_override(int path);
/* Precision of the fp16 gradients. The plain fp16 backward hands P and dS to the tensor cores as single fp16 values
 * and takes D = rowsum(dO o O) from the fp16 O it is given; where rows attend few keys (P ~ 1) each of the three costs
 * up to ~1e-3 per term, and a key that collects many such rows ends above the 2e-3 bar (4.2e-3 measured at 1000
 * queries x 88 keys). The "precise" kernels pass P and dS as hi + lo pairs of fp16 values (two tensor-core products
 * each) and re-derive D exactly as rowsum(P o dP) inside the dQ kernel: gradients within ~5e-4 (the fp16 rounding of the
 * result itself) on those cases, for ~12 % more time on HBM-bound problems.
 *   mode 0 (default): automatic; precise where every row attends at most 32 keys, and under causal rules where the
 *          sequence is short (<= 128 keys) or has >= 4 queries per key; the plain kernels elsewhere (long rows, small P;
 *          the fused head_dim-128 kernel always: its TMEM has no room for the lo halves);
 *   mode 1: precise everywhere (head_dim 128 then runs the two-kernel backward, with the hi + lo operands but D from O);
 *   mode 2: never (round-1 behaviour).
 * The reference accumulates these products in fp16 altogether (flash_attention.cu:284-286); no counterpart there.
 * bf16 follows the same three modes on the same kernels (hi + lo pairs of bf16 values).
 * Returns FA_OK or FA_EINVAL_SHAPE for an unknown mode.                                                         */
int fa_set_grad_precision(int mode);
const char* fa_version(void);
/* Launch-plan cache counters (csrc/fa_plan.h): out4 = {tensor-map encodes, tensor-map cache hits,
 * cudaFuncSetAttribute calls, attribute cache hits} since the last reset. A repeated call on the same buffers makes no
 * driver call besides its kernel launches: the first two / second two counters move only in their "hits" half.    */
int fa_plan_stats(uint64_t* out4, int reset);

/* ---- K/V ring data plane (single long sequence sharded over the GPUs of a node; new functionality, the reference is
 * single-GPU). Shards move between neighbouring ranks as peer copies on the copy engines (NVLink 5 / NVSwitch) into
 * receive slots exported with CUDA IPC; arrival and reuse are stream-ordered flag waits (no kernel, no host sync). One
 * process per GPU; every rank makes the same sequence of calls. csrc/fa_ring.cu.
 *   fa_ring_create        allocates n_slots receive slots of slot_bytes on the current device and fills handle_blob
 *                         (FA_RING_HANDLE_BYTES) for the neighbours; the caller exchanges the blobs (any channel);
 *   fa_ring_connect       opens the blobs of rank+1 (destination of fa_ring_send) and rank-1;
 *   fa_ring_slot          device pointer of a local receive slot;
 *   fa_ring_send          after the work queued on after_stream so far (and, when forwarded_slot >= 0, once that local
 *                         slot has been filled; and once the neighbour has released dst_slot), copies n_parts pieces
 *                         (each placed at the next 256-byte boundary) into dst_slot of rank+1 and marks it filled;
 *   fa_ring_recv_wait     `stream` waits until the next fill of `slot` has arrived;
 *   fa_ring_recv_release  after the work queued on `stream` so far (and after any forwarding copy of the slot), marks
 *                         the slot reusable for rank-1.                                                              */
#define FA_RING_HANDLE_BYTES 128
typedef struct fa_ring fa_ring_t;
int fa_ring_create(int32_t rank, int32_t world, size_t slot_bytes, int32_t n_slots, fa_ring_t** out, void* handle_blob);
int fa_ring_connect(fa_ring_t* ring, const void* next_rank_blob, const void* prev_rank_blob);
void* fa_ring_slot(fa_ring_t* ring, int32_t slot);
int fa_ring_send(fa_ring_t* ring, int32_t dst_slot, int32_t n_parts, const void* const* src, const size_t* bytes,
                 int32_t forwarded_slot, void* after_stream);
int fa_ring_recv_wait(fa_ring_t* ring, int32_t slot, void* stream);
int fa_ring_recv_release(fa_ring_t* ring, int32_t slot, void* stream);
int fa_ring_destroy(fa_ring_t* ring);

/* ---- K/V ring driver: causal_1d forward / backward of one sequence sharded zig-zag over the ring's ranks (rank r of G
 * holds chunks r and 2G-1-r of 2G chunks of `chunk` positions), as one call per rank on one stream. All tensors are
 * chunk-major: q2, k2, dq2, dk2 [2, batch, d, chunk]; v2, o2, do2, dv2 [2, batch, v_d, chunk]; l2, m2 [2, batch, chunk]
 * (index 0 = chunk r, 1 = chunk 2G-1-r). Per ring step: one fa_forward / fa_backward launch over both local query
 * chunks (step 0: both diagonal blocks as one causal launch plus Q_hi x K_lo; later steps: two full blocks), results
 * folded with fa_partial_merge / fa_grad_accumulate, the K/V shard of the step travelling to rank+1 on the copy
 * engines while it is being used; in the backward the fp32 dK / dV accumulators travel one hop behind their shard
 * through `acc_ring` and are home after G hops. Every rank makes the same call; nothing synchronises with the host.
 *   kv_ring : slots >= fa_ring_causal_slot_bytes(.., 0), >= 2 slots; NULL = a single rank (world 1)
 *   acc_ring: backward only, slots >= fa_ring_causal_slot_bytes(.., 1)
 *   arena   : device scratch, 256-byte aligned, >= fa_ring_causal_arena_bytes(.., world, backward)
 * Gradients are made with the FINAL o2, l2, m2 that fa_ring_causal_forward returned. The Python mirror of the same
 * schedule (ring.py: ring_forward_causal / ring_backward_causal) is what the gloo tests pin against the oracle.    */
size_t fa_ring_causal_arena_bytes(int32_t dtype, int64_t batch, int32_t d, int32_t v_d, int32_t chunk, int32_t world,
                                  int32_t backward);
size_t fa_ring_causal_slot_bytes(int32_t dtype, int64_t batch, int32_t d, int32_t v_d, int32_t chunk,
                                 int32_t accumulators);
int fa_ring_causal_forward(fa_ring_t* kv_ring, int32_t dtype, int64_t batch, int32_t d, int32_t v_d, int32_t chunk,
                           const void* q2, const void* k2, const void* v2, void* o2, void* l2, void* m2, void* arena,
                           size_t arena_bytes, void* stream);
int fa_ring_causal_backward(fa_ring_t* kv_ring, fa_ring_t* acc_ring, int32_t dtype, int64_t batch, int32_t d,
                            int32_t v_d, int32_t chunk, const void* q2, const void* k2, const void* v2, const void* o2,
                            const void* l2, const void* m2, const void* do2, void* dq2, void* dk2, void* dv2,
                            void* arena, size_t arena_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FA_B200_H_ */

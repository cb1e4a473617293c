/*
 * tpnet_b200 — C ABI of the B200 (sm_100a) temporal-walk-matrix projection library.
 *
 * This is the drop-in boundary for ONE hot path of lxd99/TPNet: the state and
 * operations of `RandomProjectionModule` (reference: models/TPNet.py:9-157).
 * The reference has no FFI of its own (it is pure PyTorch); each entry point
 * below names the reference lines it replaces.  The Python host side
 * (tpnet_b200/random_projection.py) binds these symbols with ctypes and passes
 * `tensor.data_ptr()` values and the current CUDA stream; see INTEGRATION.md.
 *
 * Conventions
 *   - extern "C", POD arguments only; every pointer named `*_dev`/documented as
 *     device memory is a CUDA device pointer, everything else is host memory.  All device
 *     pointers of one call live on ONE device; the call runs there whatever the caller's
 *     current device is (it is looked up from the state / first device pointer and the
 *     caller's current device is restored on return), and `stream` must belong to it.
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*),
 *     never synchronises, never allocates; scratch memory is supplied by the
 *     caller (size from tpn_update_workspace_bytes).
 *   - return value: TPN_OK (0) or a negative TPN_ERR_* code; never throws.
 *   - node ids are int64, 0 <= id < num_nodes (id 0 is the reference's padding
 *     node: P_0[0] random, P_{>=1}[0] zero — it is an ordinary row here).
 *
 * State layout in HBM (node-major, one contiguous block per node):
 *     value of layer l (0..L), column k (0..dim) of node u  =
 *         data[u * node_stride + l * row_stride + k]
 *   row_stride  >= dim,  multiple of 4 floats (16 B) so rows are float4-addressable;
 *   node_stride >= (L+1) * row_stride, multiple of 4.
 *   Columns [dim, row_stride) of every row MUST be zero (the kernels rely on it
 *   and preserve it).
 *   With this layout the reference's "P_i[u] += P_{i-1}[v] * w for i = L..1"
 *   (TPNet.py:90-96) is ONE contiguous axpy of L*row_stride floats per message,
 *   and the 2L+2 rows a pair-wise feature needs (TPNet.py:119-121) are two
 *   contiguous blocks.
 *
 * Time decay (TPNet.py:83-85).  The reference multiplies every row of layers
 * 1..L by the fp32 scalar c_l = f32(exp(-lambda*dt)^l) at EVERY update.  Two
 * realisations:
 *   eager : stamps == NULL.  tpn_update sweeps the whole state once per call:
 *           the reference's own multiply chain, bit for bit.
 *   lazy  : stamps != NULL (the per-node rescale of large graphs).  tpn_update
 *           appends one epoch to `decay_log` and touches only the rows of the
 *           batch.  Row e of the log holds the f64 cumulative products
 *           Q_l[e] = c_l(1)*...*c_l(e) of the fp32 factors (row 0 = 1.0).  A row
 *           last written at epoch s is brought current with ONE multiply by
 *           f32(Q[epoch]/Q[s]) — the product of exactly the factors the
 *           reference applied, rounded once instead of once per update
 *           (relative difference <= (epoch-s+1)*2^-24; identical for epoch-s <= 1).
 *           No N-proportional traffic.  Every reader (update / pairwise / gather)
 *           rescales on the fly; tpn_materialize writes all rows back current.
 */
#ifndef TPNET_B200_H_
#define TPNET_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TPN_ABI_VERSION 16

#define TPN_MAX_LAYERS 4

enum {
    TPN_OK = 0,
    TPN_ERR_INVALID_ARGUMENT = -1,   /* null pointer, bad shape, misaligned stride            */
    TPN_ERR_WORKSPACE_TOO_SMALL = -2,
    TPN_ERR_LOG_FULL = -3,           /* lazy mode: decay_log full or products near underflow    */
    TPN_ERR_CUDA = -4,               /* a CUDA runtime call failed; see tpn_last_cuda_error()   */
    TPN_ERR_UNSUPPORTED = -5,        /* num_layer outside 1..TPN_MAX_LAYERS                     */
    TPN_ERR_INDEX = -6               /* tpn_stage: a node id is out of range                    */
};

/* The L+1 projection matrices P_0..P_L of the reference's
 * `self.random_projections` (TPNet.py:39-62) plus the lazy-decay bookkeeping. */
typedef struct tpn_state {
    float*   data;          /* device, [num_nodes][node_stride] fp32                           */
    int64_t  num_nodes;     /* N, including the padding node 0                                 */
    int32_t  num_layer;     /* L, 1..TPN_MAX_LAYERS                                            */
    int32_t  dim;           /* d, logical row width (TPNet.py:30-33,45)                        */
    int64_t  row_stride;    /* floats, multiple of 4, >= dim                                   */
    int64_t  node_stride;   /* floats, multiple of 4, >= (L+1)*row_stride                      */
    int32_t* stamps;        /* device, [num_nodes][L] epoch of last write of layer 1..L; NULL = eager.
                               -1 = never written: that row MUST be all zero (update reads such target and source
                               rows as zero without loading them; gather, gather_blocks and the received-row loads of
                               tpn_update_messages read them as stored) */
    double*  decay_log;     /* device, [log_capacity][L] f64; row e = cumulative product of the
                               fp32 factors of epochs 1..e; row 0 MUST be 1.0 (caller-initialised) */
    int64_t  log_capacity;  /* rows in decay_log                                               */
    int64_t  epoch;         /* current epoch (0 = nothing logged); advanced by tpn_update      */
    double   cum_floor;     /* host mirror: smallest cumulative product in the log (1.0 at epoch 0);
                               maintained by tpn_update / tpn_reset_epoch / tpn_clear_walk_layers.
                               tpn_update returns TPN_ERR_LOG_FULL before it could underflow.   */
    int32_t* err_flag;      /* device int32 or NULL: set to 1 by tpn_pairwise / tpn_pairwise_neighbors /
                               tpn_gather / tpn_gather_blocks when a DEVICE-RESIDENT id is outside
                               [-num_nodes, num_nodes) — the reference's IndexError (TPNet.py:109), which a
                               kernel cannot raise; negative ids wrap as tensor indexing does; the access is
                               clamped only to stay in bounds.  The host polls the flag.                */
    int32_t  giant_chunk;   /* accumulation order of one target row's messages in tpn_update[_messages]:
                               0 (default) = the reference's order: one message at a time, sequentially
                                 (what CPU scatter_add_ does, TPNet.py:93-96) — bit-identical to it;
                               C > 0 (multiple of 32, 256..2048) = CHUNKED order for rows receiving >= 2048
                                 messages in one call: the messages are cut, in order, into chunks of C;
                                 every chunk is summed sequentially from +0; the chunk sums are then added
                                 to the (decayed) row in chunk order.  Deterministic and independent of the
                                 launch geometry; differs from the sequential order only by fp32 rounding
                                 (|diff| <= ~1e-6 * sum|terms|, smaller than sequential-vs-exact), and lets
                                 the add chain of a hub run in parallel.  Rows with < 2048 messages always
                                 use the reference order.                                               */
    int32_t  reserved0;
} tpn_state_t;

int tpn_version(void);
const char* tpn_error_string(int code);
/* text of the last CUDA error seen by this library on the calling thread ("" if none) */
const char* tpn_last_cuda_error(void);
/* SM count / compute capability of the current device (checks the library can run here). */
int tpn_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* Scratch bytes tpn_update needs for a batch of `batch` edges on state `st` (uses num_layer
 * and row_stride only; monotone in batch up to the snapshot threshold). */
size_t tpn_update_workspace_bytes(const tpn_state_t* st, int64_t batch);

/*
 * RandomProjectionModule.update — TPNet.py:67-99.
 *   src_dev, dst_dev : int64[batch] device   (TPNet.py:74-75)
 *   t_dev            : float64[batch] device (cast to fp32 inside, TPNet.py:77)
 *   t_last           : node_interact_times[-1] (the LAST element, TPNet.py:76)
 *   neg_lambda       : f32(-time_decay_weight)
 *   decay            : HOST pointer to c_1..c_L = f32(pow(exp(-lambda*(t_last-now)), l))
 *                      computed in f64 by the caller exactly as TPNet.py:84-85 does,
 *                      or NULL when the clock did not move (all factors are 1.0).
 *   err_flag_dev     : optional device int32; set to 1 if an id was out of range
 *                      (such edges are dropped).  May be NULL.
 * Semantics: weights w_j (TPNet.py:78); decay (eager sweep or new lazy epoch);
 * for every layer i = L..1 and every target row, messages are added one at a
 * time in the reference's order — first the row's occurrences as `src` in batch
 * order, then its occurrences as `dst` (the two scatter_add_ of TPNet.py:93-96)
 * — with the product rounded to fp32 before the add, no atomics, no FMA
 * contraction.  Layer i reads the pre-batch (decayed) layer i-1.
 * The caller's `now_time` bookkeeping (TPNet.py:99) stays on the host.
 */
int tpn_update(tpn_state_t* st,
               const int64_t* src_dev, const int64_t* dst_dev, const double* t_dev, int64_t batch,
               double t_last, float neg_lambda, const float* decay,
               void* ws_dev, size_t ws_bytes, int32_t* err_flag_dev, void* stream);

/* tpn_update in two halves (no reference counterpart; same arguments, same results, bit for bit).
 *   TPN_UPDATE_PREPARE : everything that does NOT write the state — the weights, the stable sort of the messages by
 *                        target, the work lists and (lazy decay) the pre-batch snapshot.  `st` is not modified.
 *                        May be launched on a side stream while other kernels still READ the state (the pair-wise
 *                        calls of the same batch: TPNet.py's loop computes features of a batch, then updates with it).
 *   TPN_UPDATE_APPLY   : the rest (eager sweep + snapshot, the walkers, the stamps); advances st->epoch.  Must be
 *                        ordered after the PREPARE half (caller: event) and after every read of the pre-batch state.
 *   TPN_UPDATE_WHOLE   : both, i.e. tpn_update.
 * The same workspace, arguments and `st` must be passed to both halves, with no other tpn_update* call between.
 * Batches of <= 2048 edges are not split (PREPARE is a no-op, APPLY does everything). */
#define TPN_UPDATE_WHOLE 0
#define TPN_UPDATE_PREPARE 1
#define TPN_UPDATE_APPLY 2
int tpn_update_phase(tpn_state_t* st,
                     const int64_t* src_dev, const int64_t* dst_dev, const double* t_dev, int64_t batch,
                     double t_last, float neg_lambda, const float* decay,
                     void* ws_dev, size_t ws_bytes, int32_t* err_flag_dev, void* stream, int phase);

/* Test hook: selects code paths that are otherwise chosen by size.  Returns the previous flags.
 *   TPN_DEBUG_PER_LAYER_WALK : large batches use one walk launch per layer (top-down) instead of
 *                              the pre-batch snapshot + single all-layer launch. */
#define TPN_DEBUG_PER_LAYER_WALK 1
/*   TPN_DEBUG_SERIAL_WALK    : large batches run the hub walker and the short-segment walker one
 *                              after the other on the caller's stream (default: concurrently, the
 *                              hub walker on a library-owned side stream forked/joined by events). */
#define TPN_DEBUG_SERIAL_WALK 2
/*   TPN_DEBUG_SNAPSHOT_P0    : the pre-batch snapshot also copies P_0 of every target, so the walkers read ALL
 *                              source rows from one compact buffer (A/B measurements; results are identical). */
#define TPN_DEBUG_SNAPSHOT_P0 4
/*   TPN_DEBUG_HEAD_FFMA      : tpn_head_forward runs the packed-FFMA fp32 kernel (tpn_head.cu) instead of the tcgen05
 *                              tensor-core kernel (fp16 x 2 split operands, fp32 accumulation in TMEM; tpn_head_tc.cu). */
#define TPN_DEBUG_HEAD_FFMA 8
/*   TPN_DEBUG_LEGACY_FRONT   : large batches run the sort front end as 12-13 separate launches (prep, histogram /
 *                              prefix / scatter per radix pass, payload, giant ordering) instead of the one
 *                              cooperative launch with grid barriers; results are identical. */
#define TPN_DEBUG_LEGACY_FRONT 16
/*   TPN_DEBUG_NO_STREAM      : no giant segment is streamed: the hub walker gathers and adds every one on the same SM.
 *   TPN_DEBUG_STREAM_ALL     : every giant segment (>= 2,048 messages of one target) is streamed — products
 *                              materialised by producer CTAs on every SM, add chains fed by bulk copies — instead of
 *                              only those above 1/4 of the call's messages; results are identical either way. */
#define TPN_DEBUG_NO_STREAM 32
#define TPN_DEBUG_STREAM_ALL 64
/*   TPN_DEBUG_LEGACY_PAIRWISE: tpn_pairwise calls of more than 4,096 pairs run the one-shot TMA kernel (each warp
 *                              stages one whole 4-pair tile and exits) instead of the persistent kernel that stages
 *                              tiles in column halves, the next half in flight under the current one's math;
 *                              results are identical. */
#define TPN_DEBUG_LEGACY_PAIRWISE 128
int tpn_set_debug_flags(int flags);


/*
 * Message-level form of tpn_update for a node-sharded state (SURVEY.md §8e; no reference
 * counterpart — the reference is single-device).  Message m adds source row src_dev[m] into
 * target row tgt_dev[m] with the weight of timestamp t_dev[m]; messages of one target are
 * accumulated in the order given.  Ids index rows of `st`: rows [0, num_local_rows) are this
 * shard's rows, rows [num_local_rows, num_nodes) hold copies of other ranks' blocks — they are only
 * ever read and, in lazy mode, carry their own stamps like any row (a copy that was brought current
 * by its sender is stamped with the current epoch).  Precondition (true for edge batches, which carry
 * both directions of every edge): every LOCAL source row is also a target of the same call;
 * in lazy mode a violation sets *err_flag_dev = 2 (eager mode handles it correctly).
 * num_messages_dev: NULL, or a device int32 holding the real number of messages (<= num_messages, which is then
 * only the capacity the grids are sized for) — the count the routing kernels (tpn_route_update) leave on the
 * device, so that no launch waits for a device -> host copy.
 */
int tpn_update_messages(tpn_state_t* st,
                        const int64_t* tgt_dev, const int64_t* src_dev, const double* t_dev, int64_t num_messages,
                        const int32_t* num_messages_dev, int64_t num_local_rows,
                        double t_last, float neg_lambda, const float* decay,
                        void* ws_dev, size_t ws_bytes, int32_t* err_flag_dev, void* stream);

/* Sharded exchange, sender side: out_dev[i] = whole node block (node_stride floats, rows 0..L,
 * brought current in lazy mode) of ids_dev[i] — the payload of the all-to-all. */
int tpn_gather_blocks(const tpn_state_t* st, const int64_t* ids_dev, int64_t n, float* out_dev, void* stream);

/*
 * Input of `self.mlp` in RandomProjectionModule.get_pair_wise_feature —
 * TPNet.py:112-129 without the trainable head (which stays in PyTorch).
 *   a_ids_dev, b_ids_dev : int64[n] device
 *   out_dev              : float32[n][(2L+2)^2] device, row-major (r, c) over the
 *                          rows [a:P_0..P_L, b:P_0..P_L]                (TPNet.py:119-123)
 *   apply_log_scale      : 1 -> clamp at 0 then log(x + 1.0)   (TPNet.py:127-128)
 *                          0 -> raw inner products             (`not_scale`, :124-125)
 *   n_dev                : NULL, or a device int32 with the real number of pairs (<= n; n is then the capacity
 *                          the grid is sized for; rows of out_dev past the count are not written) — routed
 *                          calls of a sharded state (tpn_route_pairs)
 */
int tpn_pairwise(const tpn_state_t* st, const int64_t* a_ids_dev, const int64_t* b_ids_dev, int64_t n,
                 const int32_t* n_dev, int apply_log_scale, float* out_dev, void* stream);

/*
 * The encoder's structured pair-wise call — the index construction and re-split around
 * get_pair_wise_feature at models/TPNet.py:313-324, without the trainable head:
 *   for every row n < m and neighbour k < num_neighbors
 *     out[n][k][0][:] = pair-wise block of (nbr[n][k], src[n])
 *     out[n][k][1][:] = pair-wise block of (nbr[n][k], dst[n])
 *   each block as tpn_pairwise writes it ((2L+2)^2 floats, rows [nbr:P_0..P_L, src|dst:P_0..P_L]).
 * This is the reference's
 *   get_pair_wise_feature(np.tile(nbr.reshape(-1), 2),
 *                         np.concatenate([np.repeat(src, K), np.repeat(dst, K)]))
 * followed by torch.cat([f[:m*K], f[m*K:]], dim=1).reshape(m, K, -1), with `self.mlp` applied
 * by the caller to the [m*K*2, (2L+2)^2] view of `out` (the head acts on each block alone).
 *   nbr_dev          : int64[m][num_neighbors] device (id 0 = padding neighbour: an ordinary row)
 *   src_dev, dst_dev : int64[m] device
 *   out_dev          : float32[m][num_neighbors][2][(2L+2)^2] device, 16-byte aligned
 * Returns TPN_ERR_UNSUPPORTED when one node block does not fit the shared-memory staging
 * (rows wider than ~8,000 floats, i.e. use_matrix on a large graph): call tpn_pairwise instead.
 */
int tpn_pairwise_neighbors(const tpn_state_t* st, const int64_t* nbr_dev, const int64_t* src_dev,
                           const int64_t* dst_dev, int64_t m, int num_neighbors, int apply_log_scale,
                           float* out_dev, void* stream);

/*
 * Forward of the pair-wise head `self.mlp` = Linear(F, 4F) -> ReLU -> Linear(4F, F)
 * (TPNet.py:64-65, applied at :125/:129) for INFERENCE: y = W2 relu(W1 x + b1) + b2, one fused kernel on the
 * tcgen05 tensor cores, the hidden layer never leaves the SM.  fp32-level accuracy without fp32 tensor cores:
 * every operand is split into two fp16 numbers (22 bits, exact power-of-two scaling), three MMAs per product,
 * fp32 accumulators in TMEM (csrc/tpn_head_tc.cu; error vs a float64 head is at the level of an fp32 SGEMM's).  Training keeps the head in
 * PyTorch (autograd); callers use this only when no gradient is required.
 *   x_dev   : float32[n][features] device, 16-byte aligned (the output of tpn_pairwise /
 *             tpn_pairwise_neighbors viewed as [n, F])
 *   w1_dev  : float32[hidden][features] (nn.Linear layout), b1_dev : float32[hidden]
 *   w2_dev  : float32[features][hidden],                    b2_dev : float32[features]
 *   y_dev   : float32[n][features] device, 16-byte aligned
 * Built for the default 3-layer configuration, features = 64 and hidden = 256; any other shape
 * returns TPN_ERR_UNSUPPORTED (the caller applies the head with its own GEMMs).
 * n_dev: NULL, or a device int32 with the real row count (<= n), as in tpn_pairwise.
 */
int tpn_head_forward(const float* x_dev, int64_t n, const int32_t* n_dev, int features, int hidden, const float* w1_dev,
                     const float* b1_dev, const float* w2_dev, const float* b2_dev, float* y_dev, void* stream);

/*
 * RandomProjectionModule.get_random_projections — TPNet.py:101-110.
 *   out_dev : float32[L+1][n][dim] device (layer-major, so out_dev + l*n*dim is the
 *             l-th [n, dim] tensor of the returned list)
 */
int tpn_gather(const tpn_state_t* st, const int64_t* ids_dev, int64_t n, float* out_dev, void* stream);

/*
 * Lazy mode only: apply the pending decay of EVERY row, write it back and set
 * all stamps to the current epoch (used before backup / state_dict / when the
 * log is full; afterwards the caller may reset epoch to 0 with tpn_reset_epoch).
 * No-op in eager mode.
 */
int tpn_materialize(tpn_state_t* st, void* stream);
/* Lazy mode: after tpn_materialize, restart the log (stamps <- 0, epoch <- 0). */
int tpn_reset_epoch(tpn_state_t* st, void* stream);

/* Zero layers 1..L of every node and all stamps; epoch <- 0 (reset_random_projections,
 * TPNet.py:135-136; P_0 is re-drawn by the caller with torch's RNG, TPNet.py:139, or with tpn_init_projection). */
int tpn_clear_walk_layers(tpn_state_t* st, void* stream);

/*
 * P_0 from a counter-based generator (no reference counterpart; the reference draws P_0 with torch's RNG,
 * TPNet.py:58/139).  The value of node u, column c < dim depends only on (seed, draw, u, c), so a sharded state
 * holds the bits of the one-GPU state whatever the world size.  With s = seed, k = draw:
 *   x[0..3] = Philox4x64-10(counter = (c / 4, u, 0, 0), key = (s, k))   (the bijection of numpy's np.random.Philox)
 *   v_i     = ((x_i >> 11) + 0.5) * 2^-53, in f64, the add rounded to nearest (exact below 2^52): uniforms in (0, 1]
 *   Box-Muller in f64 on (v_0, v_1) and (v_2, v_3): r = sqrt(-2 log v_even), theta = 6.283185307179586 * v_odd,
 *             z = (r cos theta, r sin theta) -> the normals of columns 4 (c / 4) + 0..3
 *   stored    = fl32(z * (1 / sqrt(dim))), the scale in f64: N(0, 1/sqrt(d)) as TPNet.py:58 draws it.
 * Every f64 product and sum is rounded on its own (no FMA contraction).  log / sin / cos are not correctly rounded,
 * so another implementation of the definition can differ only where the f64 value lies within a few f64 ulps of
 * an f32 rounding midpoint.
 * Local row j < rows of `st` is node first_node + j * node_step (0, 1 on one GPU; rank, world on a shard, where row
 * j of rank r is node j * world + r).  Only columns [0, dim) of layer 0 of those rows are written (the pad columns
 * of a partial block of 4 get zero); layers 1..L, the node_stride gap and rows >= rows (a shard's cache rows) are
 * not touched.  rows > num_nodes, node_step < 1, first_node < 0 or a node id past INT64_MAX:
 * TPN_ERR_INVALID_ARGUMENT.  No allocation, no synchronisation: capturable in a CUDA graph.
 */
int tpn_init_projection(const tpn_state_t* st, int64_t rows, int64_t first_node, int64_t node_step, uint64_t seed,
                        uint64_t draw, void* stream);

/*
 * Host -> device staging of the per-call id / timestamp arrays (the reference's
 * `torch.from_numpy(ids).to(device)` at TPNet.py:74-77 and the implicit conversion at :109).
 * A stager owns a ring of pinned host slots and device slots on the current device.
 * tpn_stage copies `count` host arrays of 8-byte elements back to back into the next slot,
 * issues ONE cudaMemcpyAsync and returns the device address of each array in dev_out[i]; the
 * addresses stay valid until the ring wraps (`slots` later calls).  With >= 4 slots the copy runs on
 * the stager's own stream and `stream` only waits for its event (work enqueued on `stream`
 * afterwards sees the data): the copy of one call overlaps the kernels of the two calls before it.
 * Consumers must be enqueued on `stream` (or joined into it) before the second-next tpn_stage call.
 *   kinds[i] = TPN_STAGE_RAW      : copied verbatim (float64 timestamps)
 *            = TPN_STAGE_ID_WRAP  : int64 ids, -num_nodes <= id < num_nodes, negatives wrap
 *                                   (what tensor indexing does, TPNet.py:109)
 *            = TPN_STAGE_ID       : int64 ids, 0 <= id < num_nodes (what scatter_add_ accepts, :93-96)
 * Returns TPN_ERR_INDEX if an id is out of range (nothing is launched).
 * tpn_stager_create allocates (once); tpn_stage only re-allocates if a call exceeds slot_bytes.
 */
typedef struct tpn_stager tpn_stager_t;
#define TPN_STAGE_RAW 0
#define TPN_STAGE_ID_WRAP 1
#define TPN_STAGE_ID 2
int tpn_stager_create(tpn_stager_t** out, size_t slot_bytes, int slots);
void tpn_stager_destroy(tpn_stager_t* sg);
int tpn_stage(tpn_stager_t* sg, const void* const* host, const int64_t* elems, const int* kinds, int count,
              int64_t num_nodes, void** dev_out, void* stream);

/*
 * The reference's `recent` historical-neighbour sampler — NeighborSampler.get_historical_neighbors,
 * utils/utils.py:160-224 with sample_neighbor_strategy == 'recent' (SURVEY.md 8(f) N2).
 * Adjacency as one CSR on the device: entries of node u are [offsets[u], offsets[u+1]), stably sorted by
 * time (both directions of every edge, utils/utils.py:248-251).  For query i: the num_neighbors most recent
 * entries of q_nodes[i] with time STRICTLY before q_times[i] (np.searchsorted 'left', :151), written to the
 * back of row i of the outputs; the front is zero-padded (:211-218).
 *   offsets_dev int64[num_nodes+1]; nbr_dev, eid_dev int64[2E]; times_dev float64[2E]
 *   q_nodes_dev int64[n], q_times_dev float64[n]
 *   out_nbr_dev, out_eid_dev int64[n][num_neighbors]; out_times_dev float64[n][num_neighbors]
 */
int tpn_sampler_recent(const int64_t* offsets_dev, const int64_t* nbr_dev, const int64_t* eid_dev,
                       const double* times_dev, int64_t num_nodes, const int64_t* q_nodes_dev,
                       const double* q_times_dev, int64_t n, int num_neighbors, int64_t* out_nbr_dev,
                       int64_t* out_eid_dev, double* out_times_dev, void* stream);

/*
 * Streaming `recent` sampler: the same answers as tpn_sampler_recent over every edge pushed so far, with the
 * edges fed batch by batch in time order and no adjacency of the whole stream (SURVEY.md 8(d): the power-law
 * stream is generated in batches and never materialised).  State is O(num_nodes * capacity) and lives on the device.
 *
 * Per node u two lists of at most `capacity` = C entries (neighbour, edge id, time), oldest first, row-major
 * [num_nodes][C]:
 *   ALL : the last C folded entries of u;
 *   OLD : the last C folded entries of u strictly older than newest[u], the newest folded time of u (-inf: none).
 * The latest pushed batch is PENDING: its 2B directed entries (per edge j: (dst, eid, t) for src, then (src, eid, t)
 * for dst, utils/utils.py:248-251), stably sorted by node.  A push first FOLDS the previous pending batch into the
 * lists, one warp per node with a pending segment and O(C + log B) work per node, then sorts the new batch.
 *
 * A query (u, t) returns the reference's row over all pushed edges when t >= newest[u] (the newest time of u before
 * the latest push) — which TPNet's loop guarantees: it pushes a batch, queries at that batch's times, then pushes the
 * next.  t > newest[u]: the last K of ALL ++ (pending entries of u older than t); t == newest[u]: the last K of OLD;
 * t < newest[u]: not answerable exactly: the row is zero and err_flag gets TPN_STREAM_ERR_PAST.
 *
 * Device-side validation (bits OR-ed into *err_flag, which the caller polls; the offending item is dropped):
 *   TPN_STREAM_ERR_INDEX : a pushed or queried node id outside [0, num_nodes)  (a dropped query gets a zero row)
 *   TPN_STREAM_ERR_ORDER : a pushed time below the previous edge's time (or the previous batch's last time)
 *   TPN_STREAM_ERR_PAST  : a query before newest[u]
 * After a flagged push the answers are unspecified until tpn_stream_sampler_reset.
 * Every table is allocated by the caller; tpn_stream_sampler_reset initialises them (it is the only call that
 * touches every node).  push / query do no work proportional to num_nodes.
 */
#define TPN_STREAM_ERR_INDEX 1
#define TPN_STREAM_ERR_ORDER 2
#define TPN_STREAM_ERR_PAST 4
typedef struct tpn_stream_sampler {
    int64_t   num_nodes;
    int32_t   capacity;     /* C >= 1: entries per list (the largest num_neighbors a query may ask for)      */
    int32_t   reserved0;
    int64_t   max_batch;    /* edges a push may carry: the pending arrays hold 2 * max_batch entries         */
    int64_t*  all_nbr;      /* device [num_nodes][C]   ALL: neighbour ids                                     */
    int64_t*  all_eid;      /* device [num_nodes][C]        edge ids                                          */
    double*   all_t;        /* device [num_nodes][C]        times                                             */
    int64_t*  old_nbr;      /* device [num_nodes][C]   OLD: neighbour ids                                     */
    int64_t*  old_eid;      /* device [num_nodes][C]        edge ids                                          */
    double*   old_t;        /* device [num_nodes][C]        times                                             */
    int32_t*  all_cnt;      /* device [num_nodes]           entries in ALL                                    */
    int32_t*  old_cnt;      /* device [num_nodes]           entries in OLD                                    */
    double*   newest;       /* device [num_nodes]           newest folded time, -inf if none                  */
    uint32_t* pend_node;    /* device [2 * max_batch]  pending entries sorted by node (num_nodes: dropped)    */
    int64_t*  pend_nbr;     /* device [2 * max_batch]                                                         */
    int64_t*  pend_eid;     /* device [2 * max_batch]                                                         */
    double*   pend_t;       /* device [2 * max_batch]                                                         */
    int32_t*  pend_count;   /* device int32[1]: pending entries (2B of the latest push)                       */
    double*   last_time;    /* device double[1]: time of the last pushed edge, -inf if none                   */
    int32_t*  err_flag;     /* device int32[1]: TPN_STREAM_ERR_* bits                                         */
} tpn_stream_sampler_t;

/* Scratch bytes tpn_stream_sampler_push needs for a batch of `batch` edges (the sort's buffers). */
size_t tpn_stream_sampler_workspace_bytes(int64_t batch);
/* All lists empty, newest = -inf, nothing pending, last_time = -inf, err_flag = 0. */
int tpn_stream_sampler_reset(const tpn_stream_sampler_t* s, void* stream);
/* Folds the pending batch, then makes (src_dev[j], dst_dev[j], eid_dev[j], t_dev[j]), j < batch <= max_batch, the
 * pending batch.  Times must be non-decreasing and >= the previous batch's.  batch == 0 does nothing. */
int tpn_stream_sampler_push(const tpn_stream_sampler_t* s, const int64_t* src_dev, const int64_t* dst_dev,
                            const int64_t* eid_dev, const double* t_dev, int64_t batch, void* ws_dev, size_t ws_bytes,
                            void* stream);
/* tpn_sampler_recent's outputs for the edges pushed so far (num_neighbors <= capacity), under the condition above. */
int tpn_stream_sampler_query(const tpn_stream_sampler_t* s, const int64_t* q_nodes_dev, const double* q_times_dev,
                             int64_t n, int num_neighbors, int64_t* out_nbr_dev, int64_t* out_eid_dev,
                             double* out_times_dev, void* stream);

/*
 * Host-side routing plan of the node-sharded state (tpnet_b200/sharded.py; no reference counterpart —
 * the reference is single-device).  Rows of node u live on rank u % world at local row u / world.
 * For `count` work items (first[m], second[m]) — update messages (target, source) or pairs (a, b) —
 * tpn_plan computes, for this planner's rank:
 *   keep[0..n_keep)        : indices m of the items this rank owns (owner(first[m]) == rank), ascending
 *   first_rows[i]          : local row of first[keep[i]]
 *   second_rows[i]         : local row of second[keep[i]], or n_local + receive slot if it is remote;
 *                            remote rows are de-duplicated and numbered by (owner rank, node id) ascending
 *   recv_counts[q]         : remote rows received from rank q (they arrive in that order)
 *   send_rows[0..n_send)   : local rows other ranks need, grouped by destination rank, ascending node id
 *   send_counts[q]         : rows sent to rank q
 * Output arrays hold `count` elements (send/recv_counts: `world`).  Host memory only, no CUDA calls.
 * Returns TPN_ERR_INDEX if an id is outside [0, global_nodes).
 */
typedef struct tpn_planner tpn_planner_t;
int tpn_planner_create(tpn_planner_t** out, int64_t global_nodes, int world, int rank);
void tpn_planner_destroy(tpn_planner_t* p);
int tpn_plan(tpn_planner_t* p, const int64_t* first, const int64_t* second, int64_t count, int64_t n_local,
             int64_t* keep, int64_t* first_rows, int64_t* second_rows, int64_t* n_keep,
             int64_t* send_rows, int64_t* n_send, int64_t* send_counts, int64_t* recv_counts);

/*
 * ---------------------------------------------------------------------------------------------------------
 * Node-sharded state over peer memory (SURVEY.md 8(e); no reference counterpart — the reference is
 * single-device).  Rows of node u live on rank u % world at local row u / world; rows [0, num_local_rows) of a
 * rank's state are its own, rows [num_local_rows, num_local_rows + ext_rows) cache row blocks of other ranks.
 * The batch is replicated on every rank's device.  Per call every rank runs, on its own stream and with no host
 * round trip:  tpn_route_* (which items are mine, which remote rows do I need)  ->  tpn_pull_rows (read them out
 * of the owners' HBM over NVLink: peer pointers)  ->  [tpn_peer_barrier]  ->  tpn_update_messages / tpn_pairwise
 * with the device-side count.  A cached remote row stays valid until the next write to the state: the caller
 * starts a new generation (tpn_shard_new_generation) after every update.
 * Barrier protocol (the caller's duty, tpnet_b200/sharded.py): one tpn_peer_barrier between the last write of a
 * rank and the first pull of its rows by a peer, and one between the last pull of a call and the first write.
 */
#define TPN_SHARD_CTR_NEED 0    /* extension slots handed out in this generation                              */
#define TPN_SHARD_CTR_PREV 1    /* ... before the latest tpn_route_* call (tpn_pull_rows pulls [PREV, NEED))   */
#define TPN_SHARD_CTR_ERROR 2   /* sticky: 1 = id outside the graph, 2 = extension rows exhausted, 3 = a peer
                                   never reached a barrier                                                     */
#define TPN_SHARD_COUNTERS 8
typedef struct tpn_shard {
    int32_t  world, rank;
    int64_t  global_nodes;              /* ids are 0 .. global_nodes-1                                          */
    int64_t  num_local_rows;
    int64_t  ext_rows;                  /* capacity of the remote-row cache                                     */
    const float* const* peer_data;      /* DEVICE array [world]: state buffer of rank q, mapped into this process */
    const int32_t* const* peer_stamps;  /* DEVICE array [world]: stamps of rank q (NULL in eager mode)          */
    uint32_t* const* peer_flags;        /* DEVICE array [world]: barrier words of rank q, uint32[world] each    */
    int32_t* mark;                      /* device int32[global_nodes], zero = not cached (tpn_shard_new_generation) */
    int32_t* counters;                  /* device int32[TPN_SHARD_COUNTERS]                                     */
    int64_t* need_nodes;                /* device int64[ext_rows]: global id cached in each extension row       */
    uint32_t* barrier_seq;              /* device uint32[1]: barriers passed so far (same on every rank)        */
} tpn_shard_t;

size_t tpn_route_workspace_bytes(int64_t items);
/* The 2*batch update messages of the replicated edge batch (the reference's order, TPNet.py:93-96): those whose
 * target this rank owns, in order -> tgt_rows_out / src_rows_out (local row, or num_local_rows + cache slot) /
 * t_out, their number -> *count_out_dev.  Outputs hold 2*batch elements. */
int tpn_route_update(const tpn_shard_t* sh, const int64_t* src_dev, const int64_t* dst_dev, const double* t_dev,
                     int64_t batch, int64_t* tgt_rows_out, int64_t* src_rows_out, double* t_out,
                     int32_t* count_out_dev, void* ws_dev, size_t ws_bytes, void* stream);
/* Pairs (a[i], b[i]) whose first endpoint this rank owns, in order; keep_out[j] = position i of the j-th kept pair
 * (may be NULL).  Outputs hold n elements. */
int tpn_route_pairs(const tpn_shard_t* sh, const int64_t* a_dev, const int64_t* b_dev, int64_t n,
                    int64_t* a_rows_out, int64_t* b_rows_out, int64_t* keep_out, int32_t* count_out_dev,
                    void* ws_dev, size_t ws_bytes, void* stream);
/* Global node ids -> rows of this rank's state: local row id / world if this rank owns the node, otherwise
 * num_local_rows + a cache slot handed out through the mark table (reused if the node is already cached in this
 * generation).  The slots handed out by this call are the ones the next tpn_pull_rows fills.  An id outside
 * [0, global_nodes) sets counters[ERROR] = 1 and maps to row 0; a full cache sets ERROR = 2, as tpn_route_pairs does.
 * Every id gets a row, in order (rows_out_dev holds n elements); n may be 0 (then the next pull fetches nothing). */
int tpn_route_nodes(const tpn_shard_t* sh, const int64_t* ids_dev, int64_t n, int64_t* rows_out_dev, void* stream);
/* Fills the cache slots handed out by the latest tpn_route_* call from the owners' memory (rows and, in lazy
 * mode, their stamps — a cached row is read exactly like a local one). */
int tpn_pull_rows(const tpn_state_t* st, const tpn_shard_t* sh, void* stream);
int tpn_peer_barrier(const tpn_shard_t* sh, void* stream);
int tpn_shard_new_generation(const tpn_shard_t* sh, void* stream);
/* Peer-visible device memory: cudaMalloc'ed (zero-filled) on the current device, exported / opened with CUDA IPC.
 * tpn_ipc_open maps another PROCESS's allocation and enables peer access from the current device. */
int tpn_peer_alloc(void** out, size_t bytes);
int tpn_peer_free(void* p);
int tpn_ipc_export(const void* p, unsigned char* handle64);
int tpn_ipc_open(const unsigned char* handle64, void** out);
int tpn_ipc_close(void* p);

/*
 * ---------------------------------------------------------------------------------------------------------
 * Node-sharded streaming sampler (no reference counterpart — the reference is single-device).  The lists of node u
 * (ALL, OLD, all_cnt, old_cnt, newest; see tpn_stream_sampler_t) live on rank u % world at local row u / world, the
 * state's placement rule; rows [num_local_rows, num_local_rows + ext_rows) of a rank's list tables cache other
 * ranks' lists.  The pushed batch is replicated on every rank and EVERY rank keeps all of it pending (sorted by global
 * id), so a query never needs a remote pending entry; a push folds only the segments of the nodes the rank owns.
 * A query call is routed like the state's node-list calls: tpn_route_nodes on `shard` (own row, or a cache slot of
 * the sampler's own mark table) -> tpn_stream_shard_pull (the new slots' lists, out of the owners' memory) ->
 * tpn_stream_shard_query on the translated rows.  The answers are tpn_stream_sampler_query's, bit for bit.
 * Barrier protocol (the caller's duty, tpn_peer_barrier on `shard`): one barrier between a rank's push (its fold
 * writes its lists) and any peer's next pull, and one between the last pull of a query phase and the next push.
 */
#define TPN_STREAM_PEER_TABLES 9       /* per rank: all_nbr, all_eid, all_t, old_nbr, old_eid, old_t, all_cnt, old_cnt, newest */
typedef struct tpn_stream_shard {
    tpn_stream_sampler_t local;        /* this rank's sampler: num_nodes = the GLOBAL node count (ids, pending keys);
                                          the list tables hold shard.num_local_rows + shard.ext_rows rows          */
    tpn_shard_t shard;                 /* world, rank, global_nodes (== local.num_nodes, < 2^31), num_local_rows, ext_rows
                                          (cache rows), and the sampler's OWN mark table, counters, need_nodes,
                                          peer_flags and barrier_seq; peer_data / peer_stamps are not used           */
    const void* const* peer_lists;     /* DEVICE array [world][TPN_STREAM_PEER_TABLES]: rank q's list tables, mapped
                                          into this process, in the order of TPN_STREAM_PEER_TABLES                 */
} tpn_stream_shard_t;

/* Every owned and cached row empty, nothing pending, last_time = -inf, err_flag = 0, a new generation of the cache
 * with every shard counter (the error one too) zero. */
int tpn_stream_shard_reset(const tpn_stream_shard_t* s, void* stream);
/* A new cache generation, then tpn_stream_sampler_push of the replicated batch with the fold restricted to the nodes
 * this rank owns (global ids; workspace: tpn_stream_sampler_workspace_bytes). */
int tpn_stream_shard_push(const tpn_stream_shard_t* s, const int64_t* src_dev, const int64_t* dst_dev,
                          const int64_t* eid_dev, const double* t_dev, int64_t batch, void* ws_dev, size_t ws_bytes,
                          void* stream);
/* Fills the cache slots handed out by the latest tpn_route_nodes on s->shard: newest, counts and the first count
 * entries of ALL and OLD of each slot's node, read out of its owner's tables (one warp per slot). */
int tpn_stream_shard_pull(const tpn_stream_shard_t* s, void* stream);
/* tpn_stream_sampler_query for the global ids q_nodes_dev[i], reading the lists at row q_rows_dev[i] (the rows
 * tpn_route_nodes returned: local or cache slot); the pending search uses the global id. */
int tpn_stream_shard_query(const tpn_stream_shard_t* s, const int64_t* q_nodes_dev, const int64_t* q_rows_dev,
                           const double* q_times_dev, int64_t n, int num_neighbors, int64_t* out_nbr_dev,
                           int64_t* out_eid_dev, double* out_times_dev, void* stream);

/*
 * ---------------------------------------------------------------------------------------------------------
 * Negative edge sampler on the device: DyGLib's NegativeEdgeSampler (the reference's utils/utils.py:315-505) with
 * its three strategies, drawn from a counter-based generator instead of numpy's MT19937 — the same sets, sizes and
 * ordering rule, not the same draws.  S, D = sorted unique src / dst ids; W(a, b) = the distinct (src, dst) of the
 * edges with a <= t <= b; f(key) = the first time of an edge.
 * Tables (tpn_neg_sampler_build; node ids < 2^id_bits <= 2^32, edge keys are two uint32 words):
 *   T : the edges stably sorted by time (t_src, t_dst, t_time) and, per edge, t_fpos = the F position of its key;
 *       a window [s, e] is the range [#{t < s}, #{t <= e}) of T.
 *   F : the distinct keys sorted by (f, src, dst) (f_src, f_dst, f_time): W(min t, s) is the prefix F[0, #{f <= s}).
 *   S, D.
 * A call (tpn_neg_sampler_sample, s = start, e = end, c = call index, key = (seed, c)):
 *   random     : out[i] = (S[hi64(x0 * |S|)], D[hi64(x1 * |D|)]), x = Philox4x64-10((i, 0, 4, 0), key).
 *   historical : domain F[0, h), h = #{f <= s};  inductive: F[o, max(o, h)), o = #{f <= last_observed_time}.
 *                Hc = domain minus W(s, e);  k = min(size, |Hc|): the first k elements of a keyed permutation of the
 *                domain (tag 1) that are not in W(s, e), in permutation order.
 *                If size > |Hc|: first the fill, then all of Hc.  Fill = size - |Hc| elements of
 *                U = S x D minus the batch's pairs, pair index q = i_S * |D| + i_D: the first of a permutation of
 *                [0, |S||D|) (tag 2) outside the batch; when |U| < fill: out[j] = U[hi64(x0 * |U|)] over U in index
 *                order, x = Philox((j, 0, 3, 0), key).  |U| == 0 sets TPN_NEG_ERR_EMPTY (the reference asserts) and
 *                writes -1.
 *   Permutation of [0, n): a balanced 4-round Feistel network on m bits (m the smallest even number >= 2 with
 *   2^m >= n), round r: (L, R) -> (R, L ^ (Philox((R, r, tag, 0), key).x0 mod 2^(m/2))), cycle-walking until < n.
 * Everything is integer arithmetic and exact f64 comparisons: the output depends only on (seed, c, inputs), not on
 * the grid or the device.  Every call is asynchronous, allocation-free and, with start_dev / end_dev, capturable.
 */
#define TPN_NEG_RANDOM 0
#define TPN_NEG_HISTORICAL 1
#define TPN_NEG_INDUCTIVE 2
#define TPN_NEG_ERR_EMPTY 1            /* a fill found S x D entirely inside the batch                             */
#define TPN_NEG_COUNTS 4               /* counts: [0] distinct keys, [1] |S|, [2] |D|, [3] TPN_NEG_ERR_* bits (sticky) */
typedef struct tpn_neg_sampler {
    int64_t   num_edges;               /* E, 1 .. 2^31 - 2^12                                                     */
    int32_t   id_bits;                 /* every node id < 2^id_bits, 1..32 (sets the radix passes)               */
    int32_t   timed;                   /* 1: T, F and mark are built (historical / inductive); 0: S and D only   */
    uint64_t  seed;
    double    last_observed_time;      /* inductive: observed = the keys with f <= this                          */
    uint32_t* t_src;                   /* device [E]                                                              */
    uint32_t* t_dst;                   /* device [E]                                                              */
    double*   t_time;                  /* device [E]                                                              */
    uint32_t* t_fpos;                  /* device [E]                                                              */
    uint32_t* f_src;                   /* device [E] (the first counts[0] are used)                               */
    uint32_t* f_dst;                   /* device [E]                                                              */
    double*   f_time;                  /* device [E]                                                              */
    uint32_t* mark;                    /* device [E], zero between calls                                          */
    uint32_t* uniq_src;                /* device [min(E, 2^id_bits)]: S                                           */
    uint32_t* uniq_dst;                /* device [min(E, 2^id_bits)]: D                                           */
    int32_t*  counts;                  /* device int32[TPN_NEG_COUNTS]                                            */
} tpn_neg_sampler_t;

/* Scratch bytes of a build of num_edges edges (0: none) and of a call of `size` negatives with a batch of `batch`
 * edges (0: none); the larger of the two. */
size_t tpn_neg_sampler_workspace_bytes(int64_t num_edges, int64_t size, int64_t batch);
/* Builds S, D and (timed) T and F from src_dev / dst_dev int64[E] and t_dev float64[E] (not sorted; t_dev may be
 * NULL when !timed), zeroes mark and the error bits.  Ids must lie in [0, 2^id_bits) and times must not be NaN (the
 * caller checks both). */
int tpn_neg_sampler_build(const tpn_neg_sampler_t* s, const int64_t* src_dev, const int64_t* dst_dev,
                          const double* t_dev, void* ws_dev, size_t ws_bytes, void* stream);
/* One `sample` call: out_src_dev / out_dst_dev int64[size].  batch_src_dev / batch_dst_dev int64[batch] (any ids; ids
 * outside S or D exclude nothing).  start_dev / end_dev: NULL (use start / end) or device doubles read by the kernels. */
int tpn_neg_sampler_sample(const tpn_neg_sampler_t* s, int strategy, uint64_t call, int64_t size,
                           const int64_t* batch_src_dev, const int64_t* batch_dst_dev, int64_t batch, double start,
                           double end, const double* start_dev, const double* end_dev, int64_t* out_src_dev,
                           int64_t* out_dst_dev, void* ws_dev, size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TPNET_B200_H_ */

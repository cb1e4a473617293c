// tpn_update — RandomProjectionModule.update (reference: models/TPNet.py:67-99) for sm_100a.
//
// Pipeline of one call (all on the caller's stream, no host sync):
//   1. prep      : w_j = exp(f32(-lambda) * (f32(t_last) - f32(t_j)))            (TPNet.py:77-78)
//                  2B messages  m <  B : target src[m], source dst[m]            (first scatter_add_, :93)
//                               m >= B : target dst[m-B], source src[m-B]        (second scatter_add_, :95)
//                  lazy mode: append c_1..c_L to the decay log as a new epoch.
//   2. sort      : stable sort of the messages by target id, so that each target's
//                  messages are contiguous and in the reference's accumulation order
//                  (batch order within the src role, then the dst role).
//                    2B <= 1024 : one CTA, rank sort in shared memory (one barrier)
//                    2B <= 4096 : one CTA, bitonic network on (target << 32 | m)
//                    larger     : LSD radix sort, 8-bit digits, two launches per pass (block
//                                 histograms; scatter with in-kernel offsets + warp-match
//                                 ranking); integer atomics only on histogram counts.
//   3. sweep     : eager mode only — P_l *= c_l over the whole state          (TPNet.py:83-85).
//                  For 2B <= 4096 it runs in the SAME launch as prep (block 0 sorts while
//                  the other blocks sweep).
//   4. walk      : each target row is owned by one group of lanes: read once, pending decay
//                  replayed (lazy), messages added one at a time in order as
//                  fadd_rn(acc, fmul_rn(source, w)), written once.  128-bit accesses, several
//                  source rows in flight per group.  No float atomics anywhere.
//                  Layer i must read the PRE-batch layer i-1 (TPNet.py:90 goes top-down):
//                    2B <= kSnapMaxMsgs : the pre-batch rows 1..L-1 of the batch's nodes are
//                        copied to a snapshot (every source node is also a target), then ONE
//                        launch updates all layers, reading layer 0 from the state and
//                        layers >= 1 from the snapshot;
//                    larger : one launch per layer, top-down (no extra traffic).
#include <stdlib.h>

#include "tpn_common.cuh"
#include "tpn_radix.cuh"

namespace tpn {

namespace {

int g_debug_flags = 0;
thread_local int g_dev_slot = 0;         // device of the call in progress (set by the entry point)

constexpr int kSmallMaxMsgs = 4096;      // 2B <= 4096 -> single-CTA sort
constexpr int kRankMaxMsgs = 1024;       // 2B <= 1024 -> rank sort (one barrier) instead of the bitonic network
constexpr int kPrepThreads = 1024;
constexpr int kWalkThreads = 256;
// CTA-pipelined walker for long segments (hubs)
constexpr int kHubMin = 64;              // segments at least this long leave the warp walker
constexpr int kGiantMin = 2048;          // ... and these are scheduled first
constexpr int kHubConsumers = 4;         // consumer warps (one per SM sub-partition), 1 float per lane
constexpr int kHubThreads = (kHubConsumers + 1) * 32;      // + 1 producer warp
constexpr int kHubStages = 4;            // ring stages of 32 messages
constexpr int kHubSlotFloats = kHubConsumers * 32;         // 128 floats (512 B) per message slot
constexpr int kHubMetaChunk = 512;       // messages of metadata staged per bulk copy
constexpr int kChunkMin = 256;           // smallest chunk of the chunked accumulation order (tpn_state_t::giant_chunk)
constexpr size_t kSnapMaxBytes = (size_t)8 << 30;          // 8 GiB: above this the per-layer path is used (its hub
                                                           // walker is 10x slower on giant segments: 33 ms vs ~3 ms for
                                                           // d=1024, L=3, 100k zipf(1.5) edges)
// large batches, snapshot path: short segments -> persistent warp walker, long ones -> hub2
constexpr int kSmallWalkThreads = 256;
constexpr int kHub2Producers = 7;        // producer warps: each keeps one ring stage (32 messages) of loads in flight
constexpr int kHub2Threads = (1 + kHub2Producers) * 32;    // + the consumer warp (warp 0)
constexpr int kHub2SlotFloats = 64;      // floats of one message held by a ring slot (consumer: 2 columns per lane)
#ifndef TPN_HUB2_GIANT_FLOATS
#define TPN_HUB2_GIANT_FLOATS 16         // A/B builds: -DTPN_HUB2_GIANT_FLOATS=32 (128-byte slices: full cache lines,
#endif                                   // half the work items; scripts/micro/gather_paths.cu says same message rate)
constexpr int kHub2GiantFloats = TPN_HUB2_GIANT_FLOATS;     // slice width of giant segments: an SM sustains ~10 B/clk of row gathers
                                         // (outstanding-miss capacity), so 64 B per message keeps its data path
                                         // near the add chain's 4-6 cycles per message
static_assert(kHub2GiantFloats == 8 || kHub2GiantFloats == 16 || kHub2GiantFloats == 32, "giant slices are 32, 64 or 128 bytes");
constexpr int kGiantLs = kHub2GiantFloats == 8 ? 1 : (kHub2GiantFloats == 16 ? 2 : 3);   // log2(lanes per giant message): 2, 4 or 8 lanes of 16 bytes
constexpr int kGiantSpm = 16 >> kGiantLs;                  // 32-message sub-blocks per ring stage: 8, 4 or 2
constexpr int kGiantSpmMax = kGiantSpm > 4 ? kGiantSpm : 4;
constexpr int kHub2Stages = kHub2Producers + 4;            // ring stages of 32 messages (8 KB each)
// ctr[] slots (zeroed by prep_large_kernel)
constexpr int kCtrGiant = 0, kCtrHub = 1, kCtrWork0 = 2, kCtrSmall = 6, kCtrHub2Work = 7, kCtrHub2Giant = 8;
constexpr int kCtrChunks = 9;            // chunked accumulation: partial-sum rows handed out so far
// streamed giants (walk_hub2_kernel): the first ctr[kCtrStream] entries of the (sorted) giant list have their message
// products materialised by producer CTAs and their add chains fed from that stream by bulk copies
constexpr int kCtrStream = 10, kCtrStreamBlocks = 11, kCtrStreamProd = 12, kCtrStreamActive = 13, kCtrStreamChain = 14, kCtrStreamTicket = 15;
constexpr int kStreamSlice = kHub2GiantFloats;      // floats between messages of a slice chunk: a giant's ring-stage layout
constexpr int kStreamBlock = 32 * kGiantSpm;        // messages per production block (one flag; one 8 KB bulk copy per slice)
constexpr uint32_t kNoPart = 0xffffffffu;   // hub_part[e]: the entry accumulates straight into its target row
constexpr int kCtrSmClaim = 16;          // [256] first hub2 CTA of each SM claims the SM's giant-segment slot
constexpr int kCtrSlots = kCtrSmClaim + 256;
constexpr int kBarWords = 32;            // [0]: arrivals of the fused front end's grid barrier (monotonic within a launch)

struct DecayArgs {
    float c[TPN_MAX_LAYERS];
    int has_decay;
};

// Snapshot-slot encoding (sslot): sorted position of the head of the source node's own segment, or
// kDirect: the source is not a target of this call, so its rows are not written by it and are
// read straight from the state (received rows of a sharded state; never happens in edge mode).
constexpr uint32_t kDirect = 0x80000000u;

// Where the messages come from.  Edge mode (B > 0): message m < B has target a[m] = src and
// source b[m] = dst, message m >= B the reverse (the two scatter_add_ of TPNet.py:93-96), both
// weighted by the edge's timestamp t[m mod B].  Message mode (B == 0, sharded state): message m
// has target a[m], source b[m] and timestamp t[m]; the given order is the accumulation order.
struct MsgSource {
    const long long* a;
    const long long* b;
    const double* t;
    long long B;
    long long direct_from;   // source rows >= this are read-only and current (received rows of a sharded state)
    __device__ __forceinline__ void get(int m, long long& tgt, long long& oth, int& widx) const {
        if (B > 0) {
            const int j = m < B ? m : (int)(m - B);
            tgt = m < B ? a[j] : b[j];
            oth = m < B ? b[j] : a[j];
            widx = j;
        } else {
            tgt = a[m];
            oth = b[m];
            widx = m;
        }
    }
};

struct Workspace {
    float* w;          // [B]
    uint32_t* key_a;   // [E]
    uint32_t* key_b;   // [E]
    uint32_t* val_a;   // [E]
    uint32_t* val_b;   // [E]
    uint32_t* ssrc;    // [E] source node of the p-th sorted message
    float* sw;         // [E] weight of the p-th sorted message
    uint32_t* hist;    // [256 * (nblk + 1)]
    uint32_t* hist2;   // [256 * (nblk + 1)] fused front end: histogram of the NEXT pass, counted while scattering
    uint32_t* bar;     // [kBarWords] grid barrier of the fused front end (zeroed by a memset node before the launch)
    uint32_t* sslot;   // [E] sorted position of the segment head of the p-th message's SOURCE node
    uint32_t* slen;    // [E] number of messages with the same target as the p-th sorted message
    float* snap;       // [E][(L-1)*row_stride] pre-batch rows 1..L-1 of each target (snapshot path only)
    uint32_t* hub_giant;   // [E / kGiantMin + 2] sorted positions of the heads of giant segments
    uint32_t* hub_reg;     // [E / kHubMin + 2]   ... of the other long segments
    uint32_t* ctr;         // [kCtrSlots] 0: #giant, 1: #regular, 2..5: work counters of the per-layer hub launches,
                           //     6: #short segments, 7/8: work counters of the hub2 launch, 16..: SM claims
    uint32_t* small_heads; // [E] sorted positions of the heads of short segments (scheduling order only)
    uint32_t* hub_len;     // [hub_cap] messages of the e-th entry of hub_reg (a whole segment, or one chunk of a giant)
    uint32_t* hub_part;    // [hub_cap] kNoPart, or the partial-sum row the entry accumulates into (chunked giants)
    uint32_t* giant_cbase; // [E / kGiantMin + 2] first partial-sum row of the i-th giant (chunked accumulation)
    float* partial;        // [E / kChunkMin + E / kGiantMin + 2][L*row_stride] partial sums of giant chunks
    int* svst;             // [L-1][E] pre-batch stamp of the source row of each sorted message (lazy, per-layer path)
    float* gprod;          // [E][nslice * 32] products fmul_rn(source, w) of the messages of streamed giants, per block
                           //     of 128 messages slice-major: [slice][message][32 columns]
    uint32_t* gflag;       // [E / 128 + E / kGiantMin + 2] block q of the streamed giants has been produced (zeroed per call
                           //     by sort_giants_kernel)
    uint32_t* gblk;        // [kGiantSortMax + 1] first block of the i-th giant of the sorted list (prefix sum)
    bool has_snap;
    bool has_stream;       // the product buffer of the streamed giants fits (and the giant list can always be ordered)
    size_t bytes;
};

inline size_t snap_bytes(size_t E, int num_layer, int64_t row_stride) {
    // rows 1..L-1 of every target (rows 0..L-1 with TPN_DEBUG_SNAPSHOT_P0): sized for the larger of the two
    return sizeof(float) * E * (size_t)num_layer * (size_t)row_stride;
}

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

constexpr size_t kStreamMaxBytes = (size_t)4 << 30;      // product buffer of the streamed giants: above this, hub walker
constexpr int kGiantSortMaxC = 2048;     // giants ordered (and streamed) per call; more than this: unordered, hub walker
inline int stream_slices(int num_layer, int64_t row_stride) {           // = L * spr_g of launch_walk_hub2
    return num_layer * (int)((row_stride + kStreamSlice - 1) / kStreamSlice);
}
inline size_t stream_prod_bytes(size_t E, int num_layer, int64_t row_stride) {
    return sizeof(float) * E * (size_t)stream_slices(num_layer, row_stride) * kStreamSlice + 256;
}
inline size_t stream_flag_words(size_t E) { return E / kStreamBlock + E / kGiantMin + 4; }

Workspace carve(void* base, int64_t batch, int num_layer, int64_t row_stride) {
    const size_t E = 2 * (size_t)batch;
    const size_t nblk = (E + kRadixTile - 1) / kRadixTile;
    char* p = reinterpret_cast<char*>(base);
    size_t off = 0;
    Workspace ws;
    auto take = [&](size_t bytes) { char* r = p ? p + off : nullptr; off += align_up(bytes, 256); return r; };
    ws.w = reinterpret_cast<float*>(take(sizeof(float) * E));
    ws.key_a = reinterpret_cast<uint32_t*>(take(4 * E));
    ws.key_b = reinterpret_cast<uint32_t*>(take(4 * E));
    ws.val_a = reinterpret_cast<uint32_t*>(take(4 * E));
    ws.val_b = reinterpret_cast<uint32_t*>(take(4 * E));
    ws.ssrc = reinterpret_cast<uint32_t*>(take(4 * E));
    ws.sw = reinterpret_cast<float*>(take(4 * E));
    ws.hist = reinterpret_cast<uint32_t*>(take(4 * kRadixBins * (nblk + 1)));
    ws.hist2 = reinterpret_cast<uint32_t*>(take(4 * kRadixBins * (nblk + 1)));
    ws.bar = reinterpret_cast<uint32_t*>(take(4 * kBarWords));
    ws.sslot = reinterpret_cast<uint32_t*>(take(4 * E));
    ws.slen = reinterpret_cast<uint32_t*>(take(4 * E));
    ws.has_snap = snap_bytes(E, num_layer, row_stride) <= kSnapMaxBytes;
    ws.snap = reinterpret_cast<float*>(take((ws.has_snap ? snap_bytes(E, num_layer, row_stride) : 0) + 16));
    ws.hub_giant = reinterpret_cast<uint32_t*>(take(4 * (E / kGiantMin + 2)));
    // hub_reg also holds the chunks of giants in chunked mode: <= E / kChunkMin + one ragged chunk per giant
    const size_t hub_cap = E / kHubMin + E / kChunkMin + E / kGiantMin + 4;
    const size_t part_rows = E / kChunkMin + E / kGiantMin + 2;
    ws.hub_reg = reinterpret_cast<uint32_t*>(take(4 * hub_cap));
    ws.hub_len = reinterpret_cast<uint32_t*>(take(4 * hub_cap));
    ws.hub_part = reinterpret_cast<uint32_t*>(take(4 * hub_cap));
    ws.giant_cbase = reinterpret_cast<uint32_t*>(take(4 * (E / kGiantMin + 2)));
    ws.partial = reinterpret_cast<float*>(take(ws.has_snap ? 4 * part_rows * (size_t)num_layer * (size_t)row_stride : 16));
    ws.ctr = reinterpret_cast<uint32_t*>(take(4 * kCtrSlots));
    ws.small_heads = reinterpret_cast<uint32_t*>(take(4 * E));
    ws.svst = reinterpret_cast<int*>(take(4 * (E + 4) * (size_t)(num_layer > 1 ? num_layer - 1 : 1) + 16));
    ws.gflag = reinterpret_cast<uint32_t*>(take(4 * stream_flag_words(E)));
    ws.gblk = reinterpret_cast<uint32_t*>(take(4 * (kGiantSortMaxC + 1)));
    ws.has_stream = ws.has_snap && stream_prod_bytes(E, num_layer, row_stride) <= kStreamMaxBytes &&
                    E / kGiantMin + 2 <= (size_t)kGiantSortMaxC;
    ws.gprod = reinterpret_cast<float*>(take(ws.has_stream ? stream_prod_bytes(E, num_layer, row_stride) : 16));
    ws.bytes = off;
    return ws;
}

__device__ __forceinline__ float edge_weight(double t, float t_last_f, float neg_lambda) {
    // fp32 subtract of the fp32-cast timestamps, fp32 multiply, then exp.  exp is
    // evaluated in f64 and rounded once (torch's CPU exp is a 1-ulp fp32 routine;
    // the correctly rounded value is the closest reproducible target).
    const float diff = __fsub_rn(t_last_f, (float)t);
    const float arg = __fmul_rn(neg_lambda, diff);
    return (float)exp((double)arg);
}

// ---------------------------------------------------------------- small path
// Block 0: weights + stable sort + sorted payload (+ decay-log append).  Blocks >= 1 (eager
// mode with a clock move only): the whole-state decay sweep, overlapped with the sort.
struct SweepArgs {
    long long total4;      // float4 to scale (0 = no sweep)
    int ds4;
};

__device__ __forceinline__ void sweep_body(const StateView& st, const DecayArgs& decay, long long total4, int ds4,
                                           long long first, long long stride) {
    // layers 1..L of a node are contiguous right after its layer-0 row
    const long long per_node4 = (long long)st.num_layer * ds4;
    for (long long i = first; i < total4; i += stride) {
        const long long node = i / per_node4;
        const int r = (int)(i - node * per_node4);
        const int li = r / ds4;
        float* p = st.data + node * st.node_stride + st.row_stride + (long long)r * 4;
        float4 x = ld4(p);
        scale4(x, decay.c[li]);
        st4(p, x);
    }
}

__global__ void __launch_bounds__(kPrepThreads)
prep_small_kernel(MsgSource msgs, int E, float t_last_f, float neg_lambda, long long num_nodes,
                  uint32_t* __restrict__ skey, uint32_t* __restrict__ ssrc, float* __restrict__ sw,
                  uint32_t* __restrict__ sslot, uint32_t* __restrict__ slen, int* __restrict__ err_flag,
                  double* decay_log, int L, long long new_epoch, DecayArgs decay, StateView st, SweepArgs sweep) {
    if (blockIdx.x > 0) {
        sweep_body(st, decay, sweep.total4, sweep.ds4, (long long)(blockIdx.x - 1) * kPrepThreads + threadIdx.x,
                   (long long)(gridDim.x - 1) * kPrepThreads);
        return;
    }
    __shared__ __align__(16) unsigned long long comp[kSmallMaxMsgs];   // (target << 32 | message index)
    __shared__ float wsm[kSmallMaxMsgs];
    const int n_w = msgs.B > 0 ? (int)msgs.B : E;             // distinct weights (per edge / per message)
    const bool message_mode = msgs.B == 0;
    const bool lazy = decay_log != nullptr;
    if (threadIdx.x == 0 && decay_log != nullptr && decay.has_decay) {
        for (int l = 0; l < L; ++l) decay_log[new_epoch * L + l] = decay_log[(new_epoch - 1) * L + l] * (double)decay.c[l];
    }
    if (E <= kRankMaxMsgs) {
        // ---- rank sort.  Keys are packed as (target << 10 | m) in 32 bits when the node ids
        // allow it (num_nodes < 2^22), else as 64-bit composites.  Composites are unique, so
        // "number of composites smaller than mine" IS the stable sorted position.  The same
        // scan gives, for the message's SOURCE node, where that node's own segment starts
        // (every source is also a target) and, for the target, the segment length.
        uint32_t* c32 = reinterpret_cast<uint32_t*>(comp);
        const bool narrow = num_nodes < (1ll << 22);
        const int Epad = (E + 3) & ~3;
        for (int m = threadIdx.x; m < Epad; m += kPrepThreads) {
            uint32_t key = 0xffffffffu >> 10;                 // padding: above every real key
            if (m < E) {
                long long tgt, oth;
                int widx;
                msgs.get(m, tgt, oth, widx);
                const bool ok = tgt >= 0 && tgt < num_nodes && oth >= 0 && oth < num_nodes;
                if (!ok && err_flag != nullptr) *err_flag = 1;
                key = ok ? (uint32_t)tgt : (uint32_t)num_nodes;   // sentinel: dropped by walk
                if (m < n_w) wsm[m] = edge_weight(msgs.t[m], t_last_f, neg_lambda);
            }
            if (narrow) c32[m] = (key << 10) | (uint32_t)m;
            else comp[m] = ((unsigned long long)(m < E ? key : 0xffffffffu) << 32) | (uint32_t)m;
        }
        __syncthreads();
        for (int m = threadIdx.x; m < E; m += kPrepThreads) {
            long long tgt_unused, oth;
            int j;
            msgs.get(m, tgt_unused, oth, j);
            const uint32_t other = (uint32_t)oth;
            int rank = 0, slot = 0, upper = 0, slot_hi = 0;
            uint32_t mykey;
            if (narrow) {
                const uint32_t mine = c32[m];
                mykey = mine >> 10;
                const uint32_t other_lo = other << 10, next_lo = (mykey + 1) << 10, other_hi = (other + 1) << 10;
                const uint4* c4 = reinterpret_cast<const uint4*>(c32);
                for (int i = 0; i < Epad / 4; ++i) {
                    const uint4 c = c4[i];                    // same address across the warp: broadcast
                    rank += (c.x < mine) + (c.y < mine) + (c.z < mine) + (c.w < mine);
                    slot += (c.x < other_lo) + (c.y < other_lo) + (c.z < other_lo) + (c.w < other_lo);
                    upper += (c.x < next_lo) + (c.y < next_lo) + (c.z < next_lo) + (c.w < next_lo);
                    if (message_mode)
                        slot_hi += (c.x < other_hi) + (c.y < other_hi) + (c.z < other_hi) + (c.w < other_hi);
                }
            } else {
                const unsigned long long mine = comp[m];
                mykey = (uint32_t)(mine >> 32);
                const unsigned long long other_lo = (unsigned long long)other << 32;
                const unsigned long long other_hi = (unsigned long long)(other + 1) << 32;
                const unsigned long long next_lo = (unsigned long long)(mykey + 1) << 32;
                for (int i = 0; i < E; ++i) {
                    const unsigned long long c = comp[i];
                    rank += c < mine;
                    slot += c < other_lo;
                    upper += c < next_lo;
                    slot_hi += c < other_hi;
                }
            }
            if (message_mode && slot_hi == slot) {            // the source is not a target of this call
                if (lazy && (long long)other < msgs.direct_from && err_flag != nullptr) *err_flag = 2;
                slot = (int)kDirect;
            }
            const int lower = rank - 0;      // rank counts everything below (key, m); the head is the lower bound
            skey[rank] = mykey;
            ssrc[rank] = other;
            sw[rank] = wsm[j];
            sslot[rank] = (uint32_t)slot;
            slen[rank] = (uint32_t)(upper - lower);          // at the head (lower == rank) this is the segment length
        }
        return;
    }
    // ---- bitonic network on the composite (target, message index): total order == stable order
    int P = 1;
    while (P < E) P <<= 1;
    for (int m = threadIdx.x; m < P; m += kPrepThreads) {
        unsigned long long c = ~0ull;                         // padding sorts last
        if (m < E) {
            long long tgt, oth;
            int widx;
            msgs.get(m, tgt, oth, widx);
            const bool ok = tgt >= 0 && tgt < num_nodes && oth >= 0 && oth < num_nodes;
            if (!ok && err_flag != nullptr) *err_flag = 1;
            const uint32_t key = ok ? (uint32_t)tgt : (uint32_t)num_nodes;
            c = ((unsigned long long)key << 32) | (uint32_t)m;
            if (m < n_w) wsm[m] = edge_weight(msgs.t[m], t_last_f, neg_lambda);
        }
        comp[m] = c;
    }
    __syncthreads();
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < P; i += kPrepThreads) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long a = comp[i], b = comp[ixj];
                    const bool up = (i & k) == 0;
                    if ((a > b) == up) { comp[i] = b; comp[ixj] = a; }
                }
            }
            __syncthreads();
        }
    }
    for (int p = threadIdx.x; p < E; p += kPrepThreads) {
        const unsigned long long c = comp[p];
        const uint32_t m = (uint32_t)c;
        const uint32_t mykey = (uint32_t)(c >> 32);
        long long tgt_unused, oth;
        int j;
        msgs.get((int)m, tgt_unused, oth, j);
        const uint32_t other = (uint32_t)oth;
        skey[p] = mykey;
        ssrc[p] = other;
        sw[p] = wsm[j];
        // lower bound of the source id among the sorted targets; end of my own segment
        const unsigned long long other_lo = (unsigned long long)other << 32;
        const unsigned long long next_lo = (unsigned long long)(mykey + 1) << 32;
        int lo = 0, hi = E;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (comp[mid] < other_lo) lo = mid + 1; else hi = mid;
        }
        uint32_t slot = (uint32_t)lo;
        if (message_mode && (lo >= E || (uint32_t)(comp[lo] >> 32) != other)) {
            if (lazy && (long long)other < msgs.direct_from && err_flag != nullptr) *err_flag = 2;
            slot = kDirect;
        }
        sslot[p] = slot;
        lo = p; hi = E;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (comp[mid] < next_lo) lo = mid + 1; else hi = mid;
        }
        slen[p] = (uint32_t)(lo - p);                         // messages from p to the end of the segment
    }
}

// ---------------------------------------------------------------- large path
struct PrepArgs {
    MsgSource msgs;
    Count count;
    float t_last_f, neg_lambda;
    long long num_nodes;
    float* w;
    uint32_t* key;
    uint32_t* val;
    int* err_flag;
    double* decay_log;
    int L;
    long long new_epoch;
    DecayArgs decay;
    uint32_t* ctr;
};

__device__ __forceinline__ void prep_body(const PrepArgs& a, int m) {
    if (m == 0 && a.decay_log != nullptr && a.decay.has_decay) {
        for (int l = 0; l < a.L; ++l)
            a.decay_log[a.new_epoch * a.L + l] = a.decay_log[(a.new_epoch - 1) * a.L + l] * (double)a.decay.c[l];
    }
    if (m < kCtrSlots) a.ctr[m] = 0;                     // hub lists, work counters and SM claims of this call
    // a device-side count above the capacity this call was sized for: the excess is dropped, and flagged
    if (m == 0 && a.count.dev != nullptr && *a.count.dev > a.count.cap && a.err_flag != nullptr) *a.err_flag = 4;
    const int E = a.count.get();
    if (m >= E) return;
    long long tgt, oth;
    int widx;
    a.msgs.get(m, tgt, oth, widx);
    const bool ok = tgt >= 0 && tgt < a.num_nodes && oth >= 0 && oth < a.num_nodes;
    if (!ok && a.err_flag != nullptr) *a.err_flag = 1;
    const int n_w = a.msgs.B > 0 ? (int)a.msgs.B : E;
    if (m < n_w) a.w[m] = edge_weight(a.msgs.t[m], a.t_last_f, a.neg_lambda);
    a.key[m] = ok ? (uint32_t)tgt : (uint32_t)a.num_nodes;
    a.val[m] = (uint32_t)m;
}

__global__ void __launch_bounds__(256) prep_large_kernel(PrepArgs a) {
    prep_body(a, blockIdx.x * blockDim.x + threadIdx.x);
}

struct PayloadArgs {
    const uint32_t* order;     // sorted message ids
    const uint32_t* skey;      // sorted targets (where the sort left them)
    uint32_t* key_out;         // != skey: the sorted targets are also copied here (odd number of passes)
    MsgSource msgs;
    const float* w;
    Count count;
    uint32_t* ssrc;
    float* sw;
    uint32_t* sslot;
    uint32_t* slen;
    uint32_t* hub_giant;
    uint32_t* hub_reg;
    uint32_t* small_heads;
    uint32_t* ctr;
    int* svst;
    const int* stamps;
    int L, E4;
    long long num_nodes;
    int* err_flag;
    uint32_t* hub_len;
    uint32_t* hub_part;
    uint32_t* giant_cbase;
    int chunk;                 // > 0: chunked accumulation order for giant segments (tpn_state_t::giant_chunk)
};

// sorted position p (whole warps call it together: p may be >= E)
__device__ __forceinline__ void payload_body(const PayloadArgs& a, int p) {
    const uint32_t* __restrict__ order = a.order;
    const uint32_t* __restrict__ skey = a.skey;
    const MsgSource& msgs = a.msgs;
    const float* __restrict__ w = a.w;
    const int E = a.count.get();
    uint32_t* __restrict__ ssrc = a.ssrc;
    float* __restrict__ sw = a.sw;
    uint32_t* __restrict__ sslot = a.sslot;
    uint32_t* __restrict__ slen = a.slen;
    uint32_t* __restrict__ hub_giant = a.hub_giant;
    uint32_t* __restrict__ hub_reg = a.hub_reg;
    uint32_t* __restrict__ small_heads = a.small_heads;
    uint32_t* __restrict__ ctr = a.ctr;
    int* __restrict__ svst = a.svst;
    const int* __restrict__ stamps = a.stamps;
    const int L = a.L, E4 = a.E4;
    const long long num_nodes = a.num_nodes;
    int* __restrict__ err_flag = a.err_flag;
    const int lane = threadIdx.x & 31;
    bool small_head = false;
    if (p < E) {
        const uint32_t m = order[p];
        long long tgt_unused, oth;
        int j;
        msgs.get((int)m, tgt_unused, oth, j);
        const uint32_t other = (uint32_t)oth;
        const uint32_t mykey = skey[p];
        if (a.key_out != skey) a.key_out[p] = mykey;
        ssrc[p] = other;
        float wv = w[j];
        if (sslot != nullptr) {          // snapshot path: where the source node's own segment starts
            int lo = 0, hi = E;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (skey[mid] < other) lo = mid + 1; else hi = mid;
            }
            uint32_t slot = (uint32_t)lo;
            if (msgs.B == 0 && (lo >= E || skey[lo] != other)) {      // message mode: not a target of this call
                if (stamps != nullptr && (long long)other < msgs.direct_from && err_flag != nullptr) *err_flag = 2;
                slot = kDirect;
                wv = __int_as_float(__float_as_int(wv) | 0x80000000);  // weights are >= 0: the sign bit marks
            }                                                          // a source read straight from the state
            sslot[p] = slot;
        }
        sw[p] = wv;
        uint32_t len = 0;
        if (p == 0 || skey[p - 1] != mykey) {     // heads only: end of the segment by binary search
            int lo = p, hi = E;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (skey[mid] <= mykey) lo = mid + 1; else hi = mid;
            }
            len = (uint32_t)(lo - p);
            // long segments go to the CTA-pipelined walkers; integer atomics only (the list order
            // decides scheduling, never results)
            if ((long long)mykey < num_nodes) {
                if (len >= (uint32_t)kGiantMin) {
                    const uint32_t gi = atomicAdd(&ctr[kCtrGiant], 1u);
                    hub_giant[gi] = (uint32_t)p;
                    if (a.chunk > 0) {
                        // chunked order: the giant's messages are cut into chunks of `chunk` messages, each an
                        // ordinary hub entry that sums its messages in order into its own partial row (from +0);
                        // combine_giants_kernel then adds the partial rows to the target in chunk order.
                        // Slot numbers only decide where a partial row lives, never a result.
                        const uint32_t nch = (len + (uint32_t)a.chunk - 1u) / (uint32_t)a.chunk;
                        const uint32_t cb = atomicAdd(&ctr[kCtrChunks], nch);
                        const uint32_t eb = atomicAdd(&ctr[kCtrHub], nch);
                        a.giant_cbase[gi] = cb;
                        for (uint32_t c = 0; c < nch; ++c) {
                            hub_reg[eb + c] = (uint32_t)p + c * (uint32_t)a.chunk;
                            a.hub_len[eb + c] = min((uint32_t)a.chunk, len - c * (uint32_t)a.chunk);
                            a.hub_part[eb + c] = cb + c;
                        }
                    }
                } else if (len >= (uint32_t)kHubMin) {
                    const uint32_t e = atomicAdd(&ctr[kCtrHub], 1u);
                    hub_reg[e] = (uint32_t)p;
                    a.hub_len[e] = len;
                    a.hub_part[e] = kNoPart;
                } else {
                    small_head = true;
                }
            }
        }
        slen[p] = len;
        if (svst != nullptr) {           // lazy per-layer path: pre-batch stamps of the source rows 1..L-1
            for (int l = 0; l < L - 1; ++l)
                svst[(size_t)l * E4 + p] = (long long)other < num_nodes ? stamps[(long long)other * L + l] : -1;
        }
    }
    // compacted list of short-segment heads: one atomic per warp, order within the warp kept
    const uint32_t mask = __ballot_sync(0xffffffffu, small_head);
    if (mask != 0) {
        const int leader = __ffs(mask) - 1;
        uint32_t base = 0;
        if (lane == leader) base = atomicAdd(&ctr[kCtrSmall], (uint32_t)__popc(mask));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (small_head) small_heads[base + __popc(mask & ((1u << lane) - 1u))] = (uint32_t)p;
    }
}

__global__ void __launch_bounds__(256) payload_kernel(PayloadArgs a) {
    payload_body(a, blockIdx.x * blockDim.x + threadIdx.x);
}

// Longest giant segments first: their add chains are the critical path of the hub walker.
// (Scheduling order only — results do not depend on it.)
constexpr int kGiantSortMax = kGiantSortMaxC;
struct GiantSmem {
    uint32_t head_s[kGiantSortMax], len_s[kGiantSortMax], sorted_s[kGiantSortMax];
};
// Also decides which giants are STREAMED (walk_hub2_kernel): the first n_stream entries of the sorted list;
// gblk[i] = first production block of the i-th of them.  stream_mode 0: none; 2: every giant (tests); 1: those whose
// add chain would otherwise be the critical path of the whole update.  Measured on B200 (profiles/r02_stream_giants.txt):
// the gathering hub walker adds a giant at ~10 cycles per message, the update as a whole costs ~3 cycles per message
// of the batch (throughput), a streamed chain ~4.5 cycles per message plus ~2.6 cycles per streamed message of extra
// traffic spread over all SMs — so streaming pays when the giant's chain, not the batch's throughput, bounds the call.
// Measured crossover: a giant holding 18 % of the messages (the N=1 bench batch): streaming it costs 10 % of the update;
// 30 % (the hub-owning rank at N=2): it gains 11 %; 47 % / 63 % (N=4 / N=8): much more.  Threshold: 1/4 of the messages.
__device__ __forceinline__ void sort_giants_body(GiantSmem& sm, uint32_t* __restrict__ hub_giant,
                                                 const uint32_t* __restrict__ slen, uint32_t* __restrict__ ctr,
                                                 uint32_t* __restrict__ gblk, uint32_t* __restrict__ gflag, Count count,
                                                 int stream_mode) {
    const uint32_t stream_min = stream_mode == 0 ? 0u
                                : (stream_mode == 2 ? (uint32_t)kGiantMin
                                                    : max((uint32_t)kGiantMin, (uint32_t)(count.get() >> 2)));
    const int n = (int)ctr[kCtrGiant];
    if (n < 1 || n > kGiantSortMax) return;          // ctr[kCtrStream] stays 0: the hub walker takes every giant
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        sm.head_s[i] = hub_giant[i];
        sm.len_s[i] = slen[sm.head_s[i]];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const uint32_t li = sm.len_s[i];
        int rank = 0;
        for (int j = 0; j < n; ++j) rank += (sm.len_s[j] > li || (sm.len_s[j] == li && j < i)) ? 1 : 0;
        hub_giant[rank] = sm.head_s[i];
        sm.sorted_s[rank] = li;
    }
    __syncthreads();
    if (threadIdx.x == 0 && stream_min > 0) {
        uint32_t blocks = 0;
        int ns = 0;
        for (; ns < n && sm.sorted_s[ns] >= stream_min; ++ns) {
            gblk[ns] = blocks;
            blocks += (sm.sorted_s[ns] + (uint32_t)kStreamBlock - 1u) / (uint32_t)kStreamBlock;
        }
        gblk[ns] = blocks;
        ctr[kCtrStream] = (uint32_t)ns;
        ctr[kCtrStreamBlocks] = blocks;
        sm.head_s[0] = blocks;
    }
    __syncthreads();
    if (stream_min > 0) {                      // "produced" flags of this call's blocks (uniform branch)
        const uint32_t blocks = sm.head_s[0];
        for (uint32_t i = threadIdx.x; i < blocks; i += blockDim.x) gflag[i] = 0;
    }
}
__global__ void __launch_bounds__(1024)
sort_giants_kernel(uint32_t* __restrict__ hub_giant, const uint32_t* __restrict__ slen, uint32_t* __restrict__ ctr,
                   uint32_t* __restrict__ gblk, uint32_t* __restrict__ gflag, Count count, int stream_mode) {
    __shared__ GiantSmem sm;
    sort_giants_body(sm, hub_giant, slen, ctr, gblk, gflag, count, stream_mode);
}

// ---------------------------------------------------------------- fused front end (large path)
// prep + every radix pass in ONE cooperative launch (<= one CTA per SM, all resident), phases separated by a grid
// barrier, instead of 10 dependent launches of a few microseconds each.  Payload and giant ordering stay separate
// launches: the payload's binary searches are latency-bound and want ~800 CTAs, not one per tile (measured: 100 us
// with the payload inside the 98-CTA launch, 49 us + 13 us + 4 us as three launches; profiles/r02k_*).
//   phase 0      weights, keys, tile histograms of pass 0 (the keys are still in registers); hist2 zeroed
//   per pass     per-digit prefix over tiles (one warp per digit)  | barrier |  stable scatter of every tile, which
//                also counts the NEXT pass's [tile][digit] histogram of the positions it writes (integer atomics:
//                counts are order-independent)  | barrier |
// The barrier: one arrival counter in the workspace, zeroed by a memset node in front of the launch and monotonic
// inside it; the spin is bounded (a grid that is not co-resident flags error 8 instead of hanging the GPU).
struct FrontArgs {
    PrepArgs prep;
    uint32_t *key_a, *key_b, *val_a, *val_b, *hist, *hist2, *bar;
    int passes;
};

__device__ __forceinline__ void grid_barrier(uint32_t* bar, uint32_t& target, int* err_flag) {
    __syncthreads();
    if (threadIdx.x == 0) {
        target += gridDim.x;
        __threadfence();
        atomicAdd(bar, 1u);
        uint32_t seen;
        long long spins = 0;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(bar) : "memory");
            if (seen >= target) break;
            if (++spins > (1ll << 22)) {                     // seconds: the grid is not co-resident
                if (err_flag != nullptr) *err_flag = 8;
                break;
            }
        } while (true);
    }
    __syncthreads();
}

union FrontSmem {
    uint32_t bins[kRadixBins];
    ScatterSmem scatter;
};

__global__ void __launch_bounds__(kRadixThreads)
front_kernel(FrontArgs a) {
    __shared__ FrontSmem sm;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int E = a.prep.count.get();
    const int nblk = (E + kRadixTile - 1) / kRadixTile;
    uint32_t target = 0;
    // ---- phase 0: prep + histogram of pass 0 (tile by tile), hist2 zeroed
    {
        const int ncap = (a.prep.count.cap + kRadixTile - 1) / kRadixTile;
        const int cells = (ncap + 1) * kRadixBins;
        for (int i = blockIdx.x * kRadixThreads + tid; i < cells; i += gridDim.x * kRadixThreads) a.hist2[i] = 0;
        // tiles past the count still run prep_body for their first threads: counters / flags / log row of thread m
        static_assert(kCtrSlots <= kRadixTile, "tile 0 zeroes the per-call counters");
        const int ntile0 = nblk > 0 ? nblk : 1;
        for (int tile = blockIdx.x; tile < ntile0; tile += gridDim.x) {
            sm.bins[tid] = 0;
            __syncthreads();
#pragma unroll
            for (int i = 0; i < kRadixItems; ++i) {
                const int m = tile * kRadixTile + i * kRadixThreads + tid;
                prep_body(a.prep, m);
                if (m < E) atomicAdd(&sm.bins[a.prep.key[m] & 0xff], 1u);
            }
            __syncthreads();
            if (tile < nblk) a.hist[tile * kRadixBins + tid] = sm.bins[tid];
            __syncthreads();
        }
    }
    grid_barrier(a.bar, target, a.prep.err_flag);
    uint32_t *kin = a.key_a, *kout = a.key_b, *vin = a.val_a, *vout = a.val_b;
    uint32_t *hcur = a.hist, *hnext = a.hist2;
    for (int p = 0; p < a.passes; ++p) {
        // ---- prefix over tiles, one warp per digit
        for (int dgt = blockIdx.x * kRadixWarps + wid; dgt < kRadixBins; dgt += gridDim.x * kRadixWarps)
            prefix_digit(hcur, nblk, dgt, lane);
        grid_barrier(a.bar, target, a.prep.err_flag);
        // ---- scatter (+ histogram of the next pass)
        const int shift = 8 * p;
        const bool more = p + 1 < a.passes;
        for (int tile = blockIdx.x; tile < nblk; tile += gridDim.x) {
            scatter_tile(sm.scatter, kin, vin, kout, vout, E, shift, hcur, nblk, 1, tile, more ? hnext : nullptr);
            __syncthreads();
        }
        if (!more) break;                                    // the kernel boundary orders the last scatter
        grid_barrier(a.bar, target, a.prep.err_flag);
        if (p + 2 < a.passes) {
            // the histogram just consumed becomes the one after next: zero it (nobody reads it before the next barrier)
            const int cells = (nblk + 1) * kRadixBins;
            for (int i = blockIdx.x * kRadixThreads + tid; i < cells; i += gridDim.x * kRadixThreads) hcur[i] = 0;
        }
        uint32_t* t = kin; kin = kout; kout = t;
        t = vin; vin = vout; vout = t;
        t = hcur; hcur = hnext; hnext = t;
    }
}

// cooperative launches (the fused front end) need the device attribute; queried once per device
bool front_kernel_ok() {
    static int table[kMaxDevices];          // 0 = not queried, 1 = yes, -1 = no
    int& t = table[g_dev_slot];
    if (t == 0) {
        int dev = 0, coop = 0;
        if (cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev) != cudaSuccess) {
            (void)cudaGetLastError();
            coop = 0;
        }
        t = coop ? 1 : -1;
    }
    return t == 1;
}

// ---------------------------------------------------------------- eager decay sweep (large path)
__global__ void __launch_bounds__(256)
sweep_decay_kernel(StateView st, DecayArgs decay, long long total4, int ds4) {
    sweep_body(st, decay, total4, ds4, (long long)blockIdx.x * blockDim.x + threadIdx.x,
               (long long)gridDim.x * blockDim.x);
}

// ---------------------------------------------------------------- the walk update
// Work item = (target segment, column tile), one WARP each.  The warp owns 32*V consecutive
// float4 of the target span (512*V contiguous bytes), reads them once, replays pending decay
// (lazy), then walks the segment's messages in order: the 32 lanes fetch the metadata
// (source id, weight, snapshot slot) of 32 messages with one coalesced load each and
// broadcast it by shuffle; D source rows are in flight per lane before the first add;
// every add is fadd_rn(acc, fmul_rn(source, w)); the span is written back once.
//   ALL = false : span = row `layer` of the target; sources = row layer-1 of the state
//                 (launched per layer, top-down; lazy sources are replayed in registers).
//   ALL = true  : span = rows 1..L of the target (contiguous in the node-major state);
//                 source row 0 comes from the state (P_0 is never written), source rows
//                 1..L-1 from the pre-batch snapshot taken by snapshot_kernel — one launch
//                 covers all layers and still reads only pre-batch values (TPNet.py:90).
template <int V, int D, bool LAZY, bool ALL>
__global__ void __launch_bounds__(kWalkThreads)
walk_kernel(StateView st, int layer, const uint32_t* __restrict__ skey, const uint32_t* __restrict__ ssrc,
            const float* __restrict__ sw, const uint32_t* __restrict__ sslot, const uint32_t* __restrict__ slen,
            const float* __restrict__ snap, Count count, int ds4, int write_stamp, int hub_min, DecayArgs dnow,
            int srow0) {
    const int wid = (blockIdx.x * kWalkThreads + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (wid >= count.get()) return;
    const uint32_t key = skey[wid];
    const uint32_t prev = wid > 0 ? skey[wid - 1] : 0xffffffffu;
    const int len = (int)slen[wid];
    if ((long long)key >= st.num_nodes || prev == key) return;   // dropped edge / not a segment head
    if (len >= hub_min) return;                                  // handled by walk_hub_kernel
    const int L = st.num_layer;
    const int span4 = ALL ? L * ds4 : ds4;               // float4 in the target span
    const int soff = srow0 * ds4;                        // source columns below this come from the state (P_0)
    const int snap4 = L * ds4 - soff;                    // float4 per snapshot slot
    const int col0 = blockIdx.y * (32 * V) + lane;

    float* tbase = st.data + (long long)key * st.node_stride + (long long)(ALL ? 1 : layer) * st.row_stride;
    float4 acc[V];
#pragma unroll
    for (int k = 0; k < V; ++k) {
        const int c = col0 + k * 32;
        const int tli = ALL ? (c < span4 ? c / ds4 : 0) : layer - 1;     // decay-log column of this register
        long long tstamp = 0;
        if (LAZY && c < span4) tstamp = st.stamps[(long long)key * L + tli];
        acc[k] = (c < span4 && tstamp >= 0) ? ld4(tbase + 4 * (long long)c) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (LAZY && c < span4 && tstamp >= 0) scale4(acc[k], decay_factor(st, tli, tstamp));
    }

    for (int base = 0; base < len; base += 32) {
        const int nmsg = min(32, len - base);
        // one coalesced metadata load per lane covers 32 messages
        uint32_t my_v = 0, my_slot = 0;
        float my_w = 0.f;
        long long my_vstamp = 0;
        if (lane < nmsg) {
            const int p = wid + base + lane;
            my_v = ssrc[p];
            my_w = sw[p];
            if (ALL) my_slot = sslot[p];
            else if (LAZY && layer >= 2) my_vstamp = st.stamps[(long long)my_v * L + (layer - 2)];
        }
        for (int j0 = 0; j0 < nmsg; j0 += D) {
            float4 x[D][V];
            float w[D];
            long long vstamp[D];
#pragma unroll
            for (int j = 0; j < D; ++j) {                 // issue every row load of the chunk first
                const int jj = j0 + j;
                const int sl = jj < nmsg ? jj : 0;
                const uint32_t v = __shfl_sync(0xffffffffu, my_v, sl);
                w[j] = __shfl_sync(0xffffffffu, my_w, sl);
                const uint32_t slot = ALL ? __shfl_sync(0xffffffffu, my_slot, sl) : 0u;
                vstamp[j] = (!ALL && LAZY) ? __shfl_sync(0xffffffffu, my_vstamp, sl) : 0;
                const float* sstate = st.data + (long long)v * st.node_stride +
                                      (long long)(ALL ? 0 : layer - 1) * st.row_stride;
                const bool direct = ALL && (slot & kDirect) != 0;     // rows 0..L-1 straight from the state
                const float* ssnap = ALL ? snap + (long long)(slot & ~kDirect) * snap4 * 4 : nullptr;
#pragma unroll
                for (int k = 0; k < V; ++k) {
                    const int c = col0 + k * 32;
                    float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (jj < nmsg && c < span4) {
                        if (ALL) {
                            val = (c < soff || direct) ? ld4(sstate + 4 * (long long)c)
                                                       : ld4(ssnap + 4 * (long long)(c - soff));
                            // cached rows of other ranks carry their own stamps, like any row (lazy mode;
                            // in eager mode the sweep already covered them): one multiply from the stamp
                            // to this call's epoch, exactly what the snapshot does for local sources
                            if (LAZY && direct && c >= ds4) {
                                const int sli = c / ds4 - 1;
                                const int sst = st.stamps[(long long)v * L + sli];
                                if (sst >= 0) scale4(val, decay_factor(st, sli, sst));
                            }
                        }
                        else if (vstamp[j] >= 0) val = ld4(sstate + 4 * (long long)c);
                    }
                    x[j][k] = val;
                }
            }
#pragma unroll
            for (int j = 0; j < D; ++j) {
                if (j0 + j < nmsg) {
                    if (!ALL && LAZY && layer >= 2 && vstamp[j] >= 0) {    // P_0 never decays
                        const float f = decay_factor(st, layer - 2, vstamp[j]);
#pragma unroll
                        for (int k = 0; k < V; ++k) scale4(x[j][k], f);
                    }
#pragma unroll
                    for (int k = 0; k < V; ++k) axpy4_rn(acc[k], x[j][k], w[j]);
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < V; ++k) {
        const int c = col0 + k * 32;
        if (c < span4) st4(tbase + 4 * (long long)c, acc[k]);
    }
    if (LAZY && write_stamp && lane == 0) st.stamps[(long long)key * L + (layer - 1)] = (int)st.epoch;
}

// Pre-batch copy of rows 1..L-1 of every target of the batch (brought current in lazy mode),
// one warp per segment head; slot = sorted position of the head.
template <bool LAZY>
__global__ void __launch_bounds__(256)
snapshot_kernel(StateView st, const uint32_t* __restrict__ skey, Count count, int ds4, float* __restrict__ snap,
                int srow0) {
    const int p = (blockIdx.x * 256 + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (p >= count.get()) return;
    const uint32_t key = skey[p];
    if ((long long)key >= st.num_nodes) return;
    if (p > 0 && skey[p - 1] == key) return;
    const int L = st.num_layer;
    const int snap4 = (L - srow0) * ds4;                 // rows srow0..L-1 (srow0 = 1: P_0 is read from the state)
    const float* rows = st.data + (long long)key * st.node_stride + (long long)srow0 * st.row_stride;
    float* slot = snap + (long long)p * snap4 * 4;
    // pending decay: lane j handles snapshot row j = state row srow0 + j (row 0, P_0, never decays): it fetches
    // the row's stamp and computes its factor (one f64 division per row, not per lane and column step); a
    // negative factor marks a row that was never written (all zero): it is not read at all
    float fmine = 1.0f;
    if (LAZY && lane < L - srow0 && srow0 + lane >= 1) {
        const int li = srow0 + lane - 1;                 // decay-log column of state row srow0 + lane
        const long long stamp = st.stamps[(long long)key * L + li];
        fmine = stamp >= 0 ? decay_factor(st, li, stamp) : -1.0f;
    }
    float f[TPN_MAX_LAYERS];
#pragma unroll
    for (int l = 0; l < TPN_MAX_LAYERS; ++l) f[l] = LAZY ? __shfl_sync(0xffffffffu, fmine, l) : 1.0f;
    for (int c0 = lane; c0 < snap4; c0 += 128) {        // four row requests in flight per lane
        float4 v[4];
        float fk[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int c = c0 + 32 * k;
            const int li = c / ds4;                     // layer - 1
            fk[k] = li == 0 ? f[0] : (li == 1 ? f[1] : (li == 2 ? f[2] : f[3]));
            v[k] = (c < snap4 && fk[k] >= 0.f) ? ld4(rows + 4 * (long long)c) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int c = c0 + 32 * k;
            if (c < snap4) {
                if (LAZY && fk[k] >= 0.f && fk[k] != 1.0f) scale4(v[k], fk[k]);
                st4(slot + 4 * (long long)c, v[k]);
            }
        }
    }
}

// stamps of all layers (layer == 0) or one layer of every target <- current epoch
__global__ void __launch_bounds__(256)
stamp_targets_kernel(StateView st, int layer, const uint32_t* __restrict__ skey, Count count) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= count.get()) return;
    const uint32_t key = skey[p];
    if ((long long)key >= st.num_nodes) return;
    if (p > 0 && skey[p - 1] == key) return;
    if (layer >= 1) {
        st.stamps[(long long)key * st.num_layer + (layer - 1)] = (int)st.epoch;
    } else {
        for (int l = 0; l < st.num_layer; ++l) st.stamps[(long long)key * st.num_layer + l] = (int)st.epoch;
    }
}


// ---------------------------------------------------------------- long segments (hubs)
// A target's messages must be added one at a time in order (the reference's accumulation order
// is observable), so a hub of m messages is a dependent chain of m fp32 adds per column.  The
// warp walker above pays a DRAM round trip per D rows on that chain; here the chain runs out of
// shared memory instead.  Work item = (long segment, column slice of <= 128 floats), one CTA:
//   producer warp : stages the segment's metadata (source id, weight, snapshot slot / source
//                   stamp) in chunks of 512 messages with bulk copies, then every lane issues the
//                   `cp.async.bulk` (TMA) copy of one message's source-row slice into a ring of
//                   4 stages x 32 messages (completion on the stage's `full` mbarrier);
//   4 consumer warps : one float column per lane; per message LDS + FMUL + FADD with the add
//                   chain as the only dependency (~4 cycles per message), `empty` mbarrier back.
// CTAs pull work items from an atomic counter, giant segments first.  Same arithmetic as the
// warp walker: acc = fadd_rn(acc, fmul_rn(source, w)) in sorted-message order.
struct HubSmem {
    float ring[kHubStages][32][kHubSlotFloats];
    float wring[kHubStages][32];
    int vring[kHubStages][32];
    uint32_t msrc[2][kHubMetaChunk + 4];
    float mw[2][kHubMetaChunk + 4];
    uint32_t mx[2][kHubMetaChunk + 4];
    uint64_t full[kHubStages];
    uint64_t empty[kHubStages];
    uint64_t mfull[2];
    int item[4];
};

template <bool LAZY, bool ALL>
__global__ void __launch_bounds__(kHubThreads)
walk_hub_kernel(StateView st, int layer, const uint32_t* __restrict__ skey, const uint32_t* __restrict__ ssrc,
                const float* __restrict__ sw, const uint32_t* __restrict__ xarr, const uint32_t* __restrict__ slen,
                const float* __restrict__ snap, const uint32_t* __restrict__ hub_giant,
                const uint32_t* __restrict__ hub_reg, uint32_t* __restrict__ ctr, int work_ctr, int span,
                int slice_w, int slices, DecayArgs dnow) {
    extern __shared__ __align__(128) unsigned char hub_raw[];
    HubSmem& sm = *reinterpret_cast<HubSmem*>(hub_raw);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int L = st.num_layer;
    const int rs = (int)st.row_stride;
    const bool has_x = ALL || (LAZY && layer >= 2);
    if (threadIdx.x == 0) {
        for (int i = 0; i < kHubStages; ++i) {
            mbar_init(&sm.full[i], 1);
            mbar_init(&sm.empty[i], kHubConsumers);
        }
        mbar_init(&sm.mfull[0], 1);
        mbar_init(&sm.mfull[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const uint32_t n_giant = ctr[0], n_reg = ctr[1];
    const uint32_t total = (n_giant + n_reg) * (uint32_t)slices;
    uint32_t blk = 0;       // ring blocks produced / consumed so far by this CTA (same count in every warp)
    uint32_t mit = 0;       // metadata chunks staged so far (producer warp)
    for (;;) {
        if (threadIdx.x == 0) sm.item[0] = (int)atomicAdd(&ctr[work_ctr], 1u);
        __syncthreads();
        const uint32_t work = (uint32_t)sm.item[0];
        __syncthreads();
        if (work >= total) break;
        const uint32_t it = work / (uint32_t)slices;
        const int slice = (int)(work - it * (uint32_t)slices);
        const int head = (int)(it < n_giant ? hub_giant[it] : hub_reg[it - n_giant]);
        const int len = (int)slen[head];
        const uint32_t key = skey[head];
        const int c0 = slice * slice_w;
        const int c1 = min(span, c0 + slice_w);
        const uint32_t msg_bytes = (uint32_t)(c1 - c0) * 4u;

        if (warp == kHubConsumers) {
            // ------------------------------------------------ producer
            const int nchunk = (len + kHubMetaChunk - 1) / kHubMetaChunk;
            auto issue_meta = [&](int c, uint32_t m) {
                const int cs = c * kHubMetaChunk;
                const int cn = min(kHubMetaChunk, len - cs);
                const int a0 = (head + cs) & ~3;                         // 16-byte aligned start
                const uint32_t bytes = (uint32_t)(((head + cs + cn) - a0 + 3) & ~3) * 4u;
                const int buf = (int)(m & 1u);
                fence_proxy_async_smem();
                mbar_expect_tx(&sm.mfull[buf], bytes * (has_x ? 3u : 2u));
                bulk_g2s(sm.msrc[buf], ssrc + a0, bytes, &sm.mfull[buf]);
                bulk_g2s(sm.mw[buf], sw + a0, bytes, &sm.mfull[buf]);
                if (has_x) bulk_g2s(sm.mx[buf], xarr + a0, bytes, &sm.mfull[buf]);
            };
            if (lane == 0) issue_meta(0, mit);
            for (int c = 0; c < nchunk; ++c) {
                __syncwarp();
                if (c + 1 < nchunk && lane == 0) issue_meta(c + 1, mit + 1);
                const int buf = (int)(mit & 1u);
                mbar_wait(&sm.mfull[buf], (mit >> 1) & 1u);
                const int cs = c * kHubMetaChunk;
                const int cn = min(kHubMetaChunk, len - cs);
                const int off = (head + cs) & 3;
                for (int b = 0; b < cn; b += 32) {
                    const int stage = (int)(blk % kHubStages);
                    if (blk >= (uint32_t)kHubStages) mbar_wait(&sm.empty[stage], ((blk / kHubStages) - 1u) & 1u);
                    const int j = b + lane;
                    const bool valid = j < cn;
                    uint32_t v = 0, x = 0;
                    if (valid) {
                        v = sm.msrc[buf][off + j];
                        sm.wring[stage][lane] = sm.mw[buf][off + j];
                        if (has_x) x = sm.mx[buf][off + j];
                        sm.vring[stage][lane] = (int)x;
                    }
                    __syncwarp();
                    if (lane == 0) mbar_expect_tx(&sm.full[stage], (uint32_t)min(32, cn - b) * msg_bytes);
                    __syncwarp();
                    if (valid) {
                        float* dst = &sm.ring[stage][lane][0];
                        const float* vrow = st.data + (long long)v * st.node_stride;
                        if (ALL && (x & kDirect) != 0) {
                            // not a target of this call: rows 0..L-1 are contiguous in the state
                            bulk_g2s(dst, vrow + c0, msg_bytes, &sm.full[stage]);
                        } else if (ALL) {
                            // span columns < row_stride: P_0 of the source (never written);
                            // the rest: pre-batch rows 1..L-1 from the source's snapshot slot
                            const int a_end = min(c1, rs);
                            if (c0 < a_end) bulk_g2s(dst, vrow + c0, (uint32_t)(a_end - c0) * 4u, &sm.full[stage]);
                            if (c1 > rs) {
                                const int b0 = max(c0, rs);
                                bulk_g2s(dst + (b0 - c0), snap + (long long)x * (long long)(L - 1) * rs + (b0 - rs),
                                         (uint32_t)(c1 - b0) * 4u, &sm.full[stage]);
                            }
                        } else {
                            bulk_g2s(dst, vrow + (long long)(layer - 1) * rs + c0, msg_bytes, &sm.full[stage]);
                        }
                    }
                    ++blk;
                }
                ++mit;
            }
        } else {
            // ------------------------------------------------ consumers
            const int col = c0 + warp * 32 + lane;
            const bool active = col < c1;
            const int li = ALL ? (active ? col / rs : 0) : layer - 1;
            // direct (received) source rows: this call's decay factor of the source row this
            // column reads (span column -> source row li; P_0 never decays; 1.0f is exact)
            const float dfac = (ALL && LAZY && dnow.has_decay && li >= 1) ? dnow.c[li - 1] : 1.0f;
            float* tptr = st.data + (long long)key * st.node_stride + (long long)(ALL ? 1 : layer) * rs + col;
            float acc = 0.f;
            if (active) {
                long long ts = 0;
                if (LAZY) ts = st.stamps[(long long)key * L + li];
                if (ts >= 0) {
                    acc = *tptr;
                    if (LAZY) acc = __fmul_rn(acc, decay_factor(st, li, ts));
                }
            }
            const int nblk = (len + 31) >> 5;
            for (int b = 0; b < nblk; ++b) {
                const int stage = (int)(blk % kHubStages);
                mbar_wait(&sm.full[stage], (blk / kHubStages) & 1u);
                const int nm = min(32, len - b * 32);
                const float* xs = &sm.ring[stage][0][warp * 32 + lane];
                const float* ws_ = &sm.wring[stage][0];
                const int* vs = &sm.vring[stage][0];
                if (nm == 32) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        float x = xs[j * kHubSlotFloats];
                        if (ALL && LAZY) {
                            if ((uint32_t)vs[j] & kDirect) x = __fmul_rn(x, dfac);
                        }
                        if (LAZY && !ALL && layer >= 2) {
                            const int vst = vs[j];
                            x = vst < 0 ? 0.f : __fmul_rn(x, decay_factor(st, layer - 2, vst));
                        }
                        acc = __fadd_rn(acc, __fmul_rn(x, ws_[j]));
                    }
                } else {
                    for (int j = 0; j < nm; ++j) {
                        float x = xs[j * kHubSlotFloats];
                        if (ALL && LAZY) {
                            if ((uint32_t)vs[j] & kDirect) x = __fmul_rn(x, dfac);
                        }
                        if (LAZY && !ALL && layer >= 2) {
                            const int vst = vs[j];
                            x = vst < 0 ? 0.f : __fmul_rn(x, decay_factor(st, layer - 2, vst));
                        }
                        acc = __fadd_rn(acc, __fmul_rn(x, ws_[j]));
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.empty[stage]);
                ++blk;
            }
            if (active) *tptr = acc;
        }
    }
}


// ================================================================ large batches, snapshot path
__device__ __forceinline__ float pick4(float f0, float f1, float f2, float f3, int i) {
    return i == 0 ? f0 : (i == 1 ? f1 : (i == 2 ? f2 : f3));
}

// Short segments (< kHubMin messages).  Persistent warps stride over the compacted head list
// (payload_kernel); one warp owns the whole L*row_stride span of a target (V float4 per lane;
// wider spans are tiled over blockIdx.y).  Per segment: the target span and the first D source
// spans are requested together (one DRAM round trip), the next segment's metadata and the head
// after that are prefetched behind them, pending decay is one multiply per register, messages
// are added in order as fadd_rn(acc, fmul_rn(x, w)), the span is written once.  Source row 0
// comes from the state (P_0 is never written), rows 1..L-1 from the pre-batch snapshot, or —
// message mode, weight sign bit set — all of them straight from the state (received rows).
template <int V, bool LAZY, bool DIRECT>
__global__ void __launch_bounds__(kSmallWalkThreads, 2)
walk_small_kernel(StateView st, const uint32_t* __restrict__ skey, const uint32_t* __restrict__ ssrc,
                  const float* __restrict__ sw, const uint32_t* __restrict__ sslot,
                  const uint32_t* __restrict__ slen, const float* __restrict__ snap,
                  const uint32_t* __restrict__ heads, const uint32_t* __restrict__ ctr, int E, int ds4,
                  DecayArgs dnow, int srow0) {
    constexpr int D = V >= 4 ? 2 : 4;                 // source spans in flight per round
    const int lane = threadIdx.x & 31;
    const int warps = gridDim.x * (kSmallWalkThreads / 32);
    int it = blockIdx.x * (kSmallWalkThreads / 32) + (threadIdx.x >> 5);
    const int n_items = (int)ctr[kCtrSmall];
    if (it >= n_items) return;
    const int L = st.num_layer;
    const int span4 = L * ds4;
    const int soff = srow0 * ds4;                     // source columns below this come from the state (P_0)
    const int snap4 = span4 - soff;
    int col[V], tl[V];
    bool in[V];
#pragma unroll
    for (int k = 0; k < V; ++k) {
        col[k] = blockIdx.y * (32 * V) + k * 32 + lane;
        in[k] = col[k] < span4;
        tl[k] = in[k] ? col[k] / ds4 : 0;             // target layer - 1 == source row of this register
    }
    struct Meta { uint32_t key, len, v, slot; float w; };
    auto load_meta = [&](uint32_t p) {
        Meta m;
        m.key = skey[p];
        m.len = slen[p];
        const uint32_t q = min(p + (uint32_t)lane, (uint32_t)(E - 1));     // lanes >= len read neighbours: unused
        m.v = ssrc[q];
        m.w = sw[q];
        m.slot = sslot[q];
        return m;
    };
    uint32_t p_cur = heads[it];
    uint32_t p_nxt = it + warps < n_items ? heads[it + warps] : 0u;
    Meta mc = load_meta(p_cur);
    for (; it < n_items; it += warps) {
        const uint32_t p_this = p_cur;
        const uint32_t key = mc.key;
        const int len = (int)mc.len;
        float* tbase = st.data + (long long)key * st.node_stride + st.row_stride;      // rows 1..L
        float4 acc[V];
#pragma unroll
        for (int k = 0; k < V; ++k)      // rows never written hold zeros, so the load needs no stamp check
            acc[k] = in[k] ? ld4(tbase + 4 * (long long)col[k]) : make_float4(0.f, 0.f, 0.f, 0.f);
        int stamp[TPN_MAX_LAYERS];
        if (LAZY) {
#pragma unroll
            for (int l = 0; l < TPN_MAX_LAYERS; ++l) stamp[l] = l < L ? st.stamps[(long long)key * L + l] : -1;
        }
        uint32_t my_v = mc.v, my_slot = mc.slot;
        float my_w = mc.w;
        bool first = true;
        for (int base = 0; base < len; base += 32) {
            const int nmsg = min(32, len - base);
            if (base > 0 && lane < nmsg) {            // second round of a 33..63-message segment
                const uint32_t q = p_this + (uint32_t)(base + lane);
                my_v = ssrc[q];
                my_w = sw[q];
                my_slot = sslot[q];
            }
            for (int j0 = 0; j0 < nmsg; j0 += D) {
                float4 x[D][V];
                float w[D];
#pragma unroll
                for (int j = 0; j < D; ++j) {
                    const int jj = j0 + j;
                    const int sl = jj < nmsg ? jj : 0;
                    const uint32_t v = __shfl_sync(0xffffffffu, my_v, sl);
                    const uint32_t slot = __shfl_sync(0xffffffffu, my_slot, sl);
                    float wj = __shfl_sync(0xffffffffu, my_w, sl);
                    const bool direct = DIRECT && (slot & kDirect) != 0;
                    if (DIRECT) wj = fabsf(wj);
                    w[j] = wj;
                    // cached rows of other ranks (sharded state) carry their own stamps: lane l computes the pending
                    // factor of source row l + 1 (stamp -> this call's epoch, one multiply as in the snapshot)
                    float fd1 = 1.0f, fd2 = 1.0f, fd3 = 1.0f;
                    if (DIRECT && LAZY) {
                        float fm = 1.0f;
                        if (direct && jj < nmsg && lane < L - 1) {
                            const int sst = st.stamps[(long long)v * L + lane];
                            if (sst >= 0) fm = decay_factor(st, lane, sst);
                        }
                        fd1 = __shfl_sync(0xffffffffu, fm, 0);
                        fd2 = __shfl_sync(0xffffffffu, fm, 1);
                        fd3 = __shfl_sync(0xffffffffu, fm, 2);
                    }
                    const float* sstate = st.data + (long long)v * st.node_stride;
                    const float* ssnap = snap + (long long)(slot & ~kDirect) * snap4 * 4;
#pragma unroll
                    for (int k = 0; k < V; ++k) {
                        float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (jj < nmsg && in[k]) {
                            val = (col[k] < soff || direct) ? ld4(sstate + 4 * (long long)col[k])
                                                            : ld4(ssnap + 4 * (long long)(col[k] - soff));
                            if (DIRECT && LAZY && direct && col[k] >= ds4)
                                scale4(val, pick4(fd1, fd2, fd3, 1.0f, tl[k] - 1));      // x * 1.0f is exact
                        }
                        x[j][k] = val;
                    }
                }
                if (first) {
                    first = false;
                    // behind the row requests: metadata of the next segment, head of the one after
                    if (it + warps < n_items) mc = load_meta(p_nxt);
                    p_cur = p_nxt;
                    p_nxt = it + 2 * warps < n_items ? heads[it + 2 * warps] : 0u;
                    if (LAZY) {
                        float f[TPN_MAX_LAYERS];
#pragma unroll
                        for (int l = 0; l < TPN_MAX_LAYERS; ++l)
                            f[l] = (l < L && stamp[l] >= 0) ? decay_factor(st, l, stamp[l]) : 1.0f;
#pragma unroll
                        for (int k = 0; k < V; ++k) scale4(acc[k], pick4(f[0], f[1], f[2], f[3], tl[k]));
                    }
                }
#pragma unroll
                for (int j = 0; j < D; ++j) {
                    if (j0 + j < nmsg) {
#pragma unroll
                        for (int k = 0; k < V; ++k) axpy4_rn(acc[k], x[j][k], w[j]);
                    }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < V; ++k)
            if (in[k]) st4(tbase + 4 * (long long)col[k], acc[k]);
    }
}

// Long segments (>= kHubMin messages).  A target's messages are added one at a time in order
// (the reference's accumulation order is observable), so a hub of m messages is a dependent
// chain of m fp32 adds per column.  The chain must see nothing but the add: everything else is
// moved off it.  Work item = (segment, column slice inside ONE source row), one CTA:
//   7 producer warps : warp p owns ring stages b = p, p+7, ... of 32 messages (128 for giants).  Each
//       lane fetches the (source id, snapshot slot, weight) of one message, lanes exchange row pointers
//       by shuffle so that every 128-bit load instruction covers 2 (8 for giants) whole message
//       slices, coalesced; then the slices are scaled — fmul_rn(x, w), the reference's rounded
//       product (TPNet.py:91-96), plus this call's decay for received rows of a sharded state — and
//       stored to the stage, published with the stage's `full` mbarrier.  (Measured: a warp keeps
//       only 2-3 of these scattered LDG.128 in flight, so the number of producer WARPS sets the gather
//       rate; see DESIGN.md section 4 "Hubs" for the variants that were measured and rejected.)
//   1 consumer warp  : two adjacent columns per lane; per message one LDS.64 and two scalar
//       FADDs, acc = fadd_rn(acc, product) in sorted-message order — bit-identical to the warp
//       walker — then the stage goes back through its `empty` mbarrier.
// Giant segments (>= kGiantMin messages) are cut into <= 16-float slices, sorted longest first,
// and taken only by ONE CTA per SM (first CTA to claim its SM), so a critical chain never shares
// its SM's load/store path with another; everything else uses <= 64-float slices.  CTAs pull work
// items from atomic counters.  Shared memory: ring[stages][32][64] floats | full | empty | item.
#ifdef TPN_HUB2_TIMELINE
// profiling build only (-DTPN_HUB2_TIMELINE): SM-clock timestamps of the first giant work item,
// [warp][pass][event]; read with tpn_debug_hub_timeline (not part of the shipped ABI)
__device__ unsigned long long g_hub2_timeline[8 * 256 * 8];
#define HUB2_STAMP(pass, ev) \
    do { if (work == 0 && lane == 0 && (pass) < 256) g_hub2_timeline[(warp * 256 + (pass)) * 8 + (ev)] = clock64(); } while (0)
// every 8th stage of the first chain item, so that 256 slots cover a 2,048-stage (262,144-message) chain
#define HUB2_STAMP_W0(pass, ev) \
    do { if (stamp_me && lane == 0 && ((pass) & 7) == 0 && ((pass) >> 3) < 256) \
             g_hub2_timeline[(0 * 256 + ((pass) >> 3)) * 8 + (ev)] = clock64(); } while (0)
#else
#define HUB2_STAMP(pass, ev) do { } while (0)
#define HUB2_STAMP_W0(pass, ev) do { } while (0)
#endif

// The add chain of one giant work item (consumer warp): one column per lane, stages of 128 messages x 16 floats.
// Out of line on purpose: inside the walker's 128-register allocation ptxas sinks the loads to ~10 messages ahead of
// their adds, and a shared-memory load that queues behind the other warps' global loads and stores on this SM then
// arrives late — measured 6.9 cycles per message for the chain alone where the same loop runs at 4.1 on an idle SM
// (scripts/micro/chain_bench.cu).  Here the 32 values of the NEXT group are loaded before the 32 dependent adds of the
// current one, and the next stage's barrier is tested under the adds of a stage's last group.
__device__ __noinline__ float hub2_giant_chain(float acc, const float* ring, uint64_t* full, uint64_t* empty,
                                               uint32_t blk_base, int nblk, int len, int col, int lane, bool stamp_me) {
    constexpr int mps = 32 * kGiantSpm;
    (void)stamp_me;                     // only the timeline build reads it
    bool next_full = false;             // the next stage's `full` phase was already seen complete
    for (int b = 0; b < nblk; ++b) {
        const uint32_t g = blk_base + (uint32_t)b;
        const uint32_t use = g / (uint32_t)kHub2Stages;
        const int stage = (int)(g - use * (uint32_t)kHub2Stages);
        HUB2_STAMP_W0(b, 0);
        if (!next_full) mbar_wait(&full[stage], use & 1u);
        next_full = false;
        HUB2_STAMP_W0(b, 1);
        const int nm = min(mps, len - b * mps);
        const float* xs = ring + (size_t)stage * (32 * kHub2SlotFloats) + col;
        int j0 = 0;
        if (nm == mps) {
            float va[32], vb[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) va[j] = xs[j * kHub2GiantFloats];
#pragma unroll
            for (int q = 0; q < kGiantSpm; ++q) {
                float* cur = (q & 1) ? vb : va;
                float* nxt = (q & 1) ? va : vb;
                if (q + 1 < kGiantSpm) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) nxt[j] = xs[(32 * (q + 1) + j) * kHub2GiantFloats];
                } else if (b + 1 < nblk) {
                    const uint32_t g1 = g + 1u;
                    const uint32_t use1 = g1 / (uint32_t)kHub2Stages;
                    next_full = mbar_test(&full[g1 - use1 * (uint32_t)kHub2Stages], use1 & 1u);
                }
#pragma unroll
                for (int j = 0; j < 32; ++j) acc = __fadd_rn(acc, cur[j]);
            }
            j0 = nm;
        }
        for (; j0 < nm; ++j0) acc = __fadd_rn(acc, xs[j0 * kHub2GiantFloats]);
        HUB2_STAMP_W0(b, 2);
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[stage]);
        HUB2_STAMP_W0(b, 3);
    }
    return acc;
}


// Streamed giants.  A giant's messages must be added one at a time, and in the walker above the chain's own SM also has
// to GATHER them (64-byte pieces of random rows): an SM sustains only ~6-10 B/clk of such gathers (outstanding-miss
// capacity), 10 cycles per message where the add chain alone needs 4.  For the first ctr[kCtrStream] giants of the sorted
// list the two halves are therefore split over the CTAs of walk_stream_kernel:
//   produce : a work item = block q of 128 consecutive messages of one giant.  The CTA's 8 warps read WHOLE source rows
//       (rows 0..L-1 are contiguous: full cache lines, the HBM-efficient access), form the reference's rounded products
//       fmul_rn(x, w) (TPNet.py:91-96; plus the pending decay of received rows of a sharded state) and write them
//       slice-major — [slice][message][16 floats], the layout of a ring stage — then publish the block's flag (release).
//   chain   : the (giant, slice) work item as before, but its ring is filled by ONE loader thread: flag (acquire) -> one
//       8 KB bulk copy per stage (sequential lines, 11 stages = 88 KB in flight, no per-message gather).  The consumer warp
//       is unchanged: acc = fadd_rn(acc, product) in sorted-message order, bit-identical to every other path.
// The roles and why no deadlock is possible: see walk_stream_kernel.  The flag wait is bounded anyway.
__device__ __forceinline__ void fence_proxy_async_global() {
    asm volatile("fence.proxy.async.global;" ::: "memory");
}

template <bool LAZY, bool DIRECT>
__device__ __forceinline__ void hub2_produce_block(const StateView& st, uint32_t q, uint32_t n_stream,
                                                   const uint32_t* __restrict__ ssrc, const float* __restrict__ sw,
                                                   const uint32_t* __restrict__ sslot, const uint32_t* __restrict__ slen,
                                                   const float* __restrict__ snap, const uint32_t* __restrict__ hub_giant,
                                                   const uint32_t* __restrict__ gblk, float* __restrict__ gprod,
                                                   uint32_t* __restrict__ gflag, int srow0, int spr_g, int slice_w_g) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int kWarps = kHub2Threads / 32;
    const int L = st.num_layer;
    const int rs = (int)st.row_stride;
    const int ds4 = rs >> 2;
    const int span4 = L * ds4;
    const int first_snap4 = srow0 * ds4;          // float4 index where the rows read from the snapshot start
    const size_t mstride = (size_t)(L * spr_g) * kStreamSlice;     // floats of product space per message
    uint32_t lo = 0, hi = n_stream - 1;            // giant of block q: last i with gblk[i] <= q
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (gblk[mid] <= q) lo = mid; else hi = mid - 1;
    }
    const uint32_t b = q - gblk[lo];
    const uint32_t head = hub_giant[lo];
    const int len = (int)slen[head];
    const int first = (int)(b * kStreamBlock);
    const int nm = min(kStreamBlock, len - first);
    float* const out = gprod + (size_t)(head + first) * mstride;
    const size_t sstride = (size_t)nm * kStreamSlice;              // floats between slices of this block
    // two messages per warp and pass: 8 row requests of 512 bytes in flight per warp
    for (int m0 = warp; m0 < nm; m0 += 2 * kWarps) {
        const float* bs[2];                        // rows read from the state (P_0; every row of a received row)
        const float* bn[2];                        // rows >= srow0: pre-batch snapshot of the source's own segment
        float w[2], f[2][TPN_MAX_LAYERS];
        bool have[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int m = m0 + u * kWarps;
            have[u] = m < nm;
            const uint32_t j = head + first + (have[u] ? m : m0);
            const uint32_t v = ssrc[j];
            const uint32_t x = sslot[j];
            w[u] = sw[j];
            const bool direct = DIRECT && (x & kDirect) != 0;
            float fmine = 1.0f;                     // received row of another rank: its own stamp -> this call's epoch
            if (DIRECT) {
                if (LAZY && direct && lane >= 1 && lane < L) {
                    const int sst = st.stamps[(long long)v * L + (lane - 1)];
                    if (sst >= 0) fmine = decay_factor(st, lane - 1, sst);
                }
                w[u] = fabsf(w[u]);
            }
#pragma unroll
            for (int l = 0; l < TPN_MAX_LAYERS; ++l) f[u][l] = DIRECT ? __shfl_sync(0xffffffffu, fmine, l) : 1.0f;
            bs[u] = st.data + (long long)v * st.node_stride;
            bn[u] = direct ? bs[u] : snap + (long long)x * (long long)(L - srow0) * rs - (long long)srow0 * rs;
        }
        for (int i0 = lane; i0 < span4; i0 += 128) {
            float4 xv[2][4];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int i = i0 + 32 * k;
                    if (have[u] && i < span4) xv[u][k] = ld4((i < first_snap4 ? bs[u] : bn[u]) + 4 * (long long)i);
                }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int i = i0 + 32 * k;
                if (i < span4) {
                    // float4 i of the run = row r, column col -> slice r * spr_g + col / slice_w_g (the hub walker's slices)
                    const int r = (i >= ds4 ? 1 : 0) + (i >= 2 * ds4 ? 1 : 0) + (i >= 3 * ds4 ? 1 : 0);
                    const int col = 4 * (i - r * ds4);
                    const int ks = slice_w_g == 16 ? (col >> 4) : col / slice_w_g;
                    float* const o = out + (size_t)(r * spr_g + ks) * sstride + (col - ks * slice_w_g);
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        if (have[u]) {
                            if (DIRECT) scale4(xv[u][k], r == 0 ? f[u][0] : (r == 1 ? f[u][1] : (r == 2 ? f[u][2] : f[u][3])));
                            scale4(xv[u][k], w[u]);
                            st4(o + (size_t)(m0 + u * kWarps) * kStreamSlice, xv[u][k]);
                        }
                    }
                }
            }
        }
    }
    fence_proxy_async_global();                   // these generic-proxy writes are read by bulk copies (async proxy)
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(gflag + q), "r"(1u) : "memory");
    }
}


// Feeds the ring of a streamed giant item: warp 2 polls the producers' flags, warp 1 issues the bulk copies (one lane
// each), so a flag round trip never delays a copy.  Kept out of line: the gathering path keeps its register allocation.
__device__ __forceinline__ void hub2_stream_feed(int warp, int lane, volatile int* ready_s, uint32_t q0,
                                              const uint32_t* __restrict__ gflag, const float* __restrict__ gprod,
                                              int* __restrict__ err, int nblk, uint32_t blk_base, int len, uint32_t head,
                                              int slice, int slices_g, float* ring, uint64_t* full, uint64_t* empty) {
    if (warp == 2 && lane == 0) {
        int ready = 0;                  // leading blocks known to be produced (ready_s was reset by thread 0)
        while (ready < nblk) {
            uint32_t seen = 0;
            long long spins = 0;
            for (;;) {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(gflag + q0 + ready) : "memory");
                if (seen != 0) break;
                if (++spins > (1ll << 21)) {       // seconds: cannot happen (see above); never hang the GPU
                    if (err != nullptr) *err = 8;
                    ready = nblk - 1;
                    break;
                }
                __nanosleep(32);
            }
            ++ready;
            // the producers usually run far ahead: one round trip looks at the next 12 flags
            uint32_t fl[12];
#pragma unroll
            for (int k = 0; k < 12; ++k) {
                fl[k] = 0;
                if (ready + k < nblk)
                    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(fl[k]) : "l"(gflag + q0 + ready + k) : "memory");
            }
            asm volatile("fence.acq_rel.gpu;" ::: "memory");
            int more = 0;
#pragma unroll
            for (int k = 0; k < 12; ++k)
                if (fl[k] != 0 && more == k) ++more;
            ready += more;
            __threadfence_block();
            *ready_s = ready;
        }
    } else if (warp == 1) {
        const size_t mstride = (size_t)slices_g * kStreamSlice;
        int fenced = 0;             // blocks [0, fenced) are ordered for this thread's async-proxy reads
        for (int b = 0; b < nblk; ++b) {
            const uint32_t g = blk_base + (uint32_t)b;
            const uint32_t use = g / (uint32_t)kHub2Stages;
            const int stage = (int)(g - use * (uint32_t)kHub2Stages);
            if (lane == 0) {
                if (use > 0) mbar_wait(&empty[stage], (use - 1u) & 1u);
                if (b >= fenced) {
                    // one proxy fence per batch of newly produced blocks, not per copy
                    int r;
                    while ((r = *ready_s) <= b) { }
                    __threadfence_block();
                    fence_proxy_async_global();
                    fenced = r;
                }
                const int first = b * kStreamBlock;
                const int nmb = min(kStreamBlock, len - first);
                const uint32_t bytes = (uint32_t)nmb * kStreamSlice * 4u;
                const float* src = gprod + (size_t)(head + first) * mstride + (size_t)slice * (size_t)(nmb * kStreamSlice);
                mbar_expect_tx(&full[stage], bytes);          // the stage's one arrival, plus the bytes
                bulk_g2s(ring + (size_t)stage * (32 * kHub2SlotFloats), src, bytes, &full[stage]);
            }
            __syncwarp();
        }
    }
}


// The streamed giants of one update: ONE launch beside walk_hub2_kernel (which skips them), same CTA shape and ring.
//   * CTAs take a ticket when they start.  Tickets 1..C chain: they pull (giant, slice) items — the longest giant's
//     slices first — warp 0 adds, warp 1 issues the bulk copies, warp 2 polls the flags;
//   * every other CTA (ticket 0 included) registers as a producer when it starts and takes production blocks until none
//     are left, then exits;
//   * a chaining CTA only starts once a producer is registered; if none shows up within microseconds it registers
//     itself and produces first.  A registered producer never waits for anything, so every flag a chain waits for is
//     eventually set whatever else is (or is not) resident: no co-residency assumption between CTAs or launches — valid
//     inside CUDA graphs, on aliased hardware queues and under a serialising profiler.  (The first design had producers
//     and chains as two launches on two streams: it passed the tests and then hung in the bench, where the process owns
//     more streams than hardware queues and the chain kernel was queued in front of its own producers.)
template <bool LAZY, bool DIRECT>
__global__ void __launch_bounds__(kHub2Threads, 2)
walk_stream_kernel(StateView st, const uint32_t* __restrict__ skey, const uint32_t* __restrict__ ssrc,
                   const float* __restrict__ sw, const uint32_t* __restrict__ sslot, const uint32_t* __restrict__ slen,
                   const float* __restrict__ snap, const uint32_t* __restrict__ hub_giant, uint32_t* __restrict__ ctr,
                   int spr_g, int slice_w_g, int srow0, const uint32_t* __restrict__ gblk, float* __restrict__ gprod,
                   uint32_t* __restrict__ gflag, int* __restrict__ err) {
    static_assert(kStreamSlice == kHub2GiantFloats && kStreamBlock == 32 * kGiantSpm,
                  "a production block of one slice is exactly one ring stage of a giant item");
    const uint32_t n_stream = ctr[kCtrStream];
    if (n_stream == 0) return;                       // the usual case: nothing is streamed
    extern __shared__ __align__(128) unsigned char stream_raw[];
    float* const ring = reinterpret_cast<float*>(stream_raw);                     // [stages][128 messages][16 floats]
    uint64_t* const full = reinterpret_cast<uint64_t*>(ring + (size_t)kHub2Stages * 32 * kHub2SlotFloats);
    uint64_t* const empty = full + kHub2Stages;
    int* const item = reinterpret_cast<int*>(empty + kHub2Stages);          // [0]: work item, [1]: its kind, [2]: ready blocks
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int L = st.num_layer;
    const int rs = (int)st.row_stride;
    if (threadIdx.x == 0) {
        for (int i = 0; i < kHub2Stages; ++i) {
            mbar_init(&full[i], 1);                    // the loader's expect_tx arrival; the bulk copy completes the bytes
            mbar_init(&empty[i], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        *item = (int)atomicAdd(&ctr[kCtrStreamTicket], 1u);
    }
    __syncthreads();
    const uint32_t ticket = (uint32_t)*item;
    __syncthreads();
    const uint32_t slices_g = (uint32_t)(L * spr_g);
    const uint32_t total_c = n_stream * slices_g;
    const uint32_t stream_blocks = ctr[kCtrStreamBlocks];
    // one CTA per SM (the grid): tickets 1..C chain, C = one per chain item but at most half of the grid; ticket 0 and
    // the rest produce.  The producers only have to stay ahead of the chains (a chain consumes ~0.3 messages per ns,
    // a producer CTA delivers ~8 per us), so they leave the other half of every SM to the walkers of the other segments.
    const bool chains = ticket >= 1u && ticket <= min(total_c, gridDim.x / 2u);
    // scheduling state, meaningful in thread 0 only
    bool prod_first = !chains, prod_done = false, chains_done = !chains;
    if (threadIdx.x == 0) {
        if (!chains) {
            atomicAdd(&ctr[kCtrStreamActive], 1u);
        } else {
            uint32_t active = 0;
            for (int spins = 0; spins < 16; ++spins) {               // ~15 us at most
                asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(active) : "l"(ctr + kCtrStreamActive) : "memory");
                if (active != 0) break;
                __nanosleep(200);
            }
            if (active == 0) {
                atomicAdd(&ctr[kCtrStreamActive], 1u);
                prod_first = true;
            }
        }
    }
    uint32_t blk_base = 0;      // ring stages used so far by this CTA (same count in every warp)
    for (;;) {
        if (threadIdx.x == 0) {
            int w = -1, kind = 0;        // kind 1: production block w; kind 0: chain item w; w == -1: nothing left
            if (prod_first && !prod_done) {
                const uint32_t q = atomicAdd(&ctr[kCtrStreamProd], 1u);
                if (q < stream_blocks) { w = (int)q; kind = 1; } else prod_done = true;
            }
            if (w == -1 && !chains_done) {
                const uint32_t c = atomicAdd(&ctr[kCtrStreamChain], 1u);
                if (c < total_c) w = (int)c; else chains_done = true;
            }
            if (w == -1 && !prod_done) {               // a chaining CTA that ran out of chains helps the producers
                const uint32_t q = atomicAdd(&ctr[kCtrStreamProd], 1u);
                if (q < stream_blocks) { w = (int)q; kind = 1; } else prod_done = true;
            }
            item[0] = w;
            item[1] = kind;
            item[2] = 0;
        }
        __syncthreads();
        const int work = item[0];
        const int kind = item[1];
        __syncthreads();
        if (work == -1) break;
        if (kind == 1) {
            hub2_produce_block<LAZY, DIRECT>(st, (uint32_t)work, n_stream, ssrc, sw, sslot, slen, snap, hub_giant, gblk, gprod,
                                             gflag, srow0, spr_g, slice_w_g);
            continue;
        }
        const uint32_t hub = (uint32_t)work / slices_g;              // giant-major: the longest giant's slices first
        const int slice = (int)((uint32_t)work - hub * slices_g);
        const int r = slice / spr_g;                     // source row 0..L-1 -> target layer r+1
        const int c0 = (slice - r * spr_g) * slice_w_g;  // first column of the slice inside the row
        const int width = min(rs, c0 + slice_w_g) - c0;
        const int head = (int)hub_giant[hub];
        const int len = (int)slen[head];
        const int nblk = (len + kStreamBlock - 1) / kStreamBlock;
        if (width > 0) {
            if (warp >= 1) {
                hub2_stream_feed(warp, lane, item + 2, gblk[hub], gflag, gprod, err, nblk, blk_base, len, (uint32_t)head, slice,
                                 (int)slices_g, ring, full, empty);
            } else {
                const uint32_t key = skey[head];
                const bool active = lane < width;
                float* const tptr = st.data + (long long)key * st.node_stride + (long long)(r + 1) * rs + c0 + lane;
                float acc = 0.f;
                if (active) {
                    acc = *tptr;                               // zeros if never written
                    if (LAZY) {
                        const int ts = st.stamps[(long long)key * L + r];
                        if (ts >= 0) acc = __fmul_rn(acc, decay_factor(st, r, ts));
                    }
                }
                acc = hub2_giant_chain(acc, ring, full, empty, blk_base, nblk, len, lane, lane, work == 0);
                if (active) *tptr = acc;
            }
            blk_base += (uint32_t)nblk;
        }
    }
}

__host__ __device__ inline size_t hub2_smem_bytes() {
    return (size_t)kHub2Stages * (32 * kHub2SlotFloats * 4 + 16) + 16;
}

template <bool LAZY, bool DIRECT>
__global__ void __launch_bounds__(kHub2Threads, 2)
walk_hub2_kernel(StateView st, const uint32_t* __restrict__ skey, const uint32_t* __restrict__ ssrc,
                 const float* __restrict__ sw, const uint32_t* __restrict__ sslot,
                 const uint32_t* __restrict__ slen, const float* __restrict__ snap,
                 const uint32_t* __restrict__ hub_giant, const uint32_t* __restrict__ hub_reg,
                 uint32_t* __restrict__ ctr, int spr_g, int slice_w_g, int spr_r, int slice_w_r, DecayArgs dnow,
                 const uint32_t* __restrict__ hub_len, const uint32_t* __restrict__ hub_part,
                 float* __restrict__ partial, int chunked, int srow0) {
    extern __shared__ __align__(128) unsigned char hub2_raw[];
    float* const ring = reinterpret_cast<float*>(hub2_raw);                       // [stages][32][kHub2SlotFloats]
    uint64_t* const full = reinterpret_cast<uint64_t*>(ring + (size_t)kHub2Stages * 32 * kHub2SlotFloats);
    uint64_t* const empty = full + kHub2Stages;
    int* const item = reinterpret_cast<int*>(empty + kHub2Stages);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int L = st.num_layer;
    const int rs = (int)st.row_stride;
    if (threadIdx.x == 0) {
        for (int i = 0; i < kHub2Stages; ++i) {
            mbar_init(&full[i], 32);                   // every lane of the producer warp arrives after its stores
            mbar_init(&empty[i], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        *item = (smid < 256u && atomicAdd(&ctr[kCtrSmClaim + smid], 1u) == 0u) ? 1 : 0;
    }
    __syncthreads();
    const bool prefer_giant = *item != 0;          // this CTA holds its SM's giant-segment slot
    __syncthreads();
    // giants [0, n_stream) of the sorted list belong to walk_stream_kernel (0 in chunked mode: no giant ordering)
    const uint32_t n_stream = ctr[kCtrStream];
    const uint32_t n_giant = ctr[kCtrGiant] - n_stream, n_reg = ctr[kCtrHub];
    const uint32_t slices_g = (uint32_t)(L * spr_g), slices_r = (uint32_t)(L * spr_r);
    // chunked accumulation: giants were expanded into chunk entries of the regular list (payload_kernel)
    const uint32_t total_g = chunked ? 0u : n_giant * slices_g, total_r = n_reg * slices_r;
    uint32_t blk_base = 0;      // ring blocks produced / consumed so far by this CTA (same count in every warp)
    for (;;) {
        if (threadIdx.x == 0) {
            int w = -1;          // >= 0: giant item, <= -2: regular item -(w + 2), -1: nothing left
            if (prefer_giant && total_g > 0) {
                const uint32_t g = atomicAdd(&ctr[kCtrHub2Giant], 1u);
                if (g < total_g) w = (int)g;
            }
            if (w == -1 && total_r > 0) {
                const uint32_t q = atomicAdd(&ctr[kCtrHub2Work], 1u);
                if (q < total_r) w = -(int)q - 2;
            }
            *item = w;
        }
        __syncthreads();
        const int work = *item;
        __syncthreads();
        if (work == -1) break;
        const bool giant = work >= 0;
        const uint32_t idx = giant ? (uint32_t)work : (uint32_t)(-(work + 2));
        const int spr = giant ? spr_g : spr_r;
        const int slice_w = giant ? slice_w_g : slice_w_r;
        const uint32_t slices = giant ? slices_g : slices_r;
        const uint32_t hub_i = idx / slices;
        const int slice = (int)(idx - hub_i * slices);
        const uint32_t hub = giant ? hub_i + n_stream : hub_i;
        const int r = slice / spr;                      // source row 0..L-1 -> target layer r+1
        const int c0 = (slice - r * spr) * slice_w;     // first column of the slice inside the row
        const int width = min(rs, c0 + slice_w) - c0;   // floats, multiple of 4
        const int head = (int)(giant ? hub_giant[hub] : hub_reg[hub]);
        const int len = (int)(giant ? slen[head] : hub_len[hub]);
        const uint32_t part = giant ? kNoPart : hub_part[hub];     // != kNoPart: a chunk of a giant -> its partial row
        const uint32_t key = skey[head];
        // a ring stage (8 KB) holds 32 messages of <= 64 floats, or — giants — 128 messages of <= 16 floats:
        // four times fewer full/empty handshakes on the critical chain
        const int spm = giant ? kGiantSpm : 1;          // 32-message sub-blocks per stage
        const int slot = giant ? kHub2GiantFloats : kHub2SlotFloats;      // floats between messages of a stage
        const int mps = 32 * spm;                       // messages per stage
        const int nblk = (len + mps - 1) / mps;
        if (width > 0) {
            if (warp >= 1) {
                // ------------------------------------------------ producers
                const int pw = warp - 1;
                const int nvec = width >> 2;            // 16-byte pieces per message (<= 4 giant, <= 16 otherwise)
                const int lpm_shift = giant ? kGiantLs : 4;    // lanes per message: 4 (8) or 16
                const int grp = lane >> lpm_shift, sub = lane & ((1 << lpm_shift) - 1);
                const int mpi = 32 >> lpm_shift;              // messages per load instruction: 8 (giant) or 2
                auto row_ptr = [&](uint32_t v, uint32_t x) -> const float* {
                    if (DIRECT && (x & kDirect) != 0)         // received row: rows 0..L-1 contiguous in the state
                        return st.data + (long long)v * st.node_stride + (long long)r * rs + c0;
                    if (r < srow0) return st.data + (long long)v * st.node_stride + c0;         // P_0: never written
                    return snap + (long long)x * (long long)(L - srow0) * rs + (long long)(r - srow0) * rs + c0;
                };
                for (int b = pw; b < nblk; b += kHub2Producers) {
                    const uint32_t g = blk_base + (uint32_t)b;
                    const uint32_t use = g / (uint32_t)kHub2Stages;
                    const int stage = (int)(g - use * (uint32_t)kHub2Stages);
                    const int pass = b / kHub2Producers;
                    (void)pass;                       // only the timeline build reads it
                    HUB2_STAMP(pass, 0);
                    // (1) metadata of this lane's message in each sub-block of the stage (all in flight together)
                    unsigned plo[kGiantSpmMax], phi[kGiantSpmMax];
                    float wl[kGiantSpmMax], fl[kGiantSpmMax];
#pragma unroll
                    for (int sb = 0; sb < kGiantSpmMax; ++sb) {
                        const int j = (b * spm + sb) * 32 + lane;
                        const float* ptr = st.data;
                        wl[sb] = 0.f;
                        fl[sb] = 1.0f;
                        if (sb < spm && j < len) {
                            const uint32_t v = ssrc[head + j];
                            const uint32_t x = (r >= srow0 || DIRECT) ? sslot[head + j] : 0u;
                            float w = sw[head + j];
                            if (DIRECT) {                     // sign bit of the weight = "cached row of another rank"
                                if (LAZY && r >= 1 && __float_as_int(w) < 0) {
                                    // it carries its own stamp: stamp -> this call's epoch in one multiply
                                    const int sst = st.stamps[(long long)v * L + (r - 1)];
                                    if (sst >= 0) fl[sb] = decay_factor(st, r - 1, sst);
                                }
                                w = fabsf(w);
                            }
                            wl[sb] = w;
                            ptr = row_ptr(v, x);
                        }
                        const unsigned long long mine = reinterpret_cast<unsigned long long>(ptr);
                        plo[sb] = (unsigned)mine;
                        phi[sb] = (unsigned)(mine >> 32);
                    }
                    // (2) 16 load instructions in flight: the whole stage (32 x 64 floats or 128 x 16 floats)
                    const int nm = min(mps, len - b * mps);   // messages of this stage that exist
                    HUB2_STAMP(pass, 1);
                    float4 xv[16];
#pragma unroll
                    for (int q = 0; q < 16; ++q) {
                        const int sb = giant ? (q >> kGiantLs) : 0;
                        const int i = giant ? (q & ((1 << kGiantLs) - 1)) : q;
                        const int m = mpi * i + grp;                       // message inside the sub-block
                        const unsigned lo = __shfl_sync(0xffffffffu, giant ? plo[q >> kGiantLs] : plo[0], m);
                        const unsigned hi = __shfl_sync(0xffffffffu, giant ? phi[q >> kGiantLs] : phi[0], m);
                        const float* pj = reinterpret_cast<const float*>(((unsigned long long)hi << 32) | lo);
                        xv[q] = (sb * 32 + m < nm && sub < nvec) ? ld4(pj + sub * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                    // (3) the stage is free again? then scale and store
                    HUB2_STAMP(pass, 2);
                    if (use > 0) mbar_wait(&empty[stage], (use - 1u) & 1u);
                    HUB2_STAMP(pass, 3);
                    float* dst = ring + (size_t)stage * (32 * kHub2SlotFloats) + (size_t)grp * slot + sub * 4;
#ifdef TPN_HUB2_TIMELINE
                    if (xv[0].x == 12345.678f) HUB2_STAMP(pass, 7);      // touch the first row so that stamp 4 sees its arrival
                    HUB2_STAMP(pass, 4);
#endif
#pragma unroll
                    for (int q = 0; q < 16; ++q) {
                        const int sb = giant ? (q >> kGiantLs) : 0;
                        const int i = giant ? (q & ((1 << kGiantLs) - 1)) : q;
                        const int m = mpi * i + grp;
                        const float w = __shfl_sync(0xffffffffu, giant ? wl[q >> kGiantLs] : wl[0], m);
                        if (DIRECT) scale4(xv[q], __shfl_sync(0xffffffffu, giant ? fl[q >> kGiantLs] : fl[0], m));   // x * 1.0f is exact
                        scale4(xv[q], w);
                        if (sub < nvec) st4(dst + (size_t)(sb * 32 + mpi * i) * slot, xv[q]);
                    }
                    HUB2_STAMP(pass, 5);
                    mbar_arrive(&full[stage]);         // release: this lane's stores are visible to the waiter
                    HUB2_STAMP(pass, 6);
                }
            } else {
                // ------------------------------------------------ consumer
                // regular slices (<= 64 floats): 2 columns per lane; giant slices (<= 16 floats): ONE column
                // per lane — per message one LDS + one FADD, so the warp issues less than the 4-cycle
                // latency of the add chain it is bound by
                const int col = giant ? lane : 2 * lane;
                const bool active = col < width;
                float* tptr = part == kNoPart
                                  ? st.data + (long long)key * st.node_stride + (long long)(r + 1) * rs + c0 + col
                                  : partial + ((long long)part * L + r) * rs + c0 + col;
                float2 acc = make_float2(0.f, 0.f);
                if (active && part == kNoPart) {
                    if (giant) acc.x = *tptr;
                    else acc = *reinterpret_cast<const float2*>(tptr);      // zeros if never written
                    if (LAZY) {
                        const int ts = st.stamps[(long long)key * L + r];
                        if (ts >= 0) acc = mul2_rn(acc, decay_factor(st, r, ts));
                    }
                }
                for (int b = 0; b < nblk; ++b) {
                    const uint32_t g = blk_base + (uint32_t)b;
                    const uint32_t use = g / (uint32_t)kHub2Stages;
                    const int stage = (int)(g - use * (uint32_t)kHub2Stages);
                    HUB2_STAMP(b, 0);
                    mbar_wait(&full[stage], use & 1u);
                    HUB2_STAMP(b, 1);
                    const int nm = min(mps, len - b * mps);
                    const float* xs = ring + (size_t)stage * (32 * kHub2SlotFloats) + col;
                    int j0 = 0;
                    if (giant) {
                        for (; j0 + 32 <= nm; j0 += 32) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) acc.x = __fadd_rn(acc.x, xs[(j0 + j) * kHub2GiantFloats]);
                        }
                        for (; j0 < nm; ++j0) acc.x = __fadd_rn(acc.x, xs[j0 * kHub2GiantFloats]);
                    } else {
                        for (; j0 + 32 <= nm; j0 += 32) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                const float2 p = *reinterpret_cast<const float2*>(xs + (j0 + j) * kHub2SlotFloats);
                                acc.x = __fadd_rn(acc.x, p.x);
                                acc.y = __fadd_rn(acc.y, p.y);
                            }
                        }
                        for (; j0 < nm; ++j0) {
                            const float2 p = *reinterpret_cast<const float2*>(xs + j0 * kHub2SlotFloats);
                            acc.x = __fadd_rn(acc.x, p.x);
                            acc.y = __fadd_rn(acc.y, p.y);
                        }
                    }
                    HUB2_STAMP(b, 2);
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&empty[stage]);
                    HUB2_STAMP(b, 3);
                }
                if (active) {
                    if (giant) *tptr = acc.x;
                    else *reinterpret_cast<float2*>(tptr) = acc;
                }
            }
        }
        blk_base += (width > 0) ? (uint32_t)nblk : 0u;
    }
}

// Chunked accumulation order, second half: target row of giant g  <-  ((row * pending decay) + partial_0) + partial_1 ...
// in chunk order (partial_c = the chunk's messages summed in order from +0 by walk_hub2_kernel).  One CTA per giant,
// one column per thread; the chain is the number of chunks, not the number of messages.
template <bool LAZY>
__global__ void __launch_bounds__(256)
combine_giants_kernel(StateView st, const uint32_t* __restrict__ skey, const uint32_t* __restrict__ slen,
                      const uint32_t* __restrict__ hub_giant, const uint32_t* __restrict__ giant_cbase,
                      const uint32_t* __restrict__ ctr, const float* __restrict__ partial, int chunk) {
    const int L = st.num_layer;
    const int rs = (int)st.row_stride;
    const int span = L * rs;
    const uint32_t n_giant = ctr[kCtrGiant];
    for (uint32_t g = blockIdx.x; g < n_giant; g += gridDim.x) {
        const uint32_t head = hub_giant[g];
        const uint32_t key = skey[head];
        const uint32_t nch = (slen[head] + (uint32_t)chunk - 1u) / (uint32_t)chunk;
        const float* pbase = partial + (long long)giant_cbase[g] * span;
        float* trow = st.data + (long long)key * st.node_stride + rs;          // rows 1..L
        for (int col = threadIdx.x; col < span; col += blockDim.x) {
            const int r = col / rs;
            float acc = trow[col];                                               // zeros if never written
            if (LAZY) {
                const int ts = st.stamps[(long long)key * L + r];
                if (ts >= 0) acc = __fmul_rn(acc, decay_factor(st, r, ts));
            }
            uint32_t c = 0;
            for (; c + 4 <= nch; c += 4) {                                       // four loads in flight, adds in order
                const float p0 = pbase[(long long)(c + 0) * span + col], p1 = pbase[(long long)(c + 1) * span + col];
                const float p2 = pbase[(long long)(c + 2) * span + col], p3 = pbase[(long long)(c + 3) * span + col];
                acc = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(acc, p0), p1), p2), p3);
            }
            for (; c < nch; ++c) acc = __fadd_rn(acc, pbase[(long long)c * span + col]);
            trow[col] = acc;
        }
    }
}


template <bool DIRECT>
int launch_walk_hub2(const StateView& v, const Workspace& ws, bool lazy, const DecayArgs& dnow, int chunk, int srow0,
                     cudaStream_t stream) {
    static bool configured_tab[kMaxDevices];          // per device: the shared-memory opt-in is a device attribute
    bool& configured = configured_tab[g_dev_slot];
    const int smem = (int)hub2_smem_bytes();
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(walk_hub2_kernel<false, DIRECT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(walk_hub2_kernel<true, DIRECT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) {
            set_cuda_error(e);
            return TPN_ERR_CUDA;
        }
        configured = true;
    }
    const int rs = (int)v.row_stride;
    const int spr_r = (rs + kHub2SlotFloats - 1) / kHub2SlotFloats;       // slices per row: regular hubs (<= 64 floats)
    const int slice_w_r = (((rs + spr_r - 1) / spr_r) + 3) & ~3;
    const int spr_g = (rs + kHub2GiantFloats - 1) / kHub2GiantFloats;     // giants (<= 32 floats)
    const int slice_w_g = (((rs + spr_g - 1) / spr_g) + 3) & ~3;
    // 2 CTAs (88 KB of ring each) per SM.  One per SM — leaving half of every SM to the short-segment
    // walker from the start — was measured slower (0.62 vs 0.58 ms per 100k-edge step).
    const unsigned grid = (unsigned)device_sm_count() * 2;
    const int chunked = chunk > 0 ? 1 : 0;
    if (lazy)
        walk_hub2_kernel<true, DIRECT><<<grid, kHub2Threads, smem, stream>>>(v, ws.key_a, ws.ssrc, ws.sw, ws.sslot, ws.slen,
                                                                             ws.snap, ws.hub_giant, ws.hub_reg, ws.ctr,
                                                                             spr_g, slice_w_g, spr_r, slice_w_r, dnow,
                                                                             ws.hub_len, ws.hub_part, ws.partial, chunked,
                                                                             srow0);
    else
        walk_hub2_kernel<false, DIRECT><<<grid, kHub2Threads, smem, stream>>>(v, ws.key_a, ws.ssrc, ws.sw, ws.sslot, ws.slen,
                                                                              ws.snap, ws.hub_giant, ws.hub_reg, ws.ctr,
                                                                              spr_g, slice_w_g, spr_r, slice_w_r, dnow,
                                                                              ws.hub_len, ws.hub_part, ws.partial, chunked,
                                                                              srow0);
    if (chunked) {
        const unsigned cgrid = (unsigned)device_sm_count();
        if (lazy)
            combine_giants_kernel<true><<<cgrid, 256, 0, stream>>>(v, ws.key_a, ws.slen, ws.hub_giant, ws.giant_cbase,
                                                                   ws.ctr, ws.partial, chunk);
        else
            combine_giants_kernel<false><<<cgrid, 256, 0, stream>>>(v, ws.key_a, ws.slen, ws.hub_giant, ws.giant_cbase,
                                                                    ws.ctr, ws.partial, chunk);
    }
    return TPN_OK;
}

// Streamed giants: one launch; exits at once when the front end streamed nothing (ctr[kCtrStream] == 0).
template <bool DIRECT>
int launch_walk_stream(const StateView& v, const Workspace& ws, bool lazy, int srow0, int* err_flag_dev, cudaStream_t stream) {
    static bool configured_tab[kMaxDevices];
    bool& configured = configured_tab[g_dev_slot];
    const int smem = (int)hub2_smem_bytes();
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(walk_stream_kernel<false, DIRECT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(walk_stream_kernel<true, DIRECT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) {
            set_cuda_error(e);
            return TPN_ERR_CUDA;
        }
        configured = true;
    }
    const int rs = (int)v.row_stride;
    const int spr_g = (rs + kHub2GiantFloats - 1) / kHub2GiantFloats;
    const int slice_w_g = (((rs + spr_g - 1) / spr_g) + 3) & ~3;
    const unsigned grid = (unsigned)(device_sm_count() < 2 ? 2 : device_sm_count());      // >= 1 chaining CTA + ticket 0
    if (lazy)
        walk_stream_kernel<true, DIRECT><<<grid, kHub2Threads, smem, stream>>>(v, ws.key_a, ws.ssrc, ws.sw, ws.sslot, ws.slen,
                                                                               ws.snap, ws.hub_giant, ws.ctr, spr_g, slice_w_g,
                                                                               srow0, ws.gblk, ws.gprod, ws.gflag, err_flag_dev);
    else
        walk_stream_kernel<false, DIRECT><<<grid, kHub2Threads, smem, stream>>>(v, ws.key_a, ws.ssrc, ws.sw, ws.sslot, ws.slen,
                                                                                ws.snap, ws.hub_giant, ws.ctr, spr_g, slice_w_g,
                                                                                srow0, ws.gblk, ws.gprod, ws.gflag, err_flag_dev);
    return TPN_OK;
}

template <int V, bool DIRECT>
void launch_walk_small_v(const StateView& v, const Workspace& ws, int E, int ds4, int tiles, bool lazy,
                         const DecayArgs& dnow, int srow0, cudaStream_t stream) {
    long long want = ((long long)E + kSmallWalkThreads / 32 - 1) / (kSmallWalkThreads / 32);
    const long long cap = (long long)device_sm_count() * 2 * 2;      // two resident CTAs per SM, two waves
    dim3 grid((unsigned)(want < cap ? want : cap), (unsigned)tiles);
    if (lazy)
        walk_small_kernel<V, true, DIRECT><<<grid, kSmallWalkThreads, 0, stream>>>(v, ws.key_a, ws.ssrc, ws.sw, ws.sslot,
                                                                                   ws.slen, ws.snap, ws.small_heads, ws.ctr,
                                                                                   E, ds4, dnow, srow0);
    else
        walk_small_kernel<V, false, DIRECT><<<grid, kSmallWalkThreads, 0, stream>>>(v, ws.key_a, ws.ssrc, ws.sw, ws.sslot,
                                                                                    ws.slen, ws.snap, ws.small_heads, ws.ctr,
                                                                                    E, ds4, dnow, srow0);
}

template <bool DIRECT>
void launch_walk_small(const StateView& v, const Workspace& ws, int E, int ds4, bool lazy, const DecayArgs& dnow,
                       int srow0, cudaStream_t stream) {
    const int span4 = v.num_layer * ds4;
    int vpl = (span4 + 31) / 32;
    int tiles = 1;
    if (vpl > 6) {
        tiles = (vpl + 5) / 6;
        vpl = (vpl + tiles - 1) / tiles;
    }
    switch (vpl) {
        case 1: launch_walk_small_v<1, DIRECT>(v, ws, E, ds4, tiles, lazy, dnow, srow0, stream); break;
        case 2: launch_walk_small_v<2, DIRECT>(v, ws, E, ds4, tiles, lazy, dnow, srow0, stream); break;
        case 3: launch_walk_small_v<3, DIRECT>(v, ws, E, ds4, tiles, lazy, dnow, srow0, stream); break;
        case 4: launch_walk_small_v<4, DIRECT>(v, ws, E, ds4, tiles, lazy, dnow, srow0, stream); break;
        case 5: launch_walk_small_v<5, DIRECT>(v, ws, E, ds4, tiles, lazy, dnow, srow0, stream); break;
        default: launch_walk_small_v<6, DIRECT>(v, ws, E, ds4, tiles, lazy, dnow, srow0, stream); break;
    }
}

// Library-owned side stream per device: the hub walker runs on it concurrently with the
// short-segment walker (disjoint target rows), forked from / joined back into the caller's stream
// with events, so the caller still sees one stream-ordered call (also valid under graph capture).
struct SideStream {
    cudaStream_t stream = nullptr;          // hub walker
    cudaStream_t stream2 = nullptr;         // streamed giants
    cudaEvent_t fork = nullptr, join = nullptr, join2 = nullptr;
    int state = 0;          // 0: not created, 1: ready, -1: creation failed (run serially)
};
SideStream* side_stream() {
    static SideStream table[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    SideStream& s = table[dev];
    if (s.state == 0) {
        bool ok = cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) == cudaSuccess;
        ok = ok && cudaStreamCreateWithFlags(&s.stream2, cudaStreamNonBlocking) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&s.join2, cudaEventDisableTiming) == cudaSuccess;
        if (!ok) (void)cudaGetLastError();
        s.state = ok ? 1 : -1;
    }
    return s.state == 1 ? &s : nullptr;
}

template <bool ALL>
int launch_walk_hub(const StateView& v, int layer, const Workspace& ws, int E4, bool lazy, const DecayArgs& dnow,
                    cudaStream_t stream) {
    static bool configured_tab[kMaxDevices];
    bool& configured = configured_tab[g_dev_slot];
    const int smem = (int)sizeof(HubSmem);
    if (!configured) {
        cudaError_t e = cudaSuccess;
        e = cudaFuncSetAttribute(walk_hub_kernel<false, ALL>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(walk_hub_kernel<true, ALL>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) {
            set_cuda_error(e);
            return TPN_ERR_CUDA;
        }
        configured = true;
    }
    const int rs = (int)v.row_stride;
    const int span = ALL ? v.num_layer * rs : rs;
    const int slices = (span + kHubSlotFloats - 1) / kHubSlotFloats;
    const int slice_w = (((span + slices - 1) / slices) + 3) & ~3;
    const uint32_t* xarr = ALL ? ws.sslot
                               : (lazy && layer >= 2 ? reinterpret_cast<const uint32_t*>(ws.svst) + (size_t)(layer - 2) * E4
                                                     : nullptr);
    const int work_ctr = kCtrWork0 + (ALL ? 0 : layer - 1);
    const unsigned grid = (unsigned)device_sm_count() * 2;
    if (lazy)
        walk_hub_kernel<true, ALL><<<grid, kHubThreads, smem, stream>>>(v, layer, ws.key_a, ws.ssrc, ws.sw, xarr, ws.slen,
                                                                        ws.snap, ws.hub_giant, ws.hub_reg, ws.ctr,
                                                                        work_ctr, span, slice_w, slices, dnow);
    else
        walk_hub_kernel<false, ALL><<<grid, kHubThreads, smem, stream>>>(v, layer, ws.key_a, ws.ssrc, ws.sw, xarr, ws.slen,
                                                                         ws.snap, ws.hub_giant, ws.hub_reg, ws.ctr,
                                                                         work_ctr, span, slice_w, slices, dnow);
    return TPN_OK;
}

template <int V, int D, bool ALL>
void launch_walk(const StateView& v, int layer, const Workspace& ws, Count E, int ds4, int tiles, bool lazy,
                 bool hubs, const DecayArgs& dnow, cudaStream_t stream, int srow0 = 1) {
    dim3 grid((unsigned)(((long long)E.cap * 32 + kWalkThreads - 1) / kWalkThreads), (unsigned)tiles);
    const int write_stamp = (!ALL && tiles == 1 && !hubs) ? 1 : 0;
    const int hub_min = hubs ? kHubMin : 0x7fffffff;
    if (lazy)
        walk_kernel<V, D, true, ALL><<<grid, kWalkThreads, 0, stream>>>(v, layer, ws.key_a, ws.ssrc, ws.sw, ws.sslot,
                                                                        ws.slen, ws.snap, E, ds4, write_stamp, hub_min, dnow,
                                                                        srow0);
    else
        walk_kernel<V, D, false, ALL><<<grid, kWalkThreads, 0, stream>>>(v, layer, ws.key_a, ws.ssrc, ws.sw, ws.sslot,
                                                                         ws.slen, ws.snap, E, ds4, write_stamp, hub_min, dnow,
                                                                         srow0);
}

}  // namespace

}  // namespace tpn

extern "C" size_t tpn_update_workspace_bytes(const tpn_state_t* st, int64_t batch) {
    if (batch < 1) batch = 1;
    if (st == nullptr) return 0;
    return tpn::carve(nullptr, batch, st->num_layer, st->row_stride).bytes;
}

namespace tpn {
namespace {

int update_impl(tpn_state_t* st, const MsgSource& msgs, int E, const int32_t* count_dev, int64_t ws_batch, double t_last,
                float neg_lambda, const float* decay, void* ws_dev, size_t ws_bytes, int32_t* err_flag_dev,
                cudaStream_t stream, int phase = TPN_UPDATE_WHOLE) {
    // phase (tpn_update_phase): TPN_UPDATE_PREPARE launches only what does not write the state — the sort front end
    // and, in lazy mode, the pre-batch snapshot (the eager sweep writes the state, so an eager snapshot waits for
    // TPN_UPDATE_APPLY) — and leaves the caller's struct untouched; TPN_UPDATE_APPLY launches the rest with the same
    // arguments.  The two halves may run on different streams (the caller orders them) with reads of the state between.
    // E is the number of messages, or — count_dev != nullptr, routed calls of a sharded state — its upper bound
    const Count cnt{E, reinterpret_cast<const int*>(count_dev)};
    Workspace ws = carve(ws_dev, ws_batch, st->num_layer, st->row_stride);
    if (ws.bytes > ws_bytes) return TPN_ERR_WORKSPACE_TOO_SMALL;
    const bool lazy = st->stamps != nullptr;
    const int L = st->num_layer;

    DecayArgs dargs;
    dargs.has_decay = 0;
    for (int l = 0; l < TPN_MAX_LAYERS; ++l) dargs.c[l] = 1.0f;
    if (decay != nullptr) {
        bool all_one = true;
        for (int l = 0; l < L; ++l) {
            dargs.c[l] = decay[l];
            all_one = all_one && decay[l] == 1.0f;
        }
        dargs.has_decay = all_one ? 0 : 1;      // x * 1.0f == x exactly: nothing to do
    }
    long long new_epoch = st->epoch;
    double new_floor = st->cum_floor;
    if (lazy && dargs.has_decay) {
        if (st->epoch + 1 >= st->log_capacity) return TPN_ERR_LOG_FULL;
        // the log holds f64 cumulative products: restart it (materialise) long before they underflow
        double cmin = 1.0;
        for (int l = 0; l < L; ++l) cmin = dargs.c[l] < cmin ? (double)dargs.c[l] : cmin;
        new_floor = (st->epoch == 0 ? 1.0 : st->cum_floor);
        if (st->epoch > 0 && !(new_floor * cmin >= 1e-200)) return TPN_ERR_LOG_FULL;
        new_floor *= cmin;          // tiny (or 0) only right after a restart: the next epoch restarts again
        new_epoch = st->epoch + 1;
    }

    const int ds4 = (int)(st->row_stride / 4);
    const float t_last_f = (float)t_last;
    double* log_w = lazy ? st->decay_log : nullptr;
    // Snapshot + single all-layer launch whenever the snapshot fits.  Edge mode: every source is
    // also a target, so every source has a snapshot slot.  Message mode (sharded): sources that
    // are not targets of this call (received rows) are read straight from the state (kDirect).
    const bool force_per_layer = (g_debug_flags & TPN_DEBUG_PER_LAYER_WALK) != 0;      // test hook
    const bool snapshot_path = ws.has_snap && !(force_per_layer && !(count_dev == nullptr && E <= kSmallMaxMsgs));
    const bool small_path = count_dev == nullptr && E <= kSmallMaxMsgs;
    const bool hubs = !small_path;                  // the single-CTA sort path keeps everything in the warp walker
    const int E4 = (E + 3) & ~3;                    // layer stride of svst (keeps bulk copies 16-byte aligned)
    const bool eager_sweep = !lazy && dargs.has_decay;
    // chunked accumulation order of giant segments (snapshot path only; 0 = the reference's sequential order)
    int chunk = st->giant_chunk > 0 ? (int)st->giant_chunk : 0;
    if (chunk > 0 && chunk < kChunkMin) chunk = kChunkMin;
    if (chunk > kGiantMin) chunk = kGiantMin;
    chunk &= ~31;
    const long long sweep_total4 = st->num_nodes * (long long)L * ds4;
    // streamed giants (snapshot path, reference order): decided here so that both halves of a split call agree
    const int stream_mode = (ws.has_stream && chunk == 0 && (g_debug_flags & TPN_DEBUG_NO_STREAM) == 0)
                                ? ((g_debug_flags & TPN_DEBUG_STREAM_ALL) ? 2 : 1) : 0;

    // the kernels read the NEW epoch; the caller's struct is only advanced once every launch went through
    StateView view = make_view(st);
    view.epoch = new_epoch;

    const bool do_front = phase != TPN_UPDATE_APPLY;          // sort front end
    const bool do_rest = phase != TPN_UPDATE_PREPARE;          // everything that writes the state
    // the snapshot reads decayed pre-batch rows: lazy -> with the front end; eager -> after the sweep
    const bool snap_early = lazy && !small_path;
    if (small_path) {
        if (phase == TPN_UPDATE_PREPARE) return TPN_OK;        // single-CTA sort: nothing worth splitting
        SweepArgs sw_args;
        sw_args.total4 = eager_sweep ? sweep_total4 : 0;
        sw_args.ds4 = ds4;
        unsigned grid = 1;
        if (eager_sweep) {
            const long long want = (sweep_total4 + kPrepThreads - 1) / kPrepThreads;
            const long long cap = (long long)device_sm_count() * 4;
            grid += (unsigned)(want < cap ? (want < 1 ? 1 : want) : cap);
        }
        prep_small_kernel<<<grid, kPrepThreads, 0, stream>>>(msgs, E, t_last_f, neg_lambda, st->num_nodes, ws.key_a,
                                                             ws.ssrc, ws.sw, ws.sslot, ws.slen, err_flag_dev, log_w, L,
                                                             new_epoch, dargs, view, sw_args);
    } else if (do_front) {
        int bits = 0;
        while ((1ll << bits) <= st->num_nodes) ++bits;    // keys are in [0, num_nodes] (num_nodes = dropped)
        const int passes = (bits + 7) / 8;
        const int nblk = (E + kRadixTile - 1) / kRadixTile;
        struct { PrepArgs prep; PayloadArgs pay; } fa;
        fa.prep.msgs = msgs;
        fa.prep.count = cnt;
        fa.prep.t_last_f = t_last_f;
        fa.prep.neg_lambda = neg_lambda;
        fa.prep.num_nodes = st->num_nodes;
        fa.prep.w = ws.w;
        fa.prep.key = ws.key_a;
        fa.prep.val = ws.val_a;
        fa.prep.err_flag = err_flag_dev;
        fa.prep.decay_log = log_w;
        fa.prep.L = L;
        fa.prep.new_epoch = new_epoch;
        fa.prep.decay = dargs;
        fa.prep.ctr = ws.ctr;
        fa.pay.order = nullptr;
        fa.pay.skey = nullptr;
        fa.pay.key_out = ws.key_a;
        fa.pay.msgs = msgs;
        fa.pay.w = ws.w;
        fa.pay.count = cnt;
        fa.pay.ssrc = ws.ssrc;
        fa.pay.sw = ws.sw;
        fa.pay.sslot = snapshot_path ? ws.sslot : nullptr;
        fa.pay.slen = ws.slen;
        fa.pay.hub_giant = ws.hub_giant;
        fa.pay.hub_reg = ws.hub_reg;
        fa.pay.small_heads = ws.small_heads;
        fa.pay.ctr = ws.ctr;
        fa.pay.svst = (lazy && !snapshot_path && L >= 2) ? ws.svst : nullptr;
        fa.pay.stamps = st->stamps;
        fa.pay.L = L;
        fa.pay.E4 = E4;
        fa.pay.num_nodes = st->num_nodes;
        fa.pay.err_flag = err_flag_dev;
        fa.pay.hub_len = ws.hub_len;
        fa.pay.hub_part = ws.hub_part;
        fa.pay.giant_cbase = ws.giant_cbase;
        fa.pay.chunk = (snapshot_path && hubs) ? chunk : 0;
        const bool fused_front = (g_debug_flags & TPN_DEBUG_LEGACY_FRONT) == 0 && front_kernel_ok();
        if (fused_front) {
            // ONE cooperative launch (<= one CTA per SM): prep and every radix pass
            FrontArgs fr;
            fr.prep = fa.prep;
            fr.key_a = ws.key_a; fr.key_b = ws.key_b; fr.val_a = ws.val_a; fr.val_b = ws.val_b;
            fr.hist = ws.hist; fr.hist2 = ws.hist2; fr.bar = ws.bar;
            fr.passes = passes;
            const int sms = device_sm_count();
            const unsigned grid = (unsigned)(nblk < 1 ? 1 : (nblk < sms ? nblk : sms));
            void* kargs[] = {&fr};
            if (cudaMemsetAsync(ws.bar, 0, 4 * kBarWords, stream) != cudaSuccess ||
                cudaLaunchCooperativeKernel((const void*)front_kernel, dim3(grid), dim3(kRadixThreads), kargs, 0,
                                            stream) != cudaSuccess) {
                set_cuda_error(cudaGetLastError());
                return TPN_ERR_CUDA;
            }
            const bool odd = (passes & 1) != 0;
            fa.pay.order = odd ? ws.val_b : ws.val_a;
            fa.pay.skey = odd ? ws.key_b : ws.key_a;     // odd number of passes: sorted keys in key_b; payload copies them
            payload_kernel<<<(E + 255) / 256, 256, 0, stream>>>(fa.pay);
            if (snapshot_path && chunk == 0) {
                sort_giants_kernel<<<1, 1024, 0, stream>>>(ws.hub_giant, ws.slen, ws.ctr, ws.gblk, ws.gflag, cnt, stream_mode);
            }
        } else
        {
            // >= 2 blocks: the first kCtrSlots threads also zero the per-call counters
            prep_large_kernel<<<(unsigned)((E + 255) / 256 < 2 ? 2 : (E + 255) / 256), 256, 0, stream>>>(fa.prep);
            uint32_t *kin = ws.key_a, *kout = ws.key_b, *vin = ws.val_a, *vout = ws.val_b;
            for (int p = 0; p < passes; ++p) {
                radix_hist_kernel<<<nblk, kRadixThreads, 0, stream>>>(kin, cnt, 8 * p, ws.hist);
                // few tiles: the scatter sums the columns itself (a device-side count always takes the prefix kernel)
                const int prefixed = (nblk > kRadixDirectBlocks || count_dev != nullptr) ? 1 : 0;
                if (prefixed) radix_prefix_kernel<<<kRadixBins / 8, 256, 0, stream>>>(ws.hist, cnt);
                radix_scatter_kernel<<<nblk, kRadixThreads, 0, stream>>>(kin, vin, kout, vout, cnt, 8 * p, ws.hist,
                                                                         prefixed);
                uint32_t* tk = kin; kin = kout; kout = tk;
                uint32_t* tv = vin; vin = vout; vout = tv;
            }
            fa.pay.order = vin;
            fa.pay.skey = kin;          // odd number of passes: sorted keys live in key_b; payload copies them to key_a
            payload_kernel<<<(E + 255) / 256, 256, 0, stream>>>(fa.pay);
            if (snapshot_path && chunk == 0) {
                sort_giants_kernel<<<1, 1024, 0, stream>>>(ws.hub_giant, ws.slen, ws.ctr, ws.gblk, ws.gflag, cnt, stream_mode);
            }
        }
    }
    if (!small_path && do_rest && eager_sweep) {
        const long long want = (sweep_total4 + 255) / 256;
        const long long cap = (long long)device_sm_count() * 16;
        const unsigned grid = (unsigned)(want < cap ? (want < 1 ? 1 : want) : cap);
        sweep_decay_kernel<<<grid, 256, 0, stream>>>(view, dargs, sweep_total4, ds4);
    }

    // first source row that is read from the pre-batch snapshot: 1 (P_0 is never written: read in place), or —
    // TPN_DEBUG_SNAPSHOT_P0 — 0: the snapshot also holds P_0, so every source read of the walkers hits one compact buffer
    const int srow0 = (g_debug_flags & TPN_DEBUG_SNAPSHOT_P0) ? 0 : 1;
    if (snapshot_path) {
        if (L - srow0 >= 1 && (snap_early ? do_front : do_rest)) {
            const unsigned grid = (unsigned)(((long long)E * 32 + 255) / 256);
            if (lazy) snapshot_kernel<true><<<grid, 256, 0, stream>>>(view, ws.key_a, cnt, ds4, ws.snap, srow0);
            else snapshot_kernel<false><<<grid, 256, 0, stream>>>(view, ws.key_a, cnt, ds4, ws.snap, srow0);
        }
        if (!do_rest) {
            // TPN_UPDATE_PREPARE ends here
        } else if (hubs) {
            // large batch: long segments on the CTA-pipelined hub walker, short ones on the
            // persistent warp walker (disjoint target rows; both read only pre-batch values)
            const bool direct = msgs.B == 0;
            SideStream* side = (g_debug_flags & TPN_DEBUG_SERIAL_WALK) ? nullptr : side_stream();
            cudaStream_t hub_stream = stream, giant_stream = stream;
            if (side != nullptr) {
                if (cudaEventRecord(side->fork, stream) == cudaSuccess &&
                    cudaStreamWaitEvent(side->stream, side->fork, 0) == cudaSuccess) {
                    hub_stream = side->stream;
                    if (stream_mode > 0 && cudaStreamWaitEvent(side->stream2, side->fork, 0) == cudaSuccess)
                        giant_stream = side->stream2;
                } else {
                    (void)cudaGetLastError();
                }
            }
            if (stream_mode > 0) {
                // first: its chains are the critical path when anything is streamed; otherwise it exits at once
                const int src = direct ? launch_walk_stream<true>(view, ws, lazy, srow0, err_flag_dev, giant_stream)
                                       : launch_walk_stream<false>(view, ws, lazy, srow0, err_flag_dev, giant_stream);
                if (src != TPN_OK) return src;
            }
            const int hrc = direct ? launch_walk_hub2<true>(view, ws, lazy, dargs, chunk, srow0, hub_stream)
                                   : launch_walk_hub2<false>(view, ws, lazy, dargs, chunk, srow0, hub_stream);
            if (hrc != TPN_OK) return hrc;
            if (direct) launch_walk_small<true>(view, ws, E, ds4, lazy, dargs, srow0, stream);
            else launch_walk_small<false>(view, ws, E, ds4, lazy, dargs, srow0, stream);
            if (hub_stream != stream) {
                bool ok = cudaEventRecord(side->join, hub_stream) == cudaSuccess &&
                          cudaStreamWaitEvent(stream, side->join, 0) == cudaSuccess;
                if (giant_stream != stream)
                    ok = ok && cudaEventRecord(side->join2, giant_stream) == cudaSuccess &&
                         cudaStreamWaitEvent(stream, side->join2, 0) == cudaSuccess;
                if (!ok) {
                    set_cuda_error(cudaGetLastError());
                    return TPN_ERR_CUDA;
                }
            }
        } else {
            // single-CTA sort path: one float4 per lane, a warp covers 512 contiguous bytes of the span
            const int span4 = L * ds4;
            launch_walk<1, 16, true>(view, 0, ws, cnt, ds4, (span4 + 31) / 32, lazy, false, dargs, stream, srow0);
        }
        if (lazy && do_rest) stamp_targets_kernel<<<(E + 255) / 256, 256, 0, stream>>>(view, 0, ws.key_a, cnt);
    } else if (do_rest) {
        // per-layer walk: V float4 per lane so that one tile covers rows up to 512 floats
        int vpl = (ds4 + 31) / 32;
        int tiles = 1;
        if (vpl > 4) {
            tiles = (vpl + 3) / 4;
            vpl = 4;
        }
        for (int layer = L; layer >= 1; --layer) {
            if (hubs) {
                const int hrc = launch_walk_hub<false>(view, layer, ws, E4, lazy, dargs, stream);
                if (hrc != TPN_OK) return hrc;
            }
            switch (vpl) {
                case 1: launch_walk<1, 16, false>(view, layer, ws, cnt, ds4, tiles, lazy, hubs, dargs, stream); break;
                case 2: launch_walk<2, 8, false>(view, layer, ws, cnt, ds4, tiles, lazy, hubs, dargs, stream); break;
                case 3: launch_walk<3, 4, false>(view, layer, ws, cnt, ds4, tiles, lazy, hubs, dargs, stream); break;
                default: launch_walk<4, 4, false>(view, layer, ws, cnt, ds4, tiles, lazy, hubs, dargs, stream); break;
            }
            if (lazy && (tiles > 1 || hubs))
                stamp_targets_kernel<<<(E + 255) / 256, 256, 0, stream>>>(view, layer, ws.key_a, cnt);
        }
    }
    const int lrc = check_launch();
    if (lrc == TPN_OK && do_rest) {
        st->epoch = new_epoch;
        st->cum_floor = new_floor;
    }
    return lrc;
}

}  // namespace
}  // namespace tpn

#ifdef TPN_HUB2_TIMELINE
extern "C" int tpn_debug_hub_timeline(unsigned long long* host_out, size_t count) {
    const size_t have = sizeof(tpn::g_hub2_timeline) / sizeof(unsigned long long);
    if (host_out == nullptr || count > have) return TPN_ERR_INVALID_ARGUMENT;
    return cudaMemcpyFromSymbol(host_out, tpn::g_hub2_timeline, count * sizeof(unsigned long long)) == cudaSuccess
               ? TPN_OK : TPN_ERR_CUDA;
}
#endif

namespace tpn {
int debug_flags() { return g_debug_flags; }
}  // namespace tpn

extern "C" int tpn_set_debug_flags(int flags) {
    const int old = tpn::g_debug_flags;
    tpn::g_debug_flags = flags;
    return old;
}

extern "C" int tpn_update(tpn_state_t* st, const int64_t* src_dev, const int64_t* dst_dev, const double* t_dev,
                          int64_t batch, double t_last, float neg_lambda, const float* decay, void* ws_dev,
                          size_t ws_bytes, int32_t* err_flag_dev, void* stream_v) {
    using namespace tpn;
    int rc = validate_state(st);
    if (rc != TPN_OK) return rc;
    if (batch < 1 || batch > ((int64_t)1 << 26) || src_dev == nullptr || dst_dev == nullptr || t_dev == nullptr ||
        ws_dev == nullptr || st->num_nodes >= (int64_t)0xffffffffll)
        return TPN_ERR_INVALID_ARGUMENT;
    DeviceScope scope(st->data);
    g_dev_slot = scope.slot();
    MsgSource msgs;
    msgs.a = reinterpret_cast<const long long*>(src_dev);
    msgs.b = reinterpret_cast<const long long*>(dst_dev);
    msgs.t = t_dev;
    msgs.B = batch;
    msgs.direct_from = st->num_nodes;
    return update_impl(st, msgs, (int)(2 * batch), nullptr, batch, t_last, neg_lambda, decay, ws_dev, ws_bytes,
                       err_flag_dev, reinterpret_cast<cudaStream_t>(stream_v));
}

extern "C" int tpn_update_phase(tpn_state_t* st, const int64_t* src_dev, const int64_t* dst_dev, const double* t_dev,
                                int64_t batch, double t_last, float neg_lambda, const float* decay, void* ws_dev,
                                size_t ws_bytes, int32_t* err_flag_dev, void* stream_v, int phase) {
    using namespace tpn;
    int rc = validate_state(st);
    if (rc != TPN_OK) return rc;
    if (batch < 1 || batch > ((int64_t)1 << 26) || src_dev == nullptr || dst_dev == nullptr || t_dev == nullptr ||
        ws_dev == nullptr || st->num_nodes >= (int64_t)0xffffffffll || phase < TPN_UPDATE_WHOLE || phase > TPN_UPDATE_APPLY)
        return TPN_ERR_INVALID_ARGUMENT;
    DeviceScope scope(st->data);
    g_dev_slot = scope.slot();
    MsgSource msgs;
    msgs.a = reinterpret_cast<const long long*>(src_dev);
    msgs.b = reinterpret_cast<const long long*>(dst_dev);
    msgs.t = t_dev;
    msgs.B = batch;
    msgs.direct_from = st->num_nodes;
    return update_impl(st, msgs, (int)(2 * batch), nullptr, batch, t_last, neg_lambda, decay, ws_dev, ws_bytes,
                       err_flag_dev, reinterpret_cast<cudaStream_t>(stream_v), phase);
}

extern "C" int tpn_update_messages(tpn_state_t* st, const int64_t* tgt_dev, const int64_t* src_dev,
                                   const double* t_dev, int64_t num_messages, const int32_t* num_messages_dev,
                                   int64_t num_local_rows, double t_last, float neg_lambda, const float* decay,
                                   void* ws_dev, size_t ws_bytes, int32_t* err_flag_dev, void* stream_v) {
    using namespace tpn;
    int rc = validate_state(st);
    if (rc != TPN_OK) return rc;
    if (num_messages < 1 || num_messages > ((int64_t)1 << 27) || tgt_dev == nullptr || src_dev == nullptr ||
        t_dev == nullptr || ws_dev == nullptr || st->num_nodes >= (int64_t)0x7fffffffll || num_local_rows < 0 ||
        num_local_rows > st->num_nodes)
        return TPN_ERR_INVALID_ARGUMENT;
    DeviceScope scope(st->data);
    g_dev_slot = scope.slot();
    MsgSource msgs;
    msgs.a = reinterpret_cast<const long long*>(tgt_dev);
    msgs.b = reinterpret_cast<const long long*>(src_dev);
    msgs.t = t_dev;
    msgs.B = 0;
    msgs.direct_from = num_local_rows;
    return update_impl(st, msgs, (int)num_messages, num_messages_dev, (num_messages + 1) / 2, t_last, neg_lambda,
                       decay, ws_dev, ws_bytes, err_flag_dev, reinterpret_cast<cudaStream_t>(stream_v));
}

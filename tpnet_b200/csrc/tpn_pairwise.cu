// tpn_pairwise — input of `self.mlp` in RandomProjectionModule.get_pair_wise_feature
// (reference: models/TPNet.py:112-129) for sm_100a.
//
// Per pair (a, b) the reference stacks the R = 2L+2 rows [a:P_0..P_L, b:P_0..P_L]
// (TPNet.py:119-121), forms the R x R Gram matrix with a batched fp32 GEMM (:122-123),
// clamps at 0 and takes log(x + 1.0) (:127-128).  The Gram blocks are 4x4 .. 10x10 over
// d ~ 100-200: ~3 flop/byte, far below the fp32 ridge, so this is a gather-bound kernel
// and tensor cores are deliberately not used.
//
// Mapping: G lanes per pair (G = 8: 4 pairs per warp, throughput shape; G = 32: one pair
// per warp, latency shape for the small decoder calls).  Lane j of a group reads float4
// columns j, j+G, ... of all R rows (the group reads G*16 contiguous bytes per row per
// step; a node's L+1 rows are one contiguous block in the node-major state) and keeps the
// R(R+1)/2 unique dot products in registers as packed (even, odd) float2 partial sums fed
// by the sm_100 packed FFMA2.  The sums are reduced over the group with a transposing
// butterfly (each shuffle step halves the number of live values), so every lane ends up
// owning NP/G finished entries, applies the epilogue to just those and mirrors them
// through shared memory; the warp then writes its pairs' R*R outputs as coalesced
// 128-bit streaming stores.
// Lazy-decay mode: rows of layers >= 1 are brought current in registers (one multiply by the
// row's pending decay factor) before they enter the products; nothing is written back.
#include <cuda.h>
#include <cudaTypedefs.h>
#include <string.h>

#include <mutex>

#include "tpn_pairwise.cuh"

namespace tpn {
namespace {

thread_local int g_dev_slot = 0;      // device of the call in progress (set by the entry point)


template <int LAYERS, int G, bool LAZY>
__global__ void __launch_bounds__(kPairThreads)
pairwise_kernel(StateView st, const long long* __restrict__ a_ids, const long long* __restrict__ b_ids,
                long long n, int apply_log_scale, float* __restrict__ out, int ds4, const int* __restrict__ n_dev) {
    if (n_dev != nullptr) {                // routed calls: the count lives on the device
        if (*n_dev > n && st.err != nullptr) *st.err = 4;       // more pairs than the call was sized for
        n = min(n, (long long)max(*n_dev, 0));
    }
    constexpr int H = LAYERS + 1;          // rows per endpoint
    constexpr int R = 2 * H;               // rows per pair
    constexpr int F = R * R;               // outputs per pair
    constexpr int NU = R * (R + 1) / 2;    // unique Gram entries
    constexpr int PPW = 32 / G;            // pairs per warp
    __shared__ __align__(16) float tile[kPairThreads / 32][PPW * F];
    __shared__ unsigned short tab[kPairThreads / 32][NU];

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int sub = lane / G;              // pair slot inside the warp
    const int gl = lane % G;               // lane inside the group
    const long long pair0 = ((long long)blockIdx.x * (kPairThreads / 32) + warp) * PPW;
    if (pair0 >= n) return;                // whole warp out of range
    const long long pair = pair0 + sub;
    const long long pc = pair < n ? pair : n - 1;          // inactive groups redo the last pair, never store

    long long ida = a_ids[pc], idb = b_ids[pc];
    fill_entry_table<R>(tab[warp], lane);
    // ids are validated on the host for numpy inputs; clamp so a bad device id can never fault
    ida = resolve_id(st, ida, true);
    idb = resolve_id(st, idb, true);
    const int rs4 = (int)(st.row_stride >> 2);
    const float4* pa = reinterpret_cast<const float4*>(st.data + ida * st.node_stride);
    const float4* pb = reinterpret_cast<const float4*>(st.data + idb * st.node_stride);

    // lazy decay: one pending factor per row (stamp < 0: the row is all zero in memory)
    float fac[R];
    if (LAZY) {
#pragma unroll
        for (int l = 1; l < H; ++l) {
            const long long sa = st.stamps[ida * LAYERS + (l - 1)];
            const long long sb = st.stamps[idb * LAYERS + (l - 1)];
            fac[l] = sa >= 0 ? decay_factor(st, l - 1, sa) : 1.0f;
            fac[H + l] = sb >= 0 ? decay_factor(st, l - 1, sb) : 1.0f;
        }
    }

    float2 acc[NU];
#pragma unroll
    for (int i = 0; i < NU; ++i) acc[i] = make_float2(0.f, 0.f);

    for (int c = gl; c < ds4; c += G) {
        float4 x[R];
#pragma unroll
        for (int l = 0; l < H; ++l) {
            x[l] = pa[l * rs4 + c];
            x[H + l] = pb[l * rs4 + c];
        }
        if (LAZY) {
#pragma unroll
            for (int l = 1; l < H; ++l) {
                scale4(x[l], fac[l]);
                scale4(x[H + l], fac[H + l]);
            }
        }
        gram_step<R>(acc, x);
    }

    __syncwarp();                          // entry table written by this warp is visible
    finish_pair<R, G>(acc, gl, &tile[warp][sub * F], tab[warp], apply_log_scale);
    __syncwarp();
    // coalesced write-out of the warp's pairs: PPW*F floats, contiguous in `out`
    const long long left = n - pair0;
    const int valid = (int)(left < PPW ? left : PPW) * F;     // multiple of 4 (F = 4 H^2)
    float* dst = out + pair0 * F;
    const float* srcs = &tile[warp][0];
    for (int i = lane * 4; i < valid; i += 32 * 4) {
        const float4 v = *reinterpret_cast<const float4*>(srcs + i);
        __stcs(reinterpret_cast<float4*>(dst + i), v);
    }
}

// ---------------------------------------------------------------- TMA (bulk-copy) variant
// Same math, different data movement: the L+1 rows of a node are ONE contiguous block of
// (L+1)*row_stride*4 bytes in the node-major state, so a warp fetches everything its 4 pairs
// need with at most 8 `cp.async.bulk` copies (global -> shared, completion counted on a
// per-warp mbarrier) issued by one lane.  The whole working set of the warp is in flight at
// once (no per-lane load instructions, no register staging, no dependent round trips per
// column step), and b-endpoints repeated by consecutive pairs — the encoder's pair lists
// repeat each b K times (TPNet.py:313-316) — are fetched once per warp.
template <int LAYERS, bool LAZY>
__global__ void __launch_bounds__(kPairThreads)
pairwise_tma_kernel(StateView st, const long long* __restrict__ a_ids, const long long* __restrict__ b_ids,
                    long long n, int apply_log_scale, float* __restrict__ out, int ds4, const int* __restrict__ n_dev) {
    if (n_dev != nullptr) {
        if (*n_dev > n && st.err != nullptr) *st.err = 4;
        n = min(n, (long long)max(*n_dev, 0));
    }
    constexpr int G = 8;
    constexpr int H = LAYERS + 1;
    constexpr int R = 2 * H;
    constexpr int F = R * R;
    constexpr int NU = R * (R + 1) / 2;
    constexpr int PPW = 4;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t mbar[kPairThreads / 32];
    __shared__ unsigned short tab[kPairThreads / 32][NU];

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int sub = lane / G;
    const int gl = lane % G;
    const long long pair0 = ((long long)blockIdx.x * (kPairThreads / 32) + warp) * PPW;
    if (pair0 >= n) return;
    const long long pair = pair0 + sub;
    const long long pc = pair < n ? pair : n - 1;

    long long ida = a_ids[pc], idb = b_ids[pc];
    uint64_t* bar = &mbar[warp];
    if (lane == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fill_entry_table<R>(tab[warp], lane);
    ida = resolve_id(st, ida, true);
    idb = resolve_id(st, idb, true);

    const int rs4 = (int)(st.row_stride >> 2);
    const uint32_t block_bytes = (uint32_t)(H * st.row_stride * 4);       // rows P_0..P_L of one node
    unsigned char* wbase = smem_raw + (size_t)warp * (2 * PPW) * block_bytes;

    // b endpoints of the warp's 4 pairs; a run of equal ids shares one slot
    long long bid[PPW];
#pragma unroll
    for (int s = 0; s < PPW; ++s) bid[s] = __shfl_sync(0xffffffffu, idb, s * G);
    int sb = sub;
#pragma unroll
    for (int s = PPW - 1; s >= 1; --s)
        if (sb == s && bid[s] == bid[s - 1]) sb = s - 1;
    __syncwarp();
    if (lane == 0) {
        uint32_t copies = PPW;
#pragma unroll
        for (int s = 0; s < PPW; ++s) copies += (s == 0 || bid[s] != bid[s - 1]) ? 1u : 0u;
        mbar_expect_tx(bar, copies * block_bytes);
    }
    __syncwarp();                                   // expect_tx is registered before any copy can complete
    // lanes 0, 8, 16, 24 own one pair each: fetch its a block, and its b block unless shared
    if (gl == 0) {
        bulk_g2s(wbase + (size_t)sub * block_bytes, st.data + ida * st.node_stride, block_bytes, bar);
        if (sb == sub)
            bulk_g2s(wbase + (size_t)(PPW + sub) * block_bytes, st.data + idb * st.node_stride, block_bytes, bar);
    }

    // lazy decay: one pending factor per row (stamp < 0: the row is all zero in memory)
    float fac[R];
    if (LAZY) {
#pragma unroll
        for (int l = 1; l < H; ++l) {
            const long long sa = st.stamps[ida * LAYERS + (l - 1)];
            const long long sb = st.stamps[idb * LAYERS + (l - 1)];
            fac[l] = sa >= 0 ? decay_factor(st, l - 1, sa) : 1.0f;
            fac[H + l] = sb >= 0 ? decay_factor(st, l - 1, sb) : 1.0f;
        }
    }
    float2 acc[NU];
#pragma unroll
    for (int i = 0; i < NU; ++i) acc[i] = make_float2(0.f, 0.f);

    const float4* pa = reinterpret_cast<const float4*>(wbase + (size_t)sub * block_bytes);
    const float4* pb = reinterpret_cast<const float4*>(wbase + (size_t)(PPW + sb) * block_bytes);
    mbar_wait(bar, 0);

    for (int c = gl; c < ds4; c += G) {
        float4 x[R];
#pragma unroll
        for (int l = 0; l < H; ++l) {
            x[l] = pa[l * rs4 + c];
            x[H + l] = pb[l * rs4 + c];
        }
        if (LAZY) {
#pragma unroll
            for (int l = 1; l < H; ++l) {
                scale4(x[l], fac[l]);
                scale4(x[H + l], fac[H + l]);
            }
        }
        gram_step<R>(acc, x);
    }

    __syncwarp();                                   // every lane is done reading the row buffers
    float* tile = reinterpret_cast<float*>(wbase);  // reuse them as the output staging tile
    finish_pair<R, G>(acc, gl, tile + sub * F, tab[warp], apply_log_scale);
    __syncwarp();
    const long long left = n - pair0;
    const int valid = (int)(left < PPW ? left : PPW) * F;
    float* dst = out + pair0 * F;
    for (int i = lane * 4; i < valid; i += 32 * 4) {
        const float4 v = *reinterpret_cast<const float4*>(tile + i);
        __stcs(reinterpret_cast<float4*>(dst + i), v);
    }
}

// ---------------------------------------------------------------- pipelined (column-chunk ring) variant
// The TMA kernel's warp fetches one 4-pair tile, waits for all of it, computes and exits: its copies are in flight
// only while it is not computing, which leaves HBM idle for most of a tile's lifetime.  Here the warps are
// persistent (warp w of W takes tiles w, w+W, ...) and every tile is staged in K column chunks, chunk j = float4
// columns [col0_j, col0_j + w_j), each in its own buffer with its own mbarrier.  As soon as the warp has computed
// chunk j of tile i, it issues chunk j of tile i+1 into the same buffer, so while it computes chunk j the other
// K-1 chunks (the rest of tile i, the start of tile i+1) are in flight.  Shared memory per warp is what the TMA
// kernel uses (8 node blocks), so the same number of warps stays resident.
// Lane gl of a group still visits columns gl, gl+8, ... in increasing order (the walk continues from one chunk into
// the next), so every accumulator sees the same operations in the same order: the output is bit-identical.
// The L+1 chunk-rows of a block are not contiguous, so one chunk of a block is ONE 3-D tensor-map copy (box
// {columns of the chunk, L+1 rows, 1 node} over the state viewed as [node][row][column]): at most 8 copies per
// chunk, issued by lanes 0..7.  One 1-D bulk copy per half-row (32 per half tile) measured slower than the TMA
// kernel on a B200 (137.9 against 116.3 us per 100,000-pair call; profiles/pairwise_pipeline_b200.json).
// K = 2 is the fastest measured: 3 and 4 chunks (more, smaller copies per tile) took 117.9 and 120.4 us, CTAs of
// 8 warps 107.8 us, against 106.6 us (B200; profiles/pairwise_pipeline_b200.json).
#ifndef TPN_PAIRWISE_CHUNKS
#define TPN_PAIRWISE_CHUNKS 2          // K; other values are for A/B builds (TPN_EXTRA_NVCC_FLAGS)
#endif
#ifndef TPN_PAIRWISE_CTA_WARPS
#define TPN_PAIRWISE_CTA_WARPS 4       // warps per CTA of the pipelined kernel (A/B builds: 8)
#endif
constexpr int kPipeChunks = TPN_PAIRWISE_CHUNKS;
constexpr int kPipeWarps = TPN_PAIRWISE_CTA_WARPS;
constexpr size_t kPipeSmemPerWarp = 110 * 1024 / 4;     // the TMA kernel's staging per warp

struct PipeChunks {
    int col0[kPipeChunks];             // first float4 column of chunk j
    int w[kPipeChunks];                // float4 columns of chunk j
    int buf4[kPipeChunks];             // float4 offset of chunk j's buffer in the warp's region
    int slot4[kPipeChunks];            // float4 stride of one slot (node block) in chunk j's buffer
    int warp4;                         // float4 size of one warp's region
};
struct PipeMaps {
    CUtensorMap m[kPipeChunks];        // box {4 * w[j], L+1, 1}
};

struct PipeTile {
    long long ida, idb;                // resolved ids of this lane's pair
    int sb;                            // slot of this lane's b block after dedup
    uint32_t nblk;                     // blocks actually fetched (4 + distinct b)
    int node;                          // lanes 0..7: node of slot `lane`, -1: none
};

__device__ __forceinline__ void pipe_prepare(const StateView& st, long long ida, long long idb, int lane, PipeTile& t) {
    constexpr int G = 8, PPW = 4;
    t.ida = resolve_id(st, ida, true);
    t.idb = resolve_id(st, idb, true);
    long long bid[PPW];
#pragma unroll
    for (int s = 0; s < PPW; ++s) bid[s] = __shfl_sync(0xffffffffu, t.idb, s * G);
    const int sub = lane / G;
    int sb = sub;
#pragma unroll
    for (int s = PPW - 1; s >= 1; --s)
        if (sb == s && bid[s] == bid[s - 1]) sb = s - 1;
    t.sb = sb;
    uint32_t nblk = PPW;
#pragma unroll
    for (int s = 0; s < PPW; ++s) nblk += (s == 0 || bid[s] != bid[s - 1]) ? 1u : 0u;
    t.nblk = nblk;
    // slot = lane: 0..3 are the a blocks, 4..7 the b blocks (skipped when shared)
    const int owner = (lane & (PPW - 1)) * G;
    const long long ia = __shfl_sync(0xffffffffu, t.ida, owner);
    const long long ib = __shfl_sync(0xffffffffu, t.idb, owner);
    const int osb = __shfl_sync(0xffffffffu, sb, owner);
    t.node = lane < PPW ? (int)ia : (lane < 2 * PPW && osb == lane - PPW) ? (int)ib : -1;
}

// Stages float4 columns [col0, col0 + w) of every block of the tile into `buf` (slot s at buf + s * slot4).
// The caller has synced the warp after its last read of `buf`.
__device__ __forceinline__ void pipe_issue(const PipeTile& t, const CUtensorMap* map, float4* buf, int slot4,
                                           uint64_t* bar, int H, int col0, int w, int lane) {
    if (lane == 0) mbar_expect_tx(bar, t.nblk * (uint32_t)(H * w * 16));
    __syncwarp();                                           // expect_tx is registered before any copy can complete
    if (t.node >= 0)
        asm volatile(
            "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
            ::"r"(smem_u32(buf + (size_t)lane * slot4)), "l"(reinterpret_cast<uint64_t>(map)), "r"(4 * col0), "r"(0),
              "r"(t.node), "r"(smem_u32(bar))
            : "memory");
}

template <int LAYERS, bool LAZY>
__device__ __forceinline__ void pipe_factors(const StateView& st, long long ida, long long idb, float (&fac)[2 * (LAYERS + 1)]) {
    constexpr int H = LAYERS + 1;
    if (LAZY) {
#pragma unroll
        for (int l = 1; l < H; ++l) {
            const long long sa = st.stamps[ida * LAYERS + (l - 1)];
            const long long sb = st.stamps[idb * LAYERS + (l - 1)];
            fac[l] = sa >= 0 ? decay_factor(st, l - 1, sa) : 1.0f;
            fac[H + l] = sb >= 0 ? decay_factor(st, l - 1, sb) : 1.0f;
        }
    }
}

// float4 stride of one slot of a chunk buffer: tensor copies land on 128-byte boundaries
inline int pipe_slot4(int H, int w) { return (H * w + 7) & ~7; }

template <int LAYERS, bool LAZY>
__global__ void __launch_bounds__(kPipeWarps * 32)
pairwise_pipe_kernel(StateView st, const long long* __restrict__ a_ids, const long long* __restrict__ b_ids,
                     long long n, int apply_log_scale, float* __restrict__ out, int ds4, const PipeChunks ck,
                     const __grid_constant__ PipeMaps maps, const int* __restrict__ n_dev) {
    if (n_dev != nullptr) {
        if (*n_dev > n && st.err != nullptr) *st.err = 4;
        n = min(n, (long long)max(*n_dev, 0));
    }
    constexpr int G = 8;
    constexpr int H = LAYERS + 1;
    constexpr int R = 2 * H;
    constexpr int F = R * R;
    constexpr int NU = R * (R + 1) / 2;
    constexpr int PPW = 4;
    constexpr int K = kPipeChunks;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t mbar[kPipeWarps][K];
    __shared__ unsigned short tab[kPipeWarps][NU];

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int sub = lane / G;
    const int gl = lane % G;
    const long long tiles = (n + PPW - 1) / PPW;
    const long long tstride = (long long)gridDim.x * kPipeWarps;
    long long t = (long long)blockIdx.x * kPipeWarps + warp;
    if (t >= tiles) return;

    float4* region = reinterpret_cast<float4*>(smem_raw) + (size_t)warp * ck.warp4;
    if (lane == 0) {
#pragma unroll
        for (int j = 0; j < K; ++j) mbar_init(&mbar[warp][j], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fill_entry_table<R>(tab[warp], lane);
    __syncwarp();

    PipeTile cur;
    float fac[R];
    {
        const long long pc = min(t * PPW + sub, n - 1);     // inactive groups redo the last pair, never store
        pipe_prepare(st, a_ids[pc], b_ids[pc], lane, cur);
#pragma unroll
        for (int j = 0; j < K; ++j)
            pipe_issue(cur, &maps.m[j], region + ck.buf4[j], ck.slot4[j], &mbar[warp][j], H, ck.col0[j], ck.w[j], lane);
        pipe_factors<LAYERS, LAZY>(st, cur.ida, cur.idb, fac);
    }
    for (uint32_t phase = 0;; phase ^= 1u) {
        const long long tn = t + tstride;
        const bool more = tn < tiles;                       // warp-uniform
        long long na = 0, nb = 0;
        if (more) {                                         // in flight during the wait for chunk 0
            const long long pc = min(tn * PPW + sub, n - 1);
            na = a_ids[pc];
            nb = b_ids[pc];
        }
        float2 acc[NU];
#pragma unroll
        for (int i = 0; i < NU; ++i) acc[i] = make_float2(0.f, 0.f);

        PipeTile nxt;
        float fac_n[R];
        int c = gl;
#pragma unroll
        for (int j = 0; j < K; ++j) {
            const float4* buf = region + ck.buf4[j];
            const float4* pa = buf + sub * ck.slot4[j];
            const float4* pb = buf + (PPW + cur.sb) * ck.slot4[j];
            const int w = ck.w[j], c0 = ck.col0[j];
            mbar_wait(&mbar[warp][j], phase);
            for (; c < c0 + w; c += G) {
                float4 x[R];
#pragma unroll
                for (int l = 0; l < H; ++l) {
                    x[l] = pa[l * w + (c - c0)];
                    x[H + l] = pb[l * w + (c - c0)];
                }
                if (LAZY) {
#pragma unroll
                    for (int l = 1; l < H; ++l) {
                        scale4(x[l], fac[l]);
                        scale4(x[H + l], fac[H + l]);
                    }
                }
                gram_step<R>(acc, x);
            }
            if (j < K - 1 && more) {
                if (j == 0) pipe_prepare(st, na, nb, lane, nxt);
                __syncwarp();                               // every lane is done reading chunk j
                pipe_issue(nxt, &maps.m[j], region + ck.buf4[j], ck.slot4[j], &mbar[warp][j], H, c0, w, lane);
                if (j == 0) pipe_factors<LAYERS, LAZY>(st, nxt.ida, nxt.idb, fac_n);
            }
        }

        __syncwarp();                                       // every lane is done reading the last chunk
        float* tile = reinterpret_cast<float*>(region + ck.buf4[K - 1]);   // reused as the output staging tile
        finish_pair<R, G>(acc, gl, tile + sub * F, tab[warp], apply_log_scale);
        __syncwarp();
        const long long pair0 = t * PPW;
        const long long left = n - pair0;
        const int valid = (int)(left < PPW ? left : PPW) * F;
        float* dst = out + pair0 * F;
        for (int i = lane * 4; i < valid; i += 32 * 4) {
            const float4 v = *reinterpret_cast<const float4*>(tile + i);
            __stcs(reinterpret_cast<float4*>(dst + i), v);
        }
        if (!more) break;
        fence_proxy_async_smem();                           // the generic writes and reads of the tile come first
        __syncwarp();
        pipe_issue(nxt, &maps.m[K - 1], region + ck.buf4[K - 1], ck.slot4[K - 1], &mbar[warp][K - 1], H,
                   ck.col0[K - 1], ck.w[K - 1], lane);
        cur = nxt;
#pragma unroll
        for (int i = 0; i < R; ++i) fac[i] = fac_n[i];
        t = tn;
    }
}

// The state as a [num_nodes][H][row_stride] fp32 tensor, box {4 * w columns, H rows, 1 node}.
bool encode_chunk_map(CUtensorMap* map, const StateView& v, int H, int w) {
    static const PFN_cuTensorMapEncodeTiled_v12000 encode = [] {      // thread-safe one-time lookup
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess) {
            (void)cudaGetLastError();
            fn = nullptr;
        }
        return reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
    }();
    if (encode == nullptr) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)v.row_stride, (cuuint64_t)H, (cuuint64_t)v.num_nodes};
    const cuuint64_t strides[2] = {(cuuint64_t)v.row_stride * 4, (cuuint64_t)v.node_stride * 4};
    const cuuint32_t box[3] = {(cuuint32_t)(4 * w), (cuuint32_t)H, 1};
    const cuuint32_t elem[3] = {1, 1, 1};
    return encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, v.data, dims, strides, box, elem, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Chunk widths: ds4 split as evenly as possible, each width nudged (by up to 3 columns) to the one that wastes the
// least shared memory on slot alignment.  Returns the staging bytes of one warp.
size_t pipe_layout(int H, int ds4, PipeChunks& ck) {
    int col = 0, off = 0;
    for (int j = 0; j < kPipeChunks; ++j) {
        const int left = ds4 - col, parts = kPipeChunks - j;
        int w = (left + parts - 1) / parts;
        if (j < kPipeChunks - 1) {
            int best = w;
            for (int x = w; x <= w + 3 && x < left - (parts - 1) + 1; ++x)
                if (pipe_slot4(H, x) - H * x < pipe_slot4(H, best) - H * best) best = x;
            w = best;
        } else {
            w = left;
        }
        ck.col0[j] = col;
        ck.w[j] = w;
        ck.slot4[j] = pipe_slot4(H, w);
        ck.buf4[j] = off;
        off += 8 * ck.slot4[j];
        col += w;
    }
    ck.warp4 = off;
    return (size_t)off * 16;
}

// Host state of one (device, mode): the attribute opt-in, the occupancy at the last staging size, and the tensor
// maps of the last state / layout (a launch re-encodes only when the state or the row layout changed).
struct PipeHost {
    bool configured = false;
    size_t occ_smem = 0;
    int occ_per_sm = 0;
    const void* map_data = nullptr;
    long long map_nodes = -1, map_rs = -1, map_ns = -1;
    PipeChunks map_ck{};
    PipeMaps maps;
};
std::mutex g_pipe_mutex;                                    // in-process ranks may launch from several threads

template <int LAYERS>
bool launch_pipe(const StateView& v, const long long* a, const long long* b, long long n, const int* n_dev, int scale,
                 float* out, cudaStream_t s) {
    constexpr int H = LAYERS + 1;
    constexpr int R = 2 * H;
    const int ds4 = (int)(v.row_stride / 4);
    if (ds4 < kPipeChunks) return false;
    PipeChunks ck;
    const size_t per_warp = pipe_layout(H, ds4, ck);
    const size_t smem = (size_t)kPipeWarps * per_warp;
    // same staging per warp as the TMA kernel (>= 8 warps per SM); the staging tile (4 pairs * R*R floats) aliases
    // the last chunk; tensor-map boxes are at most 256 elements wide and node ids are 32-bit coordinates
    bool fits = per_warp <= kPipeSmemPerWarp && 4 * R * R * sizeof(float) <= (size_t)8 * ck.slot4[kPipeChunks - 1] * 16 &&
                (v.node_stride & 3) == 0 && v.num_nodes <= INT32_MAX;
    for (int j = 0; j < kPipeChunks; ++j) fits = fits && ck.w[j] >= 1 && 4 * ck.w[j] <= 256;
    if (!fits) return false;
    const bool lazy = v.stamps != nullptr;
    auto kernel = lazy ? pairwise_pipe_kernel<LAYERS, true> : pairwise_pipe_kernel<LAYERS, false>;
    static PipeHost hosts[kMaxDevices][2];                  // per instantiation: the attributes are per kernel
    std::lock_guard<std::mutex> lock(g_pipe_mutex);
    PipeHost& hs = hosts[g_dev_slot][lazy ? 1 : 0];
    if (!hs.configured) {
        if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)(kPipeWarps * kPipeSmemPerWarp)) != cudaSuccess) {
            (void)cudaGetLastError();
            return false;
        }
        hs.configured = true;
    }
    if (hs.occ_smem != smem) {                              // persistent warps: one CTA per resident slot
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kPipeWarps * 32, smem) != cudaSuccess ||
            per_sm < 1) {
            (void)cudaGetLastError();
            return false;
        }
        hs.occ_smem = smem;
        hs.occ_per_sm = per_sm;
    }
    if (hs.map_data != v.data || hs.map_nodes != v.num_nodes || hs.map_rs != v.row_stride || hs.map_ns != v.node_stride ||
        memcmp(&hs.map_ck, &ck, sizeof ck) != 0) {
        hs.map_data = nullptr;
        for (int j = 0; j < kPipeChunks; ++j)
            if (!encode_chunk_map(&hs.maps.m[j], v, H, ck.w[j])) return false;
        hs.map_data = v.data;
        hs.map_nodes = v.num_nodes;
        hs.map_rs = v.row_stride;
        hs.map_ns = v.node_stride;
        hs.map_ck = ck;
    }
    const long long ctas_needed = (n + 4 * kPipeWarps - 1) / (4 * kPipeWarps);
    const long long resident_ctas = (long long)hs.occ_per_sm * device_sm_count();
    const unsigned grid = (unsigned)(ctas_needed < resident_ctas ? ctas_needed : resident_ctas);
    kernel<<<grid, kPipeWarps * 32, smem, s>>>(v, a, b, n, scale, out, ds4, ck, hs.maps, n_dev);
    return true;
}

template <int LAYERS>
bool launch_tma(const StateView& v, const long long* a, const long long* b, long long n, const int* n_dev, int scale, float* out,
                cudaStream_t s) {
    constexpr int R = 2 * (LAYERS + 1);
    const size_t block_bytes = (size_t)(LAYERS + 1) * v.row_stride * 4;
    const size_t smem = (size_t)(kPairThreads / 32) * 8 * block_bytes;
    // the staging tile (4 pairs * R*R floats) aliases the row buffers; keep >= 2 CTAs per SM
    if (smem > 110 * 1024 || 4 * R * R * sizeof(float) > 8 * block_bytes || (block_bytes & 15) != 0 ||
        (v.node_stride & 3) != 0)
        return false;
    static bool configured_tab[kMaxDevices][2];          // per device: the opt-in is a per-device attribute
    bool* configured = configured_tab[g_dev_slot];
    const bool lazy = v.stamps != nullptr;
    auto kernel = lazy ? pairwise_tma_kernel<LAYERS, true> : pairwise_tma_kernel<LAYERS, false>;
    if (!configured[lazy ? 1 : 0]) {
        if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024) != cudaSuccess) {
            (void)cudaGetLastError();
            return false;
        }
        configured[lazy ? 1 : 0] = true;
    }
    const unsigned grid = (unsigned)((n + 15) / 16);
    kernel<<<grid, kPairThreads, smem, s>>>(v, a, b, n, scale, out, (int)(v.row_stride / 4), n_dev);
    return true;
}

template <int LAYERS, int G>
void launch_g(const StateView& v, const long long* a, const long long* b, long long n, const int* n_dev, int scale, float* out,
              cudaStream_t s) {
    constexpr int pairs_per_block = kPairThreads / G;
    const unsigned grid = (unsigned)((n + pairs_per_block - 1) / pairs_per_block);
    const int ds4 = (int)(v.row_stride / 4);
    if (v.stamps != nullptr)
        pairwise_kernel<LAYERS, G, true><<<grid, kPairThreads, 0, s>>>(v, a, b, n, scale, out, ds4, n_dev);
    else
        pairwise_kernel<LAYERS, G, false><<<grid, kPairThreads, 0, s>>>(v, a, b, n, scale, out, ds4, n_dev);
}

template <int LAYERS>
void launch(const StateView& v, const long long* a, const long long* b, long long n, const int* n_dev, int scale, float* out,
            cudaStream_t s) {
    // few pairs (decoder calls): one warp per pair fills more SMs and needs fewer
    // dependent round trips per pair; many pairs: 8 lanes per pair wastes no lanes on d ~ 140
    if (n <= 4096) {
        launch_g<LAYERS, 32>(v, a, b, n, n_dev, scale, out, s);
        return;
    }
    if ((debug_flags() & TPN_DEBUG_LEGACY_PAIRWISE) == 0 && launch_pipe<LAYERS>(v, a, b, n, n_dev, scale, out, s))
        return;
    // rows too narrow for the pipelined layout take the one-shot TMA kernel;
    // rows too wide for the shared-memory staging, the register kernel
    if (!launch_tma<LAYERS>(v, a, b, n, n_dev, scale, out, s))
        launch_g<LAYERS, 8>(v, a, b, n, n_dev, scale, out, s);
}

}  // namespace
}  // namespace tpn

extern "C" int tpn_pairwise(const tpn_state_t* st, const int64_t* a_ids_dev, const int64_t* b_ids_dev, int64_t n,
                            const int32_t* n_dev, int apply_log_scale, float* out_dev, void* stream_v) {
    using namespace tpn;
    int rc = validate_state(st);
    if (rc != TPN_OK) return rc;
    if (n < 0 || n > (int64_t)1 << 34) return TPN_ERR_INVALID_ARGUMENT;
    if (n == 0) return TPN_OK;
    if (a_ids_dev == nullptr || b_ids_dev == nullptr || out_dev == nullptr ||
        (reinterpret_cast<uintptr_t>(out_dev) & 15) != 0)
        return TPN_ERR_INVALID_ARGUMENT;
    DeviceScope scope(st->data);
    g_dev_slot = scope.slot();
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_v);
    const StateView v = make_view(st);
    const long long* a = reinterpret_cast<const long long*>(a_ids_dev);
    const long long* b = reinterpret_cast<const long long*>(b_ids_dev);
    const int* nd = reinterpret_cast<const int*>(n_dev);
    switch (st->num_layer) {
        case 1: launch<1>(v, a, b, n, nd, apply_log_scale, out_dev, stream); break;
        case 2: launch<2>(v, a, b, n, nd, apply_log_scale, out_dev, stream); break;
        case 3: launch<3>(v, a, b, n, nd, apply_log_scale, out_dev, stream); break;
        case 4: launch<4>(v, a, b, n, nd, apply_log_scale, out_dev, stream); break;
        default: return TPN_ERR_UNSUPPORTED;
    }
    return check_launch();
}

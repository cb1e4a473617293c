// tpn_route — device-side routing, remote-row pulls and the rank barrier of the node-sharded state
// (SURVEY.md 8(e); no reference counterpart: the reference is single-device).
//
// Rows of node u live on rank u % world at local row u / world.  The edge batch / pair list is replicated on
// every rank's device.  Per call, on every rank, with no host involvement and no device -> host copy:
//   route   : keep the work items this rank owns (target / first endpoint owned), in order (stable compaction:
//             block counts -> one-block scan -> scatter), translate ids to local rows, and give every REMOTE second
//             endpoint a slot in the extension rows behind the local rows.  Slots are handed out through a mark
//             table indexed by global node id (int atomics; a slot number only decides where a row is cached,
//             never a result) and stay valid until the next write to the state (one "generation"), so the
//             update that follows the pair-wise calls of the same batch finds its rows already cached.
//   nodes   : (tpn_route_nodes) a plain list of global ids, every one of them this rank's to read: each id gets a
//             row — its local row if owned, else a cache slot handed out through the same mark table.  No compaction.
//   pull    : one warp per new slot reads the row block of its node straight out of the owner's HBM over
//             NVLink (peer pointers, IPC-mapped) and stores it in the extension row TOGETHER WITH THE OWNER'S
//             STAMPS (lazy decay): a cached row is then read exactly like a local row — one multiply from its
//             stamp to the reader's epoch (every rank logs the same epochs), so sharded results equal the
//             single-GPU ones bit for bit.  Never-written rows (stamp < 0) are not read, just zero-filled.
//   barrier : one tiny kernel per rank; release-store of a sequence number into every peer's flag word, then
//             acquire-spin on the own flag words.  Orders "all pulls done" before "anyone writes" and "all
//             writes done" before the next pulls.  Bounded spin: a missing peer sets the error counter instead
//             of hanging the GPU.
// After these, the rank-local kernels (tpn_update_messages / tpn_pairwise with device-side counts) run unchanged.
#include <string.h>

#include "tpn_common.cuh"

namespace tpn {
namespace {

constexpr int kRouteThreads = 256;
constexpr int kRouteItems = 8;
constexpr int kRouteTile = kRouteThreads * kRouteItems;      // 2048 items per block

struct ShardView {
    int world, rank;
    long long global_nodes, n_local, ext_rows;
    const float* const* peer_data;
    const int* const* peer_stamps;
    unsigned* const* peer_flags;
    int* mark;
    int* counters;
    long long* need_nodes;
    unsigned* barrier_seq;
};

ShardView make_shard_view(const tpn_shard_t* sh) {
    ShardView v;
    v.world = sh->world;
    v.rank = sh->rank;
    v.global_nodes = sh->global_nodes;
    v.n_local = sh->num_local_rows;
    v.ext_rows = sh->ext_rows;
    v.peer_data = sh->peer_data;
    v.peer_stamps = reinterpret_cast<const int* const*>(sh->peer_stamps);
    v.peer_flags = reinterpret_cast<unsigned* const*>(sh->peer_flags);
    v.mark = sh->mark;
    v.counters = sh->counters;
    v.need_nodes = reinterpret_cast<long long*>(sh->need_nodes);
    v.barrier_seq = sh->barrier_seq;
    return v;
}

// Work items of a call.  Edge mode (B > 0): the 2B update messages of an edge batch in the reference's
// accumulation order — item m < B is (target src[m], source dst[m]), item m >= B is (target dst[m-B],
// source src[m-B]) (the two scatter_add_ of TPNet.py:93-96).  Pair mode (B == 0): item m is (a[m], b[m]).
struct Items {
    const long long* a;
    const long long* b;
    const double* t;       // edge mode: timestamps of the edges
    long long B;
    long long n;           // number of items (2B in edge mode)
    __device__ __forceinline__ void get(long long m, long long& first, long long& second) const {
        if (B > 0 && m >= B) {
            first = b[m - B];
            second = a[m - B];
        } else {
            first = a[m];
            second = b[m];
        }
    }
};

__device__ __forceinline__ bool owned(const ShardView& sh, long long first, long long second) {
    // an id outside the graph: the item is dropped and the error counter set (the host raises IndexError)
    if (first < 0 || first >= sh.global_nodes || second < 0 || second >= sh.global_nodes) {
        sh.counters[TPN_SHARD_CTR_ERROR] = 1;
        return false;
    }
    return (int)(first % sh.world) == sh.rank;
}

// Remembers where the new extension slots of a routing call start (counters[PREV] = counters[NEED]): run by one
// thread, in a launch that precedes every slot request of the call, so tpn_pull_rows fills exactly [PREV, NEED).
__device__ __forceinline__ void mark_call_start(const ShardView& sh) {
    const int need = sh.counters[TPN_SHARD_CTR_NEED];
    sh.counters[TPN_SHARD_CTR_PREV] = need < sh.ext_rows ? need : (int)sh.ext_rows;
}

// Remote node s is read by this call: make sure it has a cache slot in this generation.  Only the first request of a
// node claims one; the slot number is final once every request of the call has run (route_resolve_kernel, a later
// launch, reads it from the mark).
__device__ __forceinline__ void request_slot(const ShardView& sh, long long s) {
    // a hub is the second endpoint of a large share of the batch (18 % on the power-law bench): test with a
    // plain load first, so that only the requests that still see 0 — the first few — reach the atomic unit
    // (measured, 800,000 pairs of the N=8 job: 47 us with the compare-and-swap alone).  The mark only moves
    // 0 -> 1 -> slot + 2 within a generation, so a stale 0 just costs one failed compare-and-swap.
    if (__ldcg(&sh.mark[s]) == 0 && atomicCAS(&sh.mark[s], 0, 1) == 0) {   // first request of this node in the generation
        int slot = atomicAdd(&sh.counters[TPN_SHARD_CTR_NEED], 1);
        if (slot >= sh.ext_rows) {                    // cache full: flagged, the access stays in bounds
            sh.counters[TPN_SHARD_CTR_ERROR] = 2;
            slot = 0;
        } else {
            sh.need_nodes[slot] = s;
        }
        atomicExch(&sh.mark[s], slot + 2);
    }
}

__global__ void __launch_bounds__(kRouteThreads)
route_count_kernel(ShardView sh, Items it, int* __restrict__ block_counts) {
    __shared__ int wsum[kRouteThreads / 32];
    const long long base = (long long)blockIdx.x * kRouteTile;
    int mine = 0;
#pragma unroll
    for (int k = 0; k < kRouteItems; ++k) {
        const long long m = base + k * kRouteThreads + threadIdx.x;
        if (m < it.n) {
            long long f, s;
            it.get(m, f, s);
            mine += owned(sh, f, s) ? 1 : 0;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
        int tot = 0;
        for (int w = 0; w < kRouteThreads / 32; ++w) tot += wsum[w];
        block_counts[blockIdx.x] = tot;
    }
}

// one block: exclusive scan of the block counts in place, total -> *count_out; remembers where this call's new
// extension slots start (counters[PREV] = counters[NEED])
__global__ void __launch_bounds__(1024)
route_scan_kernel(ShardView sh, int* __restrict__ block_counts, int nblk, int* __restrict__ count_out) {
    __shared__ int wsum[32];
    __shared__ int carry_s;
    if (threadIdx.x == 0) {
        carry_s = 0;
        mark_call_start(sh);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int b0 = 0; b0 < nblk; b0 += 1024) {
        const int b = b0 + threadIdx.x;
        const int c = b < nblk ? block_counts[b] : 0;
        int inc = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int nb = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += nb;
        }
        if (lane == 31) wsum[warp] = inc;
        __syncthreads();
        int wbase = 0;
        for (int w = 0; w < warp; ++w) wbase += wsum[w];
        const int carry = carry_s;
        if (b < nblk) block_counts[b] = carry + wbase + inc - c;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = carry + wbase + inc;
        __syncthreads();
    }
    if (threadIdx.x == 0) *count_out = carry_s;
}

// stable compaction of the owned items + slot assignment of remote second endpoints.
// second_rows_out[pos] >= 0 : local row;  < 0 : -(global id) - 1, resolved by route_resolve_kernel.
__global__ void __launch_bounds__(kRouteThreads)
route_scatter_kernel(ShardView sh, Items it, const int* __restrict__ block_offsets, long long* __restrict__ first_rows_out,
                     long long* __restrict__ second_rows_out, long long* __restrict__ keep_out,
                     double* __restrict__ t_out) {
    __shared__ int wcount[kRouteThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long base = (long long)blockIdx.x * kRouteTile;
    int running = block_offsets[blockIdx.x];
#pragma unroll 1
    for (int k = 0; k < kRouteItems; ++k) {
        const long long m = base + k * kRouteThreads + threadIdx.x;
        long long f = 0, s = 0;
        bool mine = false;
        if (m < it.n) {
            it.get(m, f, s);
            mine = owned(sh, f, s);
        }
        const unsigned mask = __ballot_sync(0xffffffffu, mine);
        if (lane == 0) wcount[warp] = __popc(mask);
        __syncthreads();
        int before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < kRouteThreads / 32; ++w) {
            const int c = wcount[w];
            before += w < warp ? c : 0;
            total += c;
        }
        if (mine) {
            const int pos = running + before + __popc(mask & ((1u << lane) - 1u));
            first_rows_out[pos] = f / sh.world;
            if (keep_out != nullptr) keep_out[pos] = m;
            if (t_out != nullptr) t_out[pos] = it.t[it.B > 0 && m >= it.B ? m - it.B : m];
            long long row;
            if ((int)(s % sh.world) == sh.rank) {
                row = s / sh.world;
            } else {
                row = -s - 1;
                request_slot(sh, s);
            }
            second_rows_out[pos] = row;
        }
        running += total;
        __syncthreads();
    }
}

// rows < 0 (-(global id) - 1) -> n_local + the node's slot.  count: device item count, or NULL when all `cap` are valid.
__global__ void __launch_bounds__(256)
route_resolve_kernel(ShardView sh, long long* __restrict__ second_rows, const int* __restrict__ count, long long cap) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long n = count != nullptr ? *count : cap;
    n = n < cap ? n : cap;
    if (i >= n) return;
    const long long v = second_rows[i];
    if (v < 0) second_rows[i] = sh.n_local + (long long)(sh.mark[-v - 1] - 2);
}

// tpn_route_nodes, first launch: the start of this call's slots (one thread).
__global__ void __launch_bounds__(32) route_nodes_start_kernel(ShardView sh) {
    if (threadIdx.x == 0) mark_call_start(sh);
}

// tpn_route_nodes, second launch: every id of the list -> local row, or -(id) - 1 with a slot requested.
// An id outside the graph is flagged and maps to row 0.
__global__ void __launch_bounds__(256)
route_nodes_kernel(ShardView sh, const long long* __restrict__ ids, long long n, long long* __restrict__ rows_out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long u = ids[i];
    long long row;
    if (u < 0 || u >= sh.global_nodes) {
        sh.counters[TPN_SHARD_CTR_ERROR] = 1;
        row = 0;
    } else if ((int)(u % sh.world) == sh.rank) {
        row = u / sh.world;
    } else {
        row = -u - 1;
        request_slot(sh, u);
    }
    rows_out[i] = row;
}

// One warp per new extension slot: the owner's row block and stamps -> this rank's extension row.
template <bool LAZY>
__global__ void __launch_bounds__(256)
pull_rows_kernel(StateView st, ShardView sh, int ds4) {
    const int lane = threadIdx.x & 31;
    const int warps = gridDim.x * (blockDim.x >> 5);
    const int first = sh.counters[TPN_SHARD_CTR_PREV];
    int last = sh.counters[TPN_SHARD_CTR_NEED];
    last = last < sh.ext_rows ? last : (int)sh.ext_rows;
    const int L = st.num_layer;
    const int rows4 = (L + 1) * ds4;
    for (int slot = first + blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); slot < last; slot += warps) {
        const long long v = sh.need_nodes[slot];
        const int q = (int)(v % sh.world);
        const long long row = v / sh.world;
        const float* src = sh.peer_data[q] + row * st.node_stride;
        float* dst = st.data + (sh.n_local + slot) * st.node_stride;
        // lane l copies the owner's stamp of layer l + 1; a negative stamp marks a row that was never written
        // (all zero): it is not fetched
        float fmine = 1.0f;
        if (LAZY && lane < L) {
            const int stamp = sh.peer_stamps[q][row * L + lane];
            fmine = stamp >= 0 ? 1.0f : -1.0f;
            st.stamps[(sh.n_local + slot) * L + lane] = stamp;
        }
        float f[TPN_MAX_LAYERS + 1];
        f[0] = 1.0f;                                                         // P_0 always exists
#pragma unroll
        for (int l = 0; l < TPN_MAX_LAYERS; ++l) f[l + 1] = LAZY ? __shfl_sync(0xffffffffu, fmine, l) : 1.0f;
        for (int c0 = lane; c0 < rows4; c0 += 128) {                         // four 16-byte requests in flight per lane
            float4 x[4];
            float fk[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int c = c0 + 32 * k;
                const int li = c < rows4 ? c / ds4 : 0;
                fk[k] = li == 0 ? f[0] : (li == 1 ? f[1] : (li == 2 ? f[2] : (li == 3 ? f[3] : f[4])));
                x[k] = (c < rows4 && fk[k] >= 0.f) ? ld4(src + 4 * (long long)c) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int c = c0 + 32 * k;
                if (c < rows4) st4(dst + 4 * (long long)c, x[k]);
            }
        }
    }
}

__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// All ranks launch this in the same order.  Thread q tells rank q "I passed barrier #seq" and waits for rank q's
// word in the own flag array.  Signed distance compare: the sequence may wrap.
__global__ void __launch_bounds__(64)
peer_barrier_kernel(ShardView sh, long long spin_limit) {
    const int q = threadIdx.x;
    const unsigned seq = *sh.barrier_seq + 1u;
    __threadfence_system();
    if (q < sh.world) st_release_sys(sh.peer_flags[q] + sh.rank, seq);
    bool ok = true;
    if (q < sh.world) {
        const unsigned* mine = sh.peer_flags[sh.rank] + q;
        const long long t0 = clock64();
        while ((int)(ld_acquire_sys(mine) - seq) < 0) {
            if (clock64() - t0 > spin_limit) {
                ok = false;
                break;
            }
            __nanosleep(40);
        }
    }
    if (!ok) sh.counters[TPN_SHARD_CTR_ERROR] = 3;          // a peer never arrived: results are void, the GPU is not hung
    __syncthreads();
    __threadfence_system();
    if (threadIdx.x == 0) *sh.barrier_seq = seq;
}

int validate_shard(const tpn_shard_t* sh) {
    if (sh == nullptr || sh->world < 1 || sh->world > 64 || sh->rank < 0 || sh->rank >= sh->world ||
        sh->global_nodes < 1 || sh->global_nodes > 0x7fffffffll || sh->num_local_rows < 0 || sh->ext_rows < 0 ||
        sh->ext_rows > 0x7ffffff0ll || sh->mark == nullptr || sh->counters == nullptr || sh->need_nodes == nullptr)
        return TPN_ERR_INVALID_ARGUMENT;
    return TPN_OK;
}

int route_impl(const tpn_shard_t* sh, const Items& it, int64_t* first_rows, int64_t* second_rows, int64_t* keep,
               double* t_out, int32_t* count_out, void* ws_dev, size_t ws_bytes, cudaStream_t stream) {
    const long long nblk = (it.n + kRouteTile - 1) / kRouteTile;
    if (ws_bytes < (size_t)(nblk + 1) * sizeof(int)) return TPN_ERR_WORKSPACE_TOO_SMALL;
    int* block_counts = reinterpret_cast<int*>(ws_dev);
    const ShardView v = make_shard_view(sh);
    route_count_kernel<<<(unsigned)nblk, kRouteThreads, 0, stream>>>(v, it, block_counts);
    route_scan_kernel<<<1, 1024, 0, stream>>>(v, block_counts, (int)nblk, reinterpret_cast<int*>(count_out));
    route_scatter_kernel<<<(unsigned)nblk, kRouteThreads, 0, stream>>>(v, it, block_counts,
                                                                        reinterpret_cast<long long*>(first_rows),
                                                                        reinterpret_cast<long long*>(second_rows),
                                                                        reinterpret_cast<long long*>(keep), t_out);
    route_resolve_kernel<<<(unsigned)((it.n + 255) / 256), 256, 0, stream>>>(v, reinterpret_cast<long long*>(second_rows),
                                                                             reinterpret_cast<const int*>(count_out), it.n);
    return check_launch();
}

}  // namespace
}  // namespace tpn

extern "C" size_t tpn_route_workspace_bytes(int64_t items) {
    if (items < 1) items = 1;
    return (size_t)((items + tpn::kRouteTile - 1) / tpn::kRouteTile + 1) * sizeof(int) + 256;
}

extern "C" int tpn_route_update(const tpn_shard_t* sh, const int64_t* src_dev, const int64_t* dst_dev, const double* t_dev,
                                int64_t batch, int64_t* tgt_rows_out, int64_t* src_rows_out, double* t_out,
                                int32_t* count_out_dev, void* ws_dev, size_t ws_bytes, void* stream_v) {
    using namespace tpn;
    int rc = validate_shard(sh);
    if (rc != TPN_OK) return rc;
    if (batch < 1 || batch > ((int64_t)1 << 29) || src_dev == nullptr || dst_dev == nullptr || t_dev == nullptr ||
        tgt_rows_out == nullptr || src_rows_out == nullptr || t_out == nullptr || count_out_dev == nullptr ||
        ws_dev == nullptr)
        return TPN_ERR_INVALID_ARGUMENT;
    DeviceScope scope(sh->mark);
    Items it;
    it.a = reinterpret_cast<const long long*>(src_dev);
    it.b = reinterpret_cast<const long long*>(dst_dev);
    it.t = t_dev;
    it.B = batch;
    it.n = 2 * batch;
    return route_impl(sh, it, tgt_rows_out, src_rows_out, nullptr, t_out, count_out_dev, ws_dev, ws_bytes,
                      reinterpret_cast<cudaStream_t>(stream_v));
}

extern "C" int tpn_route_pairs(const tpn_shard_t* sh, const int64_t* a_dev, const int64_t* b_dev, int64_t n,
                               int64_t* a_rows_out, int64_t* b_rows_out, int64_t* keep_out, int32_t* count_out_dev,
                               void* ws_dev, size_t ws_bytes, void* stream_v) {
    using namespace tpn;
    int rc = validate_shard(sh);
    if (rc != TPN_OK) return rc;
    if (n < 1 || n > ((int64_t)1 << 30) || a_dev == nullptr || b_dev == nullptr || a_rows_out == nullptr ||
        b_rows_out == nullptr || count_out_dev == nullptr || ws_dev == nullptr)
        return TPN_ERR_INVALID_ARGUMENT;
    DeviceScope scope(sh->mark);
    Items it;
    it.a = reinterpret_cast<const long long*>(a_dev);
    it.b = reinterpret_cast<const long long*>(b_dev);
    it.t = nullptr;
    it.B = 0;
    it.n = n;
    return route_impl(sh, it, a_rows_out, b_rows_out, keep_out, nullptr, count_out_dev, ws_dev, ws_bytes,
                      reinterpret_cast<cudaStream_t>(stream_v));
}

extern "C" int tpn_route_nodes(const tpn_shard_t* sh, const int64_t* ids_dev, int64_t n, int64_t* rows_out_dev,
                               void* stream_v) {
    using namespace tpn;
    int rc = validate_shard(sh);
    if (rc != TPN_OK) return rc;
    if (n < 0 || n > ((int64_t)1 << 34) || (n > 0 && (ids_dev == nullptr || rows_out_dev == nullptr)))
        return TPN_ERR_INVALID_ARGUMENT;
    DeviceScope scope(sh->mark);
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_v);
    const ShardView v = make_shard_view(sh);
    // launched for an empty list too: the following tpn_pull_rows then has nothing to pull
    route_nodes_start_kernel<<<1, 32, 0, stream>>>(v);
    if (n > 0) {
        const unsigned grid = (unsigned)((n + 255) / 256);
        long long* rows = reinterpret_cast<long long*>(rows_out_dev);
        route_nodes_kernel<<<grid, 256, 0, stream>>>(v, reinterpret_cast<const long long*>(ids_dev), n, rows);
        route_resolve_kernel<<<grid, 256, 0, stream>>>(v, rows, nullptr, n);
    }
    return check_launch();
}

extern "C" int tpn_pull_rows(const tpn_state_t* st, const tpn_shard_t* sh, void* stream_v) {
    using namespace tpn;
    int rc = validate_state(st);
    if (rc != TPN_OK) return rc;
    rc = validate_shard(sh);
    if (rc != TPN_OK) return rc;
    if (sh->peer_data == nullptr || sh->num_local_rows + sh->ext_rows > st->num_nodes ||
        (st->stamps != nullptr && sh->peer_stamps == nullptr))
        return TPN_ERR_INVALID_ARGUMENT;
    if (sh->world == 1) return TPN_OK;
    DeviceScope scope(st->data);
    const StateView v = make_view(st);
    const ShardView s = make_shard_view(sh);
    const int ds4 = (int)(st->row_stride / 4);
    const unsigned grid = (unsigned)device_sm_count() * 4;
    if (v.stamps != nullptr) pull_rows_kernel<true><<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream_v)>>>(v, s, ds4);
    else pull_rows_kernel<false><<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream_v)>>>(v, s, ds4);
    return check_launch();
}

extern "C" int tpn_peer_barrier(const tpn_shard_t* sh, void* stream_v) {
    using namespace tpn;
    int rc = validate_shard(sh);
    if (rc != TPN_OK) return rc;
    if (sh->peer_flags == nullptr || sh->barrier_seq == nullptr) return TPN_ERR_INVALID_ARGUMENT;
    DeviceScope scope(sh->mark);
    // ~2 s of SM clock at 2 GHz (a constant: querying the clock rate costs about a millisecond of host time per call)
    const long long limit = 4000000000ll;
    peer_barrier_kernel<<<1, 64, 0, reinterpret_cast<cudaStream_t>(stream_v)>>>(make_shard_view(sh), limit);
    return check_launch();
}

extern "C" int tpn_shard_new_generation(const tpn_shard_t* sh, void* stream_v) {
    using namespace tpn;
    int rc = validate_shard(sh);
    if (rc != TPN_OK) return rc;
    DeviceScope scope(sh->mark);
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_v);
    cudaError_t e = cudaMemsetAsync(sh->mark, 0, sizeof(int32_t) * (size_t)sh->global_nodes, stream);
    // NEED and PREV restart; the error counter is sticky until the host reads it
    if (e == cudaSuccess) e = cudaMemsetAsync(sh->counters, 0, sizeof(int32_t) * 2, stream);
    if (e != cudaSuccess) {
        set_cuda_error(e);
        return TPN_ERR_CUDA;
    }
    return TPN_OK;
}

// ---------------------------------------------------------------- peer-visible memory (CUDA IPC)
extern "C" int tpn_peer_alloc(void** out, size_t bytes) {
    if (out == nullptr || bytes == 0) return TPN_ERR_INVALID_ARGUMENT;
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) e = cudaMemset(p, 0, bytes);
    if (e != cudaSuccess) {
        tpn::set_cuda_error(e);
        if (p != nullptr) cudaFree(p);
        return TPN_ERR_CUDA;
    }
    *out = p;
    return TPN_OK;
}

extern "C" int tpn_peer_free(void* p) {
    if (p == nullptr) return TPN_OK;
    tpn::DeviceScope scope(p);
    const cudaError_t e = cudaFree(p);
    if (e != cudaSuccess) {
        tpn::set_cuda_error(e);
        return TPN_ERR_CUDA;
    }
    return TPN_OK;
}

extern "C" int tpn_ipc_export(const void* p, unsigned char* handle64) {
    if (p == nullptr || handle64 == nullptr) return TPN_ERR_INVALID_ARGUMENT;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handles are 64 bytes");
    tpn::DeviceScope scope(p);
    cudaIpcMemHandle_t h;
    const cudaError_t e = cudaIpcGetMemHandle(&h, const_cast<void*>(p));
    if (e != cudaSuccess) {
        tpn::set_cuda_error(e);
        return TPN_ERR_CUDA;
    }
    memcpy(handle64, &h, 64);
    return TPN_OK;
}

extern "C" int tpn_ipc_open(const unsigned char* handle64, void** out) {
    if (handle64 == nullptr || out == nullptr) return TPN_ERR_INVALID_ARGUMENT;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    void* p = nullptr;
    // maps the exporting process's allocation into this process and enables peer access from the current device
    const cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
        tpn::set_cuda_error(e);
        return TPN_ERR_CUDA;
    }
    *out = p;
    return TPN_OK;
}

extern "C" int tpn_ipc_close(void* p) {
    if (p == nullptr) return TPN_OK;
    const cudaError_t e = cudaIpcCloseMemHandle(p);
    if (e != cudaSuccess) {
        tpn::set_cuda_error(e);
        return TPN_ERR_CUDA;
    }
    return TPN_OK;
}

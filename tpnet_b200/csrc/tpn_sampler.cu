// tpn_sampler — the reference's `recent` historical-neighbour sampler on the GPU
// (utils/utils.py:160-224, NeighborSampler.get_historical_neighbors with
// sample_neighbor_strategy == 'recent'; SURVEY.md 8(f) N2).
//
// The reference walks a Python loop over the batch: per (node, time) a np.searchsorted on the node's
// time-sorted adjacency and three slice copies — 5.5 ms per 400-row batch, the end-to-end bottleneck
// once the projections are fast.  Here the adjacency is one CSR on the device (built once per sampler
// by the host class: per node, entries stably sorted by timestamp) and a query is one warp:
//   i    = first entry of the node with time >= t            (searchsorted 'left': strictly before t)
//   take = min(i - begin, K) most recent entries before t, written to the BACK of a zero row
// Outputs (neighbour ids, edge ids, times; [n, K]) stay on the device, so the structured pair-wise call
// (tpn_pairwise_neighbors) can consume the ids without a host round trip.
#include "tpn_common.cuh"
#include "tpn_radix.cuh"

namespace tpn {
namespace {

__global__ void __launch_bounds__(256)
sampler_recent_kernel(const long long* __restrict__ offsets, const long long* __restrict__ nbr,
                      const long long* __restrict__ eid, const double* __restrict__ times, long long num_nodes,
                      const long long* __restrict__ q_nodes, const double* __restrict__ q_times, long long n, int K,
                      long long* __restrict__ out_nbr, long long* __restrict__ out_eid, double* __restrict__ out_t) {
    const long long q = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (q >= n) return;
    const long long node = q_nodes[q];
    const double t = q_times[q];
    long long begin = 0, end = 0;
    if (node >= 0 && node < num_nodes) {
        begin = offsets[node];
        end = offsets[node + 1];
    }
    long long a = begin, b = end;                   // every lane runs the same search (broadcast loads)
    while (a < b) {
        const long long mid = a + ((b - a) >> 1);
        if (times[mid] < t) a = mid + 1; else b = mid;
    }
    const long long cnt = a - begin;
    const int take = (int)(cnt < (long long)K ? cnt : (long long)K);
    const long long first = a - take;               // entries first .. a-1 are the `take` most recent before t
    const int pad = K - take;
    for (int j = lane; j < K; j += 32) {
        long long vn = 0, ve = 0;
        double vt = 0.0;
        if (j >= pad) {
            const long long s = first + (j - pad);
            vn = nbr[s];
            ve = eid[s];
            vt = times[s];
        }
        out_nbr[q * K + j] = vn;
        out_eid[q * K + j] = ve;
        out_t[q * K + j] = vt;
    }
}

}  // namespace
}  // namespace tpn

extern "C" int tpn_sampler_recent(const int64_t* offsets_dev, const int64_t* nbr_dev, const int64_t* eid_dev,
                                  const double* times_dev, int64_t num_nodes, const int64_t* q_nodes_dev,
                                  const double* q_times_dev, int64_t n, int num_neighbors, int64_t* out_nbr_dev,
                                  int64_t* out_eid_dev, double* out_times_dev, void* stream_v) {
    using namespace tpn;
    if (n < 0 || num_neighbors < 1 || num_nodes < 1 || n > ((int64_t)1 << 40)) return TPN_ERR_INVALID_ARGUMENT;
    if (n == 0) return TPN_OK;
    if (offsets_dev == nullptr || nbr_dev == nullptr || eid_dev == nullptr || times_dev == nullptr ||
        q_nodes_dev == nullptr || q_times_dev == nullptr || out_nbr_dev == nullptr || out_eid_dev == nullptr ||
        out_times_dev == nullptr)
        return TPN_ERR_INVALID_ARGUMENT;
    const long long blocks = (n * 32 + 255) / 256;
    if (blocks > 0x7fffffffll) return TPN_ERR_INVALID_ARGUMENT;
    DeviceScope scope(offsets_dev);
    sampler_recent_kernel<<<(unsigned)blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream_v)>>>(
        reinterpret_cast<const long long*>(offsets_dev), reinterpret_cast<const long long*>(nbr_dev),
        reinterpret_cast<const long long*>(eid_dev), times_dev, num_nodes,
        reinterpret_cast<const long long*>(q_nodes_dev), q_times_dev, n, num_neighbors,
        reinterpret_cast<long long*>(out_nbr_dev), reinterpret_cast<long long*>(out_eid_dev), out_times_dev);
    return check_launch();
}

// ---------------------------------------------------------------- streaming sampler (tpn_stream_sampler_*)
// The lists and the pending batch are described in include/tpnet_b200.h.  Why two lists: with tied timestamps
// (day-quantised streams) a query AT a node's newest folded time needs the last K entries strictly older than it,
// which ALL may already have dropped; OLD keeps them.  Why a pending batch: a query at time t must see the entries
// of the latest batch older than t, and only those — they are a prefix of the node's pending segment.
namespace tpn {
namespace {

struct StreamView {
    long long N;           // node ids (and pending keys) are 0 .. N-1
    long long rows;        // rows of the list tables: N, or owned + cache rows of a sharded sampler
    int world, rank;       // sharded: node u's lists are at row u / world of rank u % world
    int C;
    long long* all_nbr;
    long long* all_eid;
    double* all_t;
    long long* old_nbr;
    long long* old_eid;
    double* old_t;
    int* all_cnt;
    int* old_cnt;
    double* newest;
    uint32_t* pend_node;
    long long* pend_nbr;
    long long* pend_eid;
    double* pend_t;
    int* pend_count;
    double* last_time;
    int* err;
};

StreamView make_stream_view(const tpn_stream_sampler_t* s) {
    StreamView v;
    v.N = s->num_nodes;
    v.rows = s->num_nodes;
    v.world = 1;
    v.rank = 0;
    v.C = s->capacity;
    v.all_nbr = reinterpret_cast<long long*>(s->all_nbr);
    v.all_eid = reinterpret_cast<long long*>(s->all_eid);
    v.all_t = s->all_t;
    v.old_nbr = reinterpret_cast<long long*>(s->old_nbr);
    v.old_eid = reinterpret_cast<long long*>(s->old_eid);
    v.old_t = s->old_t;
    v.all_cnt = s->all_cnt;
    v.old_cnt = s->old_cnt;
    v.newest = s->newest;
    v.pend_node = s->pend_node;
    v.pend_nbr = reinterpret_cast<long long*>(s->pend_nbr);
    v.pend_eid = reinterpret_cast<long long*>(s->pend_eid);
    v.pend_t = s->pend_t;
    v.pend_count = s->pend_count;
    v.last_time = s->last_time;
    v.err = s->err_flag;
    return v;
}

constexpr double kNegInf = -__builtin_huge_val();

__global__ void __launch_bounds__(256) stream_reset_kernel(StreamView v) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < v.rows) v.newest[i] = kNegInf;
    if (i == 0) {
        *v.pend_count = 0;
        *v.last_time = kNegInf;
        *v.err = 0;
    }
}

// Dest row <- the last C of (X[0, a) ++ pending[p, p + b)); returns the new count.  dest may be X itself: entry j
// reads position j + shift (shift >= 0), so a chunk of 32 is read before it is written and later chunks read
// positions no earlier chunk wrote.  Only the last C entries of the pending range are touched.
__device__ __forceinline__ int fold_list(const StreamView& v, long long* dn, long long* de, double* dt,
                                         const long long* xn, const long long* xe, const double* xt, int a,
                                         long long p, long long b, int lane) {
    const long long total = (long long)a + b;
    const int nc = total < v.C ? (int)total : v.C;
    const long long shift = total - nc;
    for (int j0 = 0; j0 < nc; j0 += 32) {
        const int j = j0 + lane;
        long long vn = 0, ve = 0;
        double vt = 0.0;
        if (j < nc) {
            const long long s = j + shift;
            if (s < a) {
                vn = xn[s]; ve = xe[s]; vt = xt[s];
            } else {
                const long long q = p + (s - a);
                vn = v.pend_nbr[q]; ve = v.pend_eid[q]; vt = v.pend_t[q];
            }
        }
        __syncwarp();
        if (j < nc) {
            dn[j] = vn; de[j] = ve; dt[j] = vt;
        }
        __syncwarp();
    }
    return nc;
}

// One warp per pending position; the warp at the head of a node's segment folds it (the others leave at once).
// SHARDED: only the segments of the nodes this rank owns, into row u / world (world 1 compiles to the plain fold).
template <bool SHARDED>
__global__ void __launch_bounds__(256) stream_fold_kernel(StreamView v, long long cap) {
    const long long p = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (p >= cap) return;
    const long long pc = *v.pend_count;
    if (p >= pc) return;
    const uint32_t u = v.pend_node[p];
    if ((long long)u >= v.N || (p > 0 && v.pend_node[p - 1] == u)) return;
    if (SHARDED && (int)(u % (uint32_t)v.world) != v.rank) return;
    const long long r = SHARDED ? (long long)(u / (uint32_t)v.world) : (long long)u;
    long long lo = p + 1, hi = pc;                   // end of the segment (every lane runs the same searches)
    while (lo < hi) {
        const long long mid = lo + ((hi - lo) >> 1);
        if (v.pend_node[mid] == u) lo = mid + 1; else hi = mid;
    }
    const long long e = lo;
    const double tnew = v.pend_t[e - 1];
    const long long row = r * v.C;
    const int a = v.all_cnt[r];
    if (tnew > v.newest[r]) {
        lo = p; hi = e - 1;                          // first entry of the segment at tnew
        while (lo < hi) {
            const long long mid = lo + ((hi - lo) >> 1);
            if (v.pend_t[mid] < tnew) lo = mid + 1; else hi = mid;
        }
        const int oc = fold_list(v, v.old_nbr + row, v.old_eid + row, v.old_t + row, v.all_nbr + row,
                                 v.all_eid + row, v.all_t + row, a, p, lo - p, lane);
        if (lane == 0) {
            v.old_cnt[r] = oc;
            v.newest[r] = tnew;
        }
    }
    const int ac = fold_list(v, v.all_nbr + row, v.all_eid + row, v.all_t + row, v.all_nbr + row, v.all_eid + row,
                             v.all_t + row, a, p, e - p, lane);
    if (lane == 0) v.all_cnt[r] = ac;
}

// Validation and sort keys of the new batch: entry 2j is (src[j] <- dst[j]), entry 2j+1 is (dst[j] <- src[j]).
// A dropped edge gets key N on both entries: it sorts behind every node and no fold or query reads it.
__global__ void __launch_bounds__(256)
stream_prep_kernel(StreamView v, const long long* __restrict__ src, const long long* __restrict__ dst,
                   const double* __restrict__ t, long long B, uint32_t* __restrict__ key, uint32_t* __restrict__ val) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= B) return;
    const long long a = src[j], b = dst[j];
    const double prev = j > 0 ? t[j - 1] : *v.last_time;
    const bool ids_ok = a >= 0 && a < v.N && b >= 0 && b < v.N;
    const bool t_ok = !(t[j] < prev);
    if (!ids_ok) atomicOr(v.err, TPN_STREAM_ERR_INDEX);
    if (!t_ok) atomicOr(v.err, TPN_STREAM_ERR_ORDER);
    const bool ok = ids_ok && t_ok;
    key[2 * j] = ok ? (uint32_t)a : (uint32_t)v.N;
    key[2 * j + 1] = ok ? (uint32_t)b : (uint32_t)v.N;
    val[2 * j] = (uint32_t)(2 * j);
    val[2 * j + 1] = (uint32_t)(2 * j + 1);
}

// Sorted (key, 2j + direction) -> the pending arrays; the batch's count and last time.
__global__ void __launch_bounds__(256)
stream_pending_kernel(StreamView v, const long long* __restrict__ src, const long long* __restrict__ dst,
                      const long long* __restrict__ eid, const double* __restrict__ t, long long B,
                      const uint32_t* __restrict__ skey, const uint32_t* __restrict__ sval) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= 2 * B) return;
    const uint32_t m = sval[p];
    const long long j = m >> 1;
    v.pend_node[p] = skey[p];
    v.pend_nbr[p] = (m & 1) ? src[j] : dst[j];
    v.pend_eid[p] = eid[j];
    v.pend_t[p] = t[j];
    if (p == 0) {
        *v.pend_count = (int)(2 * B);
        const double lt = *v.last_time, tl = t[B - 1];
        *v.last_time = tl > lt ? tl : lt;
    }
}

// One warp per query, like sampler_recent_kernel; the source list is ALL ++ (pending entries of u older than t),
// or OLD when t is the node's newest folded time.  ROWS: the lists of q_nodes[q] are at row q_rows[q] (sharded: own
// row or cache slot); the pending entries are still found by the global id.
template <bool ROWS>
__global__ void __launch_bounds__(256)
stream_query_kernel(StreamView v, const long long* __restrict__ q_nodes, const long long* __restrict__ q_rows,
                    const double* __restrict__ q_times, long long n, int K, long long* __restrict__ out_nbr,
                    long long* __restrict__ out_eid, double* __restrict__ out_t) {
    const long long q = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (q >= n) return;
    const long long u = q_nodes[q];
    const double t = q_times[q];
    int mode = 0;                                    // 0: zero row, 1: ALL ++ pending, 2: OLD
    long long a = 0, s0 = 0, total = 0, r = 0;
    if (u < 0 || u >= v.N) {
        if (lane == 0) atomicOr(v.err, TPN_STREAM_ERR_INDEX);
    } else {
        r = ROWS ? q_rows[q] : u;
        const double tu = v.newest[r];
        if (t > tu) {
            mode = 1;
            a = v.all_cnt[r];
            const long long pc = *v.pend_count;
            long long lo = 0, hi = pc;               // first pending entry of u
            while (lo < hi) {
                const long long mid = lo + ((hi - lo) >> 1);
                if ((long long)v.pend_node[mid] < u) lo = mid + 1; else hi = mid;
            }
            s0 = lo;
            hi = pc;                                 // first pending entry of u at or after t (or of a later node)
            while (lo < hi) {
                const long long mid = lo + ((hi - lo) >> 1);
                if ((long long)v.pend_node[mid] == u && v.pend_t[mid] < t) lo = mid + 1; else hi = mid;
            }
            total = a + (lo - s0);
        } else if (t == tu) {
            mode = 2;
            total = v.old_cnt[r];
        } else if (lane == 0) {
            atomicOr(v.err, TPN_STREAM_ERR_PAST);
        }
    }
    const int take = (int)(total < (long long)K ? total : (long long)K);
    const long long first = total - take;
    const int pad = K - take;
    const long long row = mode ? r * v.C : 0;
    for (int j = lane; j < K; j += 32) {
        long long vn = 0, ve = 0;
        double vt = 0.0;
        if (j >= pad) {
            const long long s = first + (j - pad);
            if (mode == 2) {
                vn = v.old_nbr[row + s]; ve = v.old_eid[row + s]; vt = v.old_t[row + s];
            } else if (s < a) {
                vn = v.all_nbr[row + s]; ve = v.all_eid[row + s]; vt = v.all_t[row + s];
            } else {
                const long long r = s0 + (s - a);
                vn = v.pend_nbr[r]; ve = v.pend_eid[r]; vt = v.pend_t[r];
            }
        }
        out_nbr[q * K + j] = vn;
        out_eid[q * K + j] = ve;
        out_t[q * K + j] = vt;
    }
}

// Sharded: one warp per cache slot handed out by the latest tpn_route_nodes ([PREV, NEED) of the shard counters): the
// slot's node's newest time, counts and the first count entries of ALL and OLD, read out of its owner's tables.
__global__ void __launch_bounds__(256)
stream_pull_kernel(StreamView v, const void* const* __restrict__ peer, const int* __restrict__ counters,
                   const long long* __restrict__ need_nodes, long long n_local, long long ext_rows) {
    const int lane = threadIdx.x & 31;
    const int warps = gridDim.x * (blockDim.x >> 5);
    const int first = counters[TPN_SHARD_CTR_PREV];
    int last = counters[TPN_SHARD_CTR_NEED];
    last = last < ext_rows ? last : (int)ext_rows;
    for (int slot = first + blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); slot < last; slot += warps) {
        const long long u = need_nodes[slot];
        const void* const* T = peer + (u % v.world) * TPN_STREAM_PEER_TABLES;
        const long long r = u / v.world, d = n_local + slot;
        const int ac = static_cast<const int*>(T[6])[r];
        const int oc = static_cast<const int*>(T[7])[r];
        if (lane == 0) {
            v.all_cnt[d] = ac;
            v.old_cnt[d] = oc;
            v.newest[d] = static_cast<const double*>(T[8])[r];
        }
        const long long so = r * v.C, dof = d * v.C;
        for (int j = lane; j < ac; j += 32) {
            v.all_nbr[dof + j] = static_cast<const long long*>(T[0])[so + j];
            v.all_eid[dof + j] = static_cast<const long long*>(T[1])[so + j];
            v.all_t[dof + j] = static_cast<const double*>(T[2])[so + j];
        }
        for (int j = lane; j < oc; j += 32) {
            v.old_nbr[dof + j] = static_cast<const long long*>(T[3])[so + j];
            v.old_eid[dof + j] = static_cast<const long long*>(T[4])[so + j];
            v.old_t[dof + j] = static_cast<const double*>(T[5])[so + j];
        }
    }
}

// Workspace of a push of B edges: sort keys / values (ping-pong) and the radix histograms.
struct StreamWs {
    uint32_t *key_a, *key_b, *val_a, *val_b, *hist;
};

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

size_t stream_ws_layout(long long B, void* base, StreamWs* ws) {
    const long long E = 2 * B;
    const long long nblk = (E + kRadixTile - 1) / kRadixTile;
    const size_t arr = align256((size_t)E * 4);
    const size_t hist = align256((size_t)(nblk + 1) * kRadixBins * 4);
    if (ws != nullptr) {
        char* p = static_cast<char*>(base);
        ws->key_a = reinterpret_cast<uint32_t*>(p);
        ws->key_b = reinterpret_cast<uint32_t*>(p + arr);
        ws->val_a = reinterpret_cast<uint32_t*>(p + 2 * arr);
        ws->val_b = reinterpret_cast<uint32_t*>(p + 3 * arr);
        ws->hist = reinterpret_cast<uint32_t*>(p + 4 * arr);
    }
    return 4 * arr + hist;
}

constexpr long long kStreamMaxBatch = (long long)1 << 29;   // 2B sort entries must fit an int (Count)

int validate_stream(const tpn_stream_sampler_t* s) {
    if (s == nullptr || s->capacity < 1 || s->num_nodes < 1 || s->num_nodes > 0xffffffffll || s->max_batch < 1 ||
        s->max_batch > kStreamMaxBatch)
        return TPN_ERR_INVALID_ARGUMENT;
    return TPN_OK;
}

bool stream_tables_set(const tpn_stream_sampler_t* s) {
    return s->all_nbr != nullptr && s->all_eid != nullptr && s->all_t != nullptr && s->old_nbr != nullptr &&
           s->old_eid != nullptr && s->old_t != nullptr && s->all_cnt != nullptr && s->old_cnt != nullptr &&
           s->newest != nullptr && s->pend_node != nullptr && s->pend_nbr != nullptr && s->pend_eid != nullptr &&
           s->pend_t != nullptr && s->pend_count != nullptr && s->last_time != nullptr && s->err_flag != nullptr;
}

// A sharded sampler: the plain checks, a shard whose placement matches the global node count (so every row a kernel
// computes is inside the tables), and the sampler's own routing tables.
int validate_stream_shard(const tpn_stream_shard_t* s) {
    if (s == nullptr) return TPN_ERR_INVALID_ARGUMENT;
    const int rc = validate_stream(&s->local);
    if (rc != TPN_OK) return rc;
    const tpn_shard_t& h = s->shard;
    if (h.world < 1 || h.world > 64 || h.rank < 0 || h.rank >= h.world || h.global_nodes != s->local.num_nodes ||
        h.global_nodes > 0x7fffffffll || h.ext_rows < 0 || h.ext_rows > 0x7ffffff0ll ||
        h.num_local_rows != (h.global_nodes > h.rank ? (h.global_nodes - h.rank + h.world - 1) / h.world : 0) ||
        h.mark == nullptr || h.counters == nullptr || h.need_nodes == nullptr)
        return TPN_ERR_INVALID_ARGUMENT;
    return TPN_OK;
}

StreamView make_stream_shard_view(const tpn_stream_shard_t* s) {
    StreamView v = make_stream_view(&s->local);
    v.rows = s->shard.num_local_rows + s->shard.ext_rows;
    v.world = s->shard.world;
    v.rank = s->shard.rank;
    return v;
}

int stream_reset_impl(const StreamView& v, cudaStream_t stream) {
    if (cudaMemsetAsync(v.all_cnt, 0, (size_t)v.rows * 4, stream) != cudaSuccess ||
        cudaMemsetAsync(v.old_cnt, 0, (size_t)v.rows * 4, stream) != cudaSuccess) {
        set_cuda_error(cudaGetLastError());
        return TPN_ERR_CUDA;
    }
    const long long blocks = v.rows > 0 ? (v.rows + 255) / 256 : 1;        // one block at least: the scalars
    stream_reset_kernel<<<(unsigned)blocks, 256, 0, stream>>>(v);
    return check_launch();
}

// Arguments already validated: fold the pending batch (SHARDED: the owned segments only), then sort the new one.
template <bool SHARDED>
int stream_push_impl(const tpn_stream_sampler_t* s, const StreamView& v, const int64_t* src_dev, const int64_t* dst_dev,
                     const int64_t* eid_dev, const double* t_dev, int64_t batch, const StreamWs& ws,
                     cudaStream_t stream) {
    const auto* src = reinterpret_cast<const long long*>(src_dev);
    const auto* dst = reinterpret_cast<const long long*>(dst_dev);
    const auto* eid = reinterpret_cast<const long long*>(eid_dev);

    // 1. fold the previous pending batch (its size is on the device: the grid covers the largest one)
    const long long cap = 2 * s->max_batch;
    stream_fold_kernel<SHARDED><<<(unsigned)((cap * 32 + 255) / 256), 256, 0, stream>>>(v, cap);
    // 2. the new batch, stably sorted by node
    const int E = (int)(2 * batch);
    stream_prep_kernel<<<(unsigned)((batch + 255) / 256), 256, 0, stream>>>(v, src, dst, t_dev, batch, ws.key_a,
                                                                             ws.val_a);
    int passes = 1;
    while (passes < 4 && ((unsigned long long)s->num_nodes >> (8 * passes)) != 0) ++passes;   // key N must sort too
    const int nblk = (E + kRadixTile - 1) / kRadixTile;
    const Count cnt{E, nullptr};
    const int prefixed = nblk > kRadixDirectBlocks ? 1 : 0;
    uint32_t *kin = ws.key_a, *kout = ws.key_b, *vin = ws.val_a, *vout = ws.val_b;
    for (int p = 0; p < passes; ++p) {
        radix_hist_kernel<<<nblk, kRadixThreads, 0, stream>>>(kin, cnt, 8 * p, ws.hist);
        if (prefixed) radix_prefix_kernel<<<kRadixBins / 8, 256, 0, stream>>>(ws.hist, cnt);
        radix_scatter_kernel<<<nblk, kRadixThreads, 0, stream>>>(kin, vin, kout, vout, cnt, 8 * p, ws.hist, prefixed);
        uint32_t* tk = kin; kin = kout; kout = tk;
        uint32_t* tv = vin; vin = vout; vout = tv;
    }
    stream_pending_kernel<<<(unsigned)((E + 255) / 256), 256, 0, stream>>>(v, src, dst, eid, t_dev, batch, kin, vin);
    return check_launch();
}

// Argument checks shared by the plain and the sharded push: TPN_OK with *ws laid out, or an error code; batch == 0
// returns TPN_OK with *launch = false.
int stream_push_args(const tpn_stream_sampler_t* s, const int64_t* src_dev, const int64_t* dst_dev,
                     const int64_t* eid_dev, const double* t_dev, int64_t batch, void* ws_dev, size_t ws_bytes,
                     StreamWs* ws, bool* launch) {
    *launch = false;
    if (batch < 0 || batch > s->max_batch) return TPN_ERR_INVALID_ARGUMENT;
    if (batch == 0) return TPN_OK;
    if (!stream_tables_set(s) || src_dev == nullptr || dst_dev == nullptr || eid_dev == nullptr || t_dev == nullptr ||
        ws_dev == nullptr)
        return TPN_ERR_INVALID_ARGUMENT;
    if (ws_bytes < stream_ws_layout(batch, ws_dev, ws)) return TPN_ERR_WORKSPACE_TOO_SMALL;
    *launch = true;
    return TPN_OK;
}

// Argument checks shared by the plain and the sharded query; *launch = false for n == 0.
int stream_query_args(const tpn_stream_sampler_t* s, const int64_t* q_nodes_dev, const double* q_times_dev, int64_t n,
                      int num_neighbors, const int64_t* out_nbr_dev, const int64_t* out_eid_dev,
                      const double* out_times_dev, bool* launch) {
    *launch = false;
    if (n < 0 || num_neighbors < 1 || num_neighbors > s->capacity || n > ((int64_t)1 << 40))
        return TPN_ERR_INVALID_ARGUMENT;
    if (n == 0) return TPN_OK;
    if (!stream_tables_set(s) || q_nodes_dev == nullptr || q_times_dev == nullptr || out_nbr_dev == nullptr ||
        out_eid_dev == nullptr || out_times_dev == nullptr)
        return TPN_ERR_INVALID_ARGUMENT;
    if ((n * 32 + 255) / 256 > 0x7fffffffll) return TPN_ERR_INVALID_ARGUMENT;
    *launch = true;
    return TPN_OK;
}

}  // namespace
}  // namespace tpn

extern "C" size_t tpn_stream_sampler_workspace_bytes(int64_t batch) {
    if (batch < 1) batch = 1;
    if (batch > tpn::kStreamMaxBatch) batch = tpn::kStreamMaxBatch;
    return tpn::stream_ws_layout(batch, nullptr, nullptr);
}

extern "C" int tpn_stream_sampler_reset(const tpn_stream_sampler_t* s, void* stream_v) {
    using namespace tpn;
    int rc = validate_stream(s);
    if (rc != TPN_OK) return rc;
    if (!stream_tables_set(s)) return TPN_ERR_INVALID_ARGUMENT;
    DeviceScope scope(s->newest);
    return stream_reset_impl(make_stream_view(s), reinterpret_cast<cudaStream_t>(stream_v));
}

extern "C" int tpn_stream_sampler_push(const tpn_stream_sampler_t* s, const int64_t* src_dev, const int64_t* dst_dev,
                                       const int64_t* eid_dev, const double* t_dev, int64_t batch, void* ws_dev,
                                       size_t ws_bytes, void* stream_v) {
    using namespace tpn;
    int rc = validate_stream(s);
    if (rc != TPN_OK) return rc;
    StreamWs ws;
    bool launch;
    rc = stream_push_args(s, src_dev, dst_dev, eid_dev, t_dev, batch, ws_dev, ws_bytes, &ws, &launch);
    if (rc != TPN_OK || !launch) return rc;
    DeviceScope scope(s->newest);
    return stream_push_impl<false>(s, make_stream_view(s), src_dev, dst_dev, eid_dev, t_dev, batch, ws,
                                   reinterpret_cast<cudaStream_t>(stream_v));
}

extern "C" int tpn_stream_sampler_query(const tpn_stream_sampler_t* s, const int64_t* q_nodes_dev,
                                        const double* q_times_dev, int64_t n, int num_neighbors, int64_t* out_nbr_dev,
                                        int64_t* out_eid_dev, double* out_times_dev, void* stream_v) {
    using namespace tpn;
    int rc = validate_stream(s);
    if (rc != TPN_OK) return rc;
    bool launch;
    rc = stream_query_args(s, q_nodes_dev, q_times_dev, n, num_neighbors, out_nbr_dev, out_eid_dev, out_times_dev,
                           &launch);
    if (rc != TPN_OK || !launch) return rc;
    DeviceScope scope(s->newest);
    stream_query_kernel<false><<<(unsigned)((n * 32 + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream_v)>>>(
        make_stream_view(s), reinterpret_cast<const long long*>(q_nodes_dev), nullptr, q_times_dev, n, num_neighbors,
        reinterpret_cast<long long*>(out_nbr_dev), reinterpret_cast<long long*>(out_eid_dev), out_times_dev);
    return check_launch();
}

// ---------------------------------------------------------------- sharded streaming sampler (tpn_stream_shard_*)
extern "C" int tpn_stream_shard_reset(const tpn_stream_shard_t* s, void* stream_v) {
    using namespace tpn;
    int rc = validate_stream_shard(s);
    if (rc != TPN_OK) return rc;
    if (!stream_tables_set(&s->local)) return TPN_ERR_INVALID_ARGUMENT;
    DeviceScope scope(s->local.newest);
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_v);
    const cudaError_t e1 = cudaMemsetAsync(s->shard.mark, 0, sizeof(int32_t) * (size_t)s->shard.global_nodes, stream);
    const cudaError_t e2 = cudaMemsetAsync(s->shard.counters, 0, sizeof(int32_t) * TPN_SHARD_COUNTERS, stream);
    if (e1 != cudaSuccess || e2 != cudaSuccess) {
        set_cuda_error(e1 != cudaSuccess ? e1 : e2);
        return TPN_ERR_CUDA;
    }
    return stream_reset_impl(make_stream_shard_view(s), stream);
}

extern "C" int tpn_stream_shard_push(const tpn_stream_shard_t* s, const int64_t* src_dev, const int64_t* dst_dev,
                                     const int64_t* eid_dev, const double* t_dev, int64_t batch, void* ws_dev,
                                     size_t ws_bytes, void* stream_v) {
    using namespace tpn;
    int rc = validate_stream_shard(s);
    if (rc != TPN_OK) return rc;
    StreamWs ws;
    bool launch;
    rc = stream_push_args(&s->local, src_dev, dst_dev, eid_dev, t_dev, batch, ws_dev, ws_bytes, &ws, &launch);
    if (rc != TPN_OK || !launch) return rc;
    DeviceScope scope(s->local.newest);
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_v);
    // the fold rewrites lists that other ranks may hold in their caches, and this rank's cache is of the old lists:
    // a new generation (NEED and PREV restart; the error counter is sticky until the host reads it)
    cudaError_t e = cudaMemsetAsync(s->shard.mark, 0, sizeof(int32_t) * (size_t)s->shard.global_nodes, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(s->shard.counters, 0, sizeof(int32_t) * 2, stream);
    if (e != cudaSuccess) {
        set_cuda_error(e);
        return TPN_ERR_CUDA;
    }
    const StreamView v = make_stream_shard_view(s);
    if (s->shard.world == 1)
        return stream_push_impl<false>(&s->local, v, src_dev, dst_dev, eid_dev, t_dev, batch, ws, stream);
    return stream_push_impl<true>(&s->local, v, src_dev, dst_dev, eid_dev, t_dev, batch, ws, stream);
}

extern "C" int tpn_stream_shard_pull(const tpn_stream_shard_t* s, void* stream_v) {
    using namespace tpn;
    int rc = validate_stream_shard(s);
    if (rc != TPN_OK) return rc;
    if (!stream_tables_set(&s->local) || s->peer_lists == nullptr) return TPN_ERR_INVALID_ARGUMENT;
    if (s->shard.world == 1) return TPN_OK;
    DeviceScope scope(s->local.newest);
    const unsigned grid = (unsigned)device_sm_count() * 4;
    stream_pull_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream_v)>>>(
        make_stream_shard_view(s), s->peer_lists, s->shard.counters, reinterpret_cast<const long long*>(s->shard.need_nodes),
        s->shard.num_local_rows, s->shard.ext_rows);
    return check_launch();
}

extern "C" int tpn_stream_shard_query(const tpn_stream_shard_t* s, const int64_t* q_nodes_dev, const int64_t* q_rows_dev,
                                      const double* q_times_dev, int64_t n, int num_neighbors, int64_t* out_nbr_dev,
                                      int64_t* out_eid_dev, double* out_times_dev, void* stream_v) {
    using namespace tpn;
    int rc = validate_stream_shard(s);
    if (rc != TPN_OK) return rc;
    bool launch;
    rc = stream_query_args(&s->local, q_nodes_dev, q_times_dev, n, num_neighbors, out_nbr_dev, out_eid_dev,
                           out_times_dev, &launch);
    if (rc != TPN_OK || !launch) return rc;
    if (q_rows_dev == nullptr) return TPN_ERR_INVALID_ARGUMENT;
    DeviceScope scope(s->local.newest);
    stream_query_kernel<true><<<(unsigned)((n * 32 + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream_v)>>>(
        make_stream_shard_view(s), reinterpret_cast<const long long*>(q_nodes_dev),
        reinterpret_cast<const long long*>(q_rows_dev), q_times_dev, n, num_neighbors,
        reinterpret_cast<long long*>(out_nbr_dev), reinterpret_cast<long long*>(out_eid_dev), out_times_dev);
    return check_launch();
}

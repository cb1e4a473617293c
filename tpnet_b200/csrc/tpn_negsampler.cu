// Negative edge sampler (tpn_neg_sampler_*; DyGLib's NegativeEdgeSampler, the reference's utils/utils.py:315-505):
// tables built once on the device, then per call k distinct elements of an index range minus an excluded set, drawn
// through a keyed Feistel permutation of the range.  Semantics and the exact draw rule: include/tpnet_b200.h.
#include "tpn_radix.cuh"

namespace tpn {
namespace {

constexpr long long kNegMaxEdges = 0x7fffffffll - 4096;     // radix and scan counts are int
constexpr int kNegTagHist = 1, kNegTagFill = 2, kNegTagReplace = 3, kNegTagRandom = 4;
constexpr int kScanThreads = 256, kScanItems = 8, kScanTile = kScanThreads * kScanItems;
constexpr int kDrawThreads = 256;
constexpr int kDrawMaxBlocks = 1024;

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// order-preserving map of an f64 (no NaN) to uint64: sorting the words sorts the times
__device__ __forceinline__ unsigned long long time_key(double t) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(t);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

struct NegView {
    long long E;
    int timed;
    unsigned long long seed;
    double lot;
    const uint32_t *t_src, *t_dst, *t_fpos;
    const double* t_time;
    const uint32_t *f_src, *f_dst;
    const double* f_time;
    uint32_t* mark;
    const uint32_t *uniq_src, *uniq_dst;
    int* counts;
};

NegView make_neg_view(const tpn_neg_sampler_t* s) {
    NegView v;
    v.E = s->num_edges;
    v.timed = s->timed;
    v.seed = s->seed;
    v.lot = s->last_observed_time;
    v.t_src = s->t_src;
    v.t_dst = s->t_dst;
    v.t_fpos = s->t_fpos;
    v.t_time = s->t_time;
    v.f_src = s->f_src;
    v.f_dst = s->f_dst;
    v.f_time = s->f_time;
    v.mark = s->mark;
    v.uniq_src = s->uniq_src;
    v.uniq_dst = s->uniq_dst;
    v.counts = s->counts;
    return v;
}

// ---------------------------------------------------------------- radix passes over (uint32 key, uint32 value)
struct SortBufs {
    uint32_t *k, *v, *k2, *v2;     // k, v: current data; k2, v2: free
    uint32_t* hist;
    void swap() {
        uint32_t* t = k; k = k2; k2 = t;
        t = v; v = v2; v2 = t;
    }
};

void sort_passes(SortBufs& b, Count cnt, int first, int passes, cudaStream_t stream) {
    const int nblk = (cnt.cap + kRadixTile - 1) / kRadixTile;
    const int prefixed = nblk > kRadixDirectBlocks ? 1 : 0;
    for (int p = first; p < first + passes; ++p) {
        radix_hist_kernel<<<nblk, kRadixThreads, 0, stream>>>(b.k, cnt, 8 * p, b.hist);
        if (prefixed) radix_prefix_kernel<<<kRadixBins / 8, 256, 0, stream>>>(b.hist, cnt);
        radix_scatter_kernel<<<nblk, kRadixThreads, 0, stream>>>(b.k, b.v, b.k2, b.v2, cnt, 8 * p, b.hist, prefixed);
        b.swap();
    }
}

unsigned grid_for(long long n, int threads = 256) { return (unsigned)((n + threads - 1) / threads); }

// ---------------------------------------------------------------- exclusive scan of head flags (three launches)
// Flag::head(r): does item r < n start a new run?  Emit::emit(r, run index of r, head).
struct KeyHead {        // T positions in (src, dst, time) order: a new key
    const uint32_t *perm, *src, *dst;
    __device__ bool head(long long r) const {
        if (r == 0) return true;
        const uint32_t p = perm[r], q = perm[r - 1];
        return src[p] != src[q] || dst[p] != dst[q];
    }
};
struct IdHead {         // sorted ids: a new id
    const uint32_t* a;
    __device__ bool head(long long r) const { return r == 0 || a[r] != a[r - 1]; }
};
struct KeyEmit {        // K: the first (earliest) edge of each key; every T position learns its key's index
    const uint32_t *perm, *src, *dst;
    const double* time;
    uint32_t *ksrc, *kdst, *kid_of_t;
    double* kf;
    __device__ void emit(long long r, uint32_t kid, bool head) const {
        const uint32_t p = perm[r];
        kid_of_t[p] = kid;
        if (head) {
            ksrc[kid] = src[p];
            kdst[kid] = dst[p];
            kf[kid] = time[p];
        }
    }
};
struct IdEmit {
    const uint32_t* a;
    uint32_t* out;
    __device__ void emit(long long r, uint32_t idx, bool head) const {
        if (head) out[idx] = a[r];
    }
};

template <class Flag>
__global__ void __launch_bounds__(kScanThreads) scan_count_kernel(Flag f, Count cnt, uint32_t* __restrict__ bsum) {
    const int n = cnt.get();
    const long long base = (long long)blockIdx.x * kScanTile + threadIdx.x * kScanItems;
    int c = 0;
#pragma unroll
    for (int i = 0; i < kScanItems; ++i)
        if (base + i < n && f.head(base + i)) ++c;
    __shared__ int red[kScanThreads / 32];
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < kScanThreads / 32; ++w) t += red[w];
        bsum[blockIdx.x] = (uint32_t)t;
    }
}

// one block: exclusive prefix of the tile counts in place, the total to *total
__global__ void __launch_bounds__(1024) scan_top_kernel(uint32_t* __restrict__ bsum, Count cnt, int* total) {
    __shared__ uint32_t wsum[32];
    const int nblk = (cnt.get() + kScanTile - 1) / kScanTile;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t carry = 0;
    for (int b0 = 0; b0 < nblk; b0 += 1024) {
        const int b = b0 + threadIdx.x;
        const uint32_t c = b < nblk ? bsum[b] : 0u;
        uint32_t inc = c;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t nb = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += nb;
        }
        if (lane == 31) wsum[wid] = inc;
        __syncthreads();
        uint32_t before = 0, all = 0;
        for (int w = 0; w < 32; ++w) {
            before += w < wid ? wsum[w] : 0u;
            all += wsum[w];
        }
        if (b < nblk) bsum[b] = carry + before + inc - c;
        carry += all;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = (int)carry;
}

template <class Flag, class Emit>
__global__ void __launch_bounds__(kScanThreads) scan_emit_kernel(Flag f, Emit em, Count cnt,
                                                                 const uint32_t* __restrict__ bsum) {
    __shared__ uint32_t wsum[kScanThreads / 32];
    const int n = cnt.get();
    if ((long long)blockIdx.x * kScanTile >= n) return;
    const long long base = (long long)blockIdx.x * kScanTile + threadIdx.x * kScanItems;
    bool h[kScanItems];
    uint32_t c = 0;
#pragma unroll
    for (int i = 0; i < kScanItems; ++i) {
        h[i] = base + i < n && f.head(base + i);
        c += h[i] ? 1u : 0u;
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t inc = c;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t nb = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += nb;
    }
    if (lane == 31) wsum[wid] = inc;
    __syncthreads();
    uint32_t run = bsum[blockIdx.x] + inc - c;
    for (int w = 0; w < wid; ++w) run += wsum[w];
#pragma unroll
    for (int i = 0; i < kScanItems; ++i) {
        if (base + i >= n) break;
        run += h[i] ? 1u : 0u;
        em.emit(base + i, run - 1, h[i]);          // run index = inclusive head count - 1
    }
}

template <class Flag, class Emit>
void scan_emit(Flag f, Emit em, Count cnt, uint32_t* bsum, int* total, cudaStream_t stream) {
    const int nblk = (cnt.cap + kScanTile - 1) / kScanTile;
    scan_count_kernel<<<nblk, kScanThreads, 0, stream>>>(f, cnt, bsum);
    scan_top_kernel<<<1, 1024, 0, stream>>>(bsum, cnt, total);
    scan_emit_kernel<<<nblk, kScanThreads, 0, stream>>>(f, em, cnt, bsum);
}

// ---------------------------------------------------------------- build kernels
__global__ void time_lo_kernel(const double* __restrict__ t, Count cnt, uint32_t* __restrict__ k,
                               uint32_t* __restrict__ v) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cnt.get()) return;
    k[i] = (uint32_t)time_key(t[i]);
    v[i] = (uint32_t)i;
}
// second word of a 64-bit time sort: the high word of the time of the element the first pass put at r
__global__ void time_hi_kernel(const double* __restrict__ t, Count cnt, const uint32_t* __restrict__ vin,
                               uint32_t* __restrict__ k, uint32_t* __restrict__ v) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= cnt.get()) return;
    const uint32_t i = vin[r];
    k[r] = (uint32_t)(time_key(t[i]) >> 32);
    v[r] = i;
}
__global__ void fill_t_kernel(const long long* __restrict__ src, const long long* __restrict__ dst,
                              const double* __restrict__ t, long long E, const uint32_t* __restrict__ perm,
                              uint32_t* __restrict__ t_src, uint32_t* __restrict__ t_dst, double* __restrict__ t_time) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= E) return;
    const uint32_t i = perm[r];
    t_src[r] = (uint32_t)src[i];
    t_dst[r] = (uint32_t)dst[i];
    t_time[r] = t[i];
}
// k[r] = word[perm[r]] (perm == nullptr: identity), v[r] = perm[r] (or r)
__global__ void gather_word_kernel(const uint32_t* __restrict__ word, const uint32_t* __restrict__ perm, long long E,
                                   uint32_t* __restrict__ k, uint32_t* __restrict__ v) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= E) return;
    const uint32_t i = perm != nullptr ? perm[r] : (uint32_t)r;
    k[r] = word[i];
    v[r] = i;
}
__global__ void ids_kernel(const long long* __restrict__ ids, long long E, uint32_t* __restrict__ k,
                           uint32_t* __restrict__ v) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= E) return;
    k[i] = (uint32_t)ids[i];
    v[i] = (uint32_t)i;
}
// F position p holds K entry permF[p]; fpos_of_k is its inverse
__global__ void fill_f_kernel(Count cnt, const uint32_t* __restrict__ perm_f, const uint32_t* __restrict__ ksrc,
                              const uint32_t* __restrict__ kdst, const double* __restrict__ kf,
                              uint32_t* __restrict__ f_src, uint32_t* __restrict__ f_dst, double* __restrict__ f_time,
                              uint32_t* __restrict__ fpos_of_k) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= cnt.get()) return;
    const uint32_t q = perm_f[p];
    f_src[p] = ksrc[q];
    f_dst[p] = kdst[q];
    f_time[p] = kf[q];
    fpos_of_k[q] = (uint32_t)p;
}
__global__ void t_fpos_kernel(long long E, const uint32_t* __restrict__ kid_of_t, const uint32_t* __restrict__ fpos_of_k,
                              uint32_t* __restrict__ t_fpos) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < E) t_fpos[j] = fpos_of_k[kid_of_t[j]];
}

// ---------------------------------------------------------------- workspaces
struct BuildWs {
    uint32_t *k, *k2, *v, *v2, *hist, *bsum, *ksrc, *kdst, *kid_of_t;
    double* kf;
};

size_t build_ws_layout(long long E, void* base, BuildWs* ws) {
    const long long nblk = (E + kRadixTile - 1) / kRadixTile;
    const size_t a4 = align256((size_t)E * 4), a8 = align256((size_t)E * 8);
    const size_t hist = align256((size_t)(nblk + 1) * kRadixBins * 4), bsum = align256((size_t)(nblk + 1) * 4);
    if (ws != nullptr) {
        char* p = static_cast<char*>(base);
        uint32_t** w4[] = {&ws->k, &ws->k2, &ws->v, &ws->v2, &ws->ksrc, &ws->kdst, &ws->kid_of_t};
        for (uint32_t** w : w4) {
            *w = reinterpret_cast<uint32_t*>(p);
            p += a4;
        }
        ws->kf = reinterpret_cast<double*>(p);
        p += a8;
        ws->hist = reinterpret_cast<uint32_t*>(p);
        p += hist;
        ws->bsum = reinterpret_cast<uint32_t*>(p);
    }
    return 7 * a4 + a8 + hist + bsum;
}

// per-call parameters, written by the setup kernel
struct NegParams {
    long long a, b;          // the domain: F[a, b)
    long long lo, hi;        // the window: T[lo, hi)
    int xh;                  // distinct keys of the window inside F[a, b)
    int xf;                  // distinct batch pairs inside S x D
};

struct SampleWs {
    NegParams* prm;
    unsigned long long *bcount_h, *bcount_f;
    uint32_t *k, *k2, *v, *v2, *hist;
    uint32_t* hist_idx;
    unsigned long long* fill_idx;
};

size_t sample_ws_layout(long long size, long long batch, void* base, SampleWs* ws) {
    const long long nb = batch > 0 ? batch : 1;
    const long long nblk = (nb + kRadixTile - 1) / kRadixTile;
    const size_t prm = align256(sizeof(NegParams)), bc = align256((size_t)kDrawMaxBlocks * 8);
    const size_t a4 = align256((size_t)nb * 4), hist = align256((size_t)(nblk + 1) * kRadixBins * 4);
    const size_t hidx = align256((size_t)(size > 0 ? size : 1) * 4), fidx = align256((size_t)(size + nb) * 8);
    if (ws != nullptr) {
        char* p = static_cast<char*>(base);
        ws->prm = reinterpret_cast<NegParams*>(p);
        p += prm;
        ws->bcount_h = reinterpret_cast<unsigned long long*>(p);
        p += bc;
        ws->bcount_f = reinterpret_cast<unsigned long long*>(p);
        p += bc;
        uint32_t** w4[] = {&ws->k, &ws->k2, &ws->v, &ws->v2};
        for (uint32_t** w : w4) {
            *w = reinterpret_cast<uint32_t*>(p);
            p += a4;
        }
        ws->hist = reinterpret_cast<uint32_t*>(p);
        p += hist;
        ws->hist_idx = reinterpret_cast<uint32_t*>(p);
        p += hidx;
        ws->fill_idx = reinterpret_cast<unsigned long long*>(p);
    }
    return prm + 2 * bc + 4 * a4 + hist + hidx + fidx;
}

// ---------------------------------------------------------------- the draw primitive
__device__ __forceinline__ unsigned long long philox_x0(unsigned long long c0, unsigned long long c1, int tag,
                                                        unsigned long long seed, unsigned long long call) {
    unsigned long long x[4] = {c0, c1, (unsigned long long)tag, 0ull};
    philox4x64_10(x, seed, call);
    return x[0];
}

// position p of the keyed permutation of [0, n): 4-round balanced Feistel on m bits, cycle-walking into [0, n)
__device__ unsigned long long permute(unsigned long long p, unsigned long long n, int tag, unsigned long long seed,
                                      unsigned long long call) {
    int m = 2;
    while (m < 62 && (1ull << m) < n) m += 2;
    const int half = m / 2;
    const unsigned long long mask = (1ull << half) - 1;
    unsigned long long y = p;
    do {
        unsigned long long L = y >> half, R = y & mask;
#pragma unroll 1
        for (int r = 0; r < 4; ++r) {
            const unsigned long long nl = R;
            R = L ^ (philox_x0(R, (unsigned long long)r, tag, seed, call) & mask);
            L = nl;
        }
        y = (L << half) | R;
    } while (y >= n);
    return y;
}

// #{i < n : a[i] < x} (strict) or #{a[i] <= x}; a sorted
__device__ long long count_below(const double* a, long long n, double x, bool strict) {
    long long lo = 0, hi = n;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        const double v = a[mid];
        if (strict ? v < x : v <= x) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}
// index of x in the sorted ids a[0, n), or -1
__device__ long long find_id(const uint32_t* a, long long n, long long x) {
    if (x < 0 || x > 0xffffffffll) return -1;
    long long lo = 0, hi = n;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if ((long long)a[mid] < x) lo = mid + 1;
        else hi = mid;
    }
    return lo < n && (long long)a[lo] == x ? lo : -1;
}

struct CallArgs {
    int strategy;
    unsigned long long call;
    long long size, batch;
    double start, end;
    const double *start_dev, *end_dev;
};

// one warp: the window, the domain, zero counters
__global__ void setup_kernel(NegView v, CallArgs c, NegParams* prm) {
    __shared__ long long r[4];
    const int lane = threadIdx.x;
    const double s = c.start_dev != nullptr ? *c.start_dev : c.start;
    const double e = c.end_dev != nullptr ? *c.end_dev : c.end;
    const long long U = v.counts[0];
    if (lane == 0) r[0] = count_below(v.t_time, v.E, s, true);
    if (lane == 1) r[1] = count_below(v.t_time, v.E, e, false);
    if (lane == 2) r[2] = count_below(v.f_time, U, s, false);
    if (lane == 3) r[3] = c.strategy == TPN_NEG_INDUCTIVE ? count_below(v.f_time, U, v.lot, false) : 0;
    __syncwarp();
    if (lane == 0) {
        const long long h = r[2], o = r[3];
        prm->a = o;
        prm->b = h > o ? h : o;
        prm->lo = r[0];
        prm->hi = r[1] > r[0] ? r[1] : r[0];
        prm->xh = 0;
        prm->xf = 0;
    }
}

// W(s, e): mark the F positions of the window's keys that lie in the domain, count them once each
__global__ void mark_kernel(NegView v, NegParams* __restrict__ prm) {
    const long long lo = prm->lo, hi = prm->hi, a = prm->a, b = prm->b;
    int found = 0;
    for (long long j = lo + (long long)blockIdx.x * blockDim.x + threadIdx.x; j < hi;
         j += (long long)gridDim.x * blockDim.x) {
        const uint32_t p = v.t_fpos[j];
        if (p >= a && p < b && atomicExch(&v.mark[p], 1u) == 0u) ++found;     // exactly one winner per key
    }
    for (int o = 16; o > 0; o >>= 1) found += __shfl_xor_sync(0xffffffffu, found, o);
    if ((threadIdx.x & 31) == 0 && found) atomicAdd(&prm->xh, found);         // integer count: order-free
}
__global__ void unmark_kernel(NegView v, const NegParams* __restrict__ prm) {
    const long long lo = prm->lo, hi = prm->hi;
    for (long long j = lo + (long long)blockIdx.x * blockDim.x + threadIdx.x; j < hi;
         j += (long long)gridDim.x * blockDim.x)
        v.mark[v.t_fpos[j]] = 0u;
}

// the batch's pairs as indices into S x D (|S||D|: not a pair of S x D), split into two words
__global__ void batch_keys_kernel(NegView v, const long long* __restrict__ bsrc, const long long* __restrict__ bdst,
                                  long long B, uint32_t* __restrict__ klo, uint32_t* __restrict__ khi) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= B) return;
    const long long nS = v.counts[1], nD = v.counts[2];
    const long long is = find_id(v.uniq_src, nS, bsrc[j]), id = find_id(v.uniq_dst, nD, bdst[j]);
    const unsigned long long q = (is >= 0 && id >= 0) ? (unsigned long long)is * nD + id
                                                       : (unsigned long long)nS * (unsigned long long)nD;
    klo[j] = (uint32_t)q;
    khi[j] = (uint32_t)(q >> 32);
}
__global__ void batch_count_kernel(NegView v, const uint32_t* __restrict__ klo, const uint32_t* __restrict__ khi,
                                   long long B, NegParams* prm) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int c = 0;
    if (j < B) {
        const unsigned long long nsd = (unsigned long long)v.counts[1] * (unsigned long long)v.counts[2];
        const unsigned long long q = ((unsigned long long)khi[j] << 32) | klo[j];
        const unsigned long long pq = j > 0 ? ((unsigned long long)khi[j - 1] << 32) | klo[j - 1] : ~0ull;
        c = (q < nsd && q != pq) ? 1 : 0;
    }
    c = __syncthreads_count(c);
    if (threadIdx.x == 0 && c) atomicAdd(&prm->xf, c);
}

struct Batch {
    const uint32_t *lo, *hi;
    long long n;
    __device__ bool contains(unsigned long long q) const {
        long long a = 0, b = n;
        while (a < b) {
            const long long mid = (a + b) >> 1;
            const unsigned long long x = ((unsigned long long)hi[mid] << 32) | lo[mid];
            if (x < q) a = mid + 1;
            else b = mid;
        }
        return a < n && (((unsigned long long)hi[a] << 32) | lo[a]) == q;
    }
};

// One part of a call: draw the first k survivors among positions [0, P) of the (keyed or identity) order of [0, n).
struct Domain {
    unsigned long long n, k, P;
    bool identity;
};
__device__ __forceinline__ unsigned long long hist_size(const NegParams& p) {
    return (unsigned long long)(p.b - p.a) - (unsigned long long)p.xh;
}
template <int PART>
__device__ Domain domain(const NegView& v, const NegParams& p, long long size) {
    Domain d{0, 0, 0, false};
    const unsigned long long hc = hist_size(p), sz = (unsigned long long)size;
    if (PART == kNegTagHist) {
        d.n = (unsigned long long)(p.b - p.a);
        d.k = sz < hc ? sz : hc;
        d.P = d.k + (unsigned long long)p.xh;
    } else {
        const unsigned long long kf = sz > hc ? sz - hc : 0;
        d.n = (unsigned long long)v.counts[1] * (unsigned long long)v.counts[2];
        const unsigned long long u = d.n - (unsigned long long)p.xf;
        if (kf == 0 || u == 0) return d;
        if (u >= kf) {
            d.k = kf;
            d.P = kf + (unsigned long long)p.xf;
        } else {                                  // with replacement: enumerate U in index order
            d.k = u;
            d.P = d.n;
            d.identity = true;
        }
    }
    return d;
}
template <int PART>
__device__ __forceinline__ bool survivor(const NegView& v, const NegParams& p, const Domain& d, const Batch& bt,
                                         unsigned long long call, unsigned long long pos, unsigned long long& val) {
    if (PART == kNegTagHist) {
        val = (unsigned long long)p.a + permute(pos, d.n, kNegTagHist, v.seed, call);
        return v.mark[val] == 0u;
    }
    val = d.identity ? pos : permute(pos, d.n, kNegTagFill, v.seed, call);
    return !bt.contains(val);
}

template <int PART>
__global__ void __launch_bounds__(kDrawThreads) draw_count_kernel(NegView v, const NegParams* __restrict__ prm,
                                                                  Batch bt, unsigned long long call, long long size,
                                                                  unsigned long long* __restrict__ bcount) {
    const NegParams p = *prm;
    const Domain d = domain<PART>(v, p, size);
    const unsigned long long chunk = (d.P + gridDim.x - 1) / gridDim.x;
    const unsigned long long begin = chunk * blockIdx.x, end = begin + chunk < d.P ? begin + chunk : d.P;
    unsigned long long c = 0;
    for (unsigned long long base = begin; base < end; base += kDrawThreads) {
        const unsigned long long pos = base + threadIdx.x;
        unsigned long long val;
        const bool s = pos < end && survivor<PART>(v, p, d, bt, call, pos, val);
        c += (unsigned long long)__syncthreads_count(s);
    }
    if (threadIdx.x == 0) bcount[blockIdx.x] = c;
}

template <int PART>
__global__ void __launch_bounds__(kDrawThreads) draw_write_kernel(NegView v, const NegParams* __restrict__ prm,
                                                                  Batch bt, unsigned long long call, long long size,
                                                                  const unsigned long long* __restrict__ bcount,
                                                                  uint32_t* __restrict__ out32,
                                                                  unsigned long long* __restrict__ out64) {
    __shared__ unsigned long long red[kDrawThreads / 32];
    __shared__ uint32_t wtot[kDrawThreads / 32];
    const NegParams p = *prm;
    const Domain d = domain<PART>(v, p, size);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    unsigned long long before = 0;
    for (unsigned b = threadIdx.x; b < blockIdx.x; b += kDrawThreads) before += bcount[b];
    for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    if (lane == 0) red[wid] = before;
    __syncthreads();
    unsigned long long offset = 0;
    for (int w = 0; w < kDrawThreads / 32; ++w) offset += red[w];
    if (offset >= d.k) return;                                   // block-uniform
    const unsigned long long chunk = (d.P + gridDim.x - 1) / gridDim.x;
    const unsigned long long begin = chunk * blockIdx.x, end = begin + chunk < d.P ? begin + chunk : d.P;
    for (unsigned long long base = begin; base < end && offset < d.k; base += kDrawThreads) {
        const unsigned long long pos = base + threadIdx.x;
        unsigned long long val = 0;
        const bool s = pos < end && survivor<PART>(v, p, d, bt, call, pos, val);
        const uint32_t bal = __ballot_sync(0xffffffffu, s);
        __syncthreads();                                         // wtot of the previous tile is read
        if (lane == 0) wtot[wid] = __popc(bal);
        __syncthreads();
        unsigned long long r = offset + __popc(bal & ((1u << lane) - 1u));
        uint32_t tile = 0;
        for (int w = 0; w < kDrawThreads / 32; ++w) {
            r += w < wid ? wtot[w] : 0u;
            tile += wtot[w];
        }
        if (s && r < d.k) {
            if (PART == kNegTagHist) out32[r] = (uint32_t)val;
            else out64[r] = val;
        }
        offset += tile;
    }
}

// [size] pairs: the fill first, then the historical part
__global__ void finalize_kernel(NegView v, const NegParams* __restrict__ prm, unsigned long long call, long long size,
                                const uint32_t* __restrict__ hist_idx, const unsigned long long* __restrict__ fill_idx,
                                long long* __restrict__ out_src, long long* __restrict__ out_dst) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= size) return;
    const NegParams p = *prm;
    const unsigned long long hc = hist_size(p);
    const unsigned long long kf = (unsigned long long)size > hc ? (unsigned long long)size - hc : 0;
    if ((unsigned long long)j < kf) {
        const Domain d = domain<kNegTagFill>(v, p, size);
        if (d.k == 0) {                                          // U is empty: the reference's assert
            if (j == 0) atomicOr(&v.counts[3], TPN_NEG_ERR_EMPTY);
            out_src[j] = -1;
            out_dst[j] = -1;
            return;
        }
        unsigned long long q;
        if (d.identity) q = fill_idx[__umul64hi(philox_x0((unsigned long long)j, 0, kNegTagReplace, v.seed, call), d.k)];
        else q = fill_idx[j];
        const unsigned long long nD = (unsigned long long)v.counts[2];
        out_src[j] = v.uniq_src[q / nD];
        out_dst[j] = v.uniq_dst[q % nD];
    } else {
        const uint32_t i = hist_idx[j - kf];
        out_src[j] = v.f_src[i];
        out_dst[j] = v.f_dst[i];
    }
}

__global__ void random_kernel(NegView v, unsigned long long call, long long size, long long* __restrict__ out_src,
                              long long* __restrict__ out_dst) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= size) return;
    unsigned long long x[4] = {(unsigned long long)i, 0ull, (unsigned long long)kNegTagRandom, 0ull};
    philox4x64_10(x, v.seed, call);
    out_src[i] = v.uniq_src[__umul64hi(x[0], (unsigned long long)v.counts[1])];
    out_dst[i] = v.uniq_dst[__umul64hi(x[1], (unsigned long long)v.counts[2])];
}

int passes_for_bits(int bits) { return (bits + 7) / 8; }

bool tables_set(const tpn_neg_sampler_t* s) {
    if (s->uniq_src == nullptr || s->uniq_dst == nullptr || s->counts == nullptr) return false;
    return !s->timed || (s->t_src != nullptr && s->t_dst != nullptr && s->t_time != nullptr && s->t_fpos != nullptr &&
                         s->f_src != nullptr && s->f_dst != nullptr && s->f_time != nullptr && s->mark != nullptr);
}

int validate_neg(const tpn_neg_sampler_t* s) {
    if (s == nullptr || s->num_edges < 1 || s->num_edges > kNegMaxEdges || s->id_bits < 1 || s->id_bits > 32 ||
        (s->timed != 0 && s->timed != 1) || !tables_set(s))
        return TPN_ERR_INVALID_ARGUMENT;
    return TPN_OK;
}

}  // namespace
}  // namespace tpn

extern "C" size_t tpn_neg_sampler_workspace_bytes(int64_t num_edges, int64_t size, int64_t batch) {
    using namespace tpn;
    size_t b = 0;
    if (num_edges > 0) b = build_ws_layout(num_edges < kNegMaxEdges ? num_edges : kNegMaxEdges, nullptr, nullptr);
    const long long sz = size < 0 ? 0 : (size > kNegMaxEdges ? kNegMaxEdges : size);
    const long long bt = batch < 0 ? 0 : (batch > kNegMaxEdges ? kNegMaxEdges : batch);
    const size_t c = sample_ws_layout(sz, bt, nullptr, nullptr);
    return b > c ? b : c;
}

extern "C" int tpn_neg_sampler_build(const tpn_neg_sampler_t* s, const int64_t* src_dev, const int64_t* dst_dev,
                                     const double* t_dev, void* ws_dev, size_t ws_bytes, void* stream_v) {
    using namespace tpn;
    int rc = validate_neg(s);
    if (rc != TPN_OK) return rc;
    if (src_dev == nullptr || dst_dev == nullptr || ws_dev == nullptr || (s->timed && t_dev == nullptr))
        return TPN_ERR_INVALID_ARGUMENT;
    const long long E = s->num_edges;
    BuildWs ws;
    if (ws_bytes < build_ws_layout(E, ws_dev, &ws)) return TPN_ERR_WORKSPACE_TOO_SMALL;
    DeviceScope scope(s->counts);
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_v);
    const auto* src = reinterpret_cast<const long long*>(src_dev);
    const auto* dst = reinterpret_cast<const long long*>(dst_dev);
    const Count all{(int)E, nullptr};
    const int id_passes = passes_for_bits(s->id_bits);
    const unsigned g = grid_for(E);
    SortBufs b{ws.k, ws.v, ws.k2, ws.v2, ws.hist};
    if (cudaMemsetAsync(s->counts, 0, sizeof(int32_t) * TPN_NEG_COUNTS, stream) != cudaSuccess) {
        set_cuda_error(cudaGetLastError());
        return TPN_ERR_CUDA;
    }
    if (s->timed) {
        if (cudaMemsetAsync(s->mark, 0, sizeof(uint32_t) * (size_t)E, stream) != cudaSuccess) {
            set_cuda_error(cudaGetLastError());
            return TPN_ERR_CUDA;
        }
        // T: the edges stably sorted by time, low word then high word
        time_lo_kernel<<<g, 256, 0, stream>>>(t_dev, all, b.k, b.v);
        sort_passes(b, all, 0, 4, stream);
        time_hi_kernel<<<g, 256, 0, stream>>>(t_dev, all, b.v, b.k2, b.v2);
        b.swap();
        sort_passes(b, all, 0, 4, stream);
        fill_t_kernel<<<g, 256, 0, stream>>>(src, dst, t_dev, E, b.v, s->t_src, s->t_dst, s->t_time);
        // K: T positions stably by dst, then by src -> (src, dst, time); the first of each key has its first time
        gather_word_kernel<<<g, 256, 0, stream>>>(s->t_dst, nullptr, E, b.k2, b.v2);
        b.swap();
        sort_passes(b, all, 0, id_passes, stream);
        gather_word_kernel<<<g, 256, 0, stream>>>(s->t_src, b.v, E, b.k2, b.v2);
        b.swap();
        sort_passes(b, all, 0, id_passes, stream);
        scan_emit(KeyHead{b.v, s->t_src, s->t_dst},
                  KeyEmit{b.v, s->t_src, s->t_dst, s->t_time, ws.ksrc, ws.kdst, ws.kid_of_t, ws.kf}, all, ws.bsum,
                  s->counts + 0, stream);
        // F: K (in key order) stably by first time -> (f, src, dst)
        const Count keys{(int)E, s->counts + 0};
        time_lo_kernel<<<g, 256, 0, stream>>>(ws.kf, keys, b.k2, b.v2);
        b.swap();
        sort_passes(b, keys, 0, 4, stream);
        time_hi_kernel<<<g, 256, 0, stream>>>(ws.kf, keys, b.v, b.k2, b.v2);
        b.swap();
        sort_passes(b, keys, 0, 4, stream);
        fill_f_kernel<<<g, 256, 0, stream>>>(keys, b.v, ws.ksrc, ws.kdst, ws.kf, s->f_src, s->f_dst, s->f_time, b.k2);
        t_fpos_kernel<<<g, 256, 0, stream>>>(E, ws.kid_of_t, b.k2, s->t_fpos);
    }
    // S and D: sorted unique ids
    const long long* ids[2] = {src, dst};
    uint32_t* uniq[2] = {s->uniq_src, s->uniq_dst};
    for (int w = 0; w < 2; ++w) {
        ids_kernel<<<g, 256, 0, stream>>>(ids[w], E, b.k2, b.v2);
        b.swap();
        sort_passes(b, all, 0, id_passes, stream);
        scan_emit(IdHead{b.k}, IdEmit{b.k, uniq[w]}, all, ws.bsum, s->counts + 1 + w, stream);
    }
    return check_launch();
}

extern "C" int tpn_neg_sampler_sample(const tpn_neg_sampler_t* s, int strategy, uint64_t call, int64_t size,
                                      const int64_t* batch_src_dev, const int64_t* batch_dst_dev, int64_t batch,
                                      double start, double end, const double* start_dev, const double* end_dev,
                                      int64_t* out_src_dev, int64_t* out_dst_dev, void* ws_dev, size_t ws_bytes,
                                      void* stream_v) {
    using namespace tpn;
    int rc = validate_neg(s);
    if (rc != TPN_OK) return rc;
    if (strategy < TPN_NEG_RANDOM || strategy > TPN_NEG_INDUCTIVE || size < 0 || size > kNegMaxEdges || batch < 0 ||
        batch > kNegMaxEdges)
        return TPN_ERR_INVALID_ARGUMENT;
    if (size == 0) return TPN_OK;
    if (out_src_dev == nullptr || out_dst_dev == nullptr) return TPN_ERR_INVALID_ARGUMENT;
    DeviceScope scope(s->counts);
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_v);
    const NegView v = make_neg_view(s);
    auto* osrc = reinterpret_cast<long long*>(out_src_dev);
    auto* odst = reinterpret_cast<long long*>(out_dst_dev);
    if (strategy == TPN_NEG_RANDOM) {
        random_kernel<<<grid_for(size), 256, 0, stream>>>(v, call, size, osrc, odst);
        return check_launch();
    }
    if (!s->timed || ws_dev == nullptr || (batch > 0 && (batch_src_dev == nullptr || batch_dst_dev == nullptr)))
        return TPN_ERR_INVALID_ARGUMENT;
    SampleWs ws;
    if (ws_bytes < sample_ws_layout(size, batch, ws_dev, &ws)) return TPN_ERR_WORKSPACE_TOO_SMALL;
    const CallArgs c{strategy, call, size, batch, start, end, start_dev, end_dev};
    setup_kernel<<<1, 32, 0, stream>>>(v, c, ws.prm);
    // a fixed grid: the number of positions (k + x) is only known on the device, and a call whose window holds many
    // ties (day-quantised times) evaluates thousands of them; blocks past the work return at once
    long long gd = 2 * (long long)device_sm_count();
    if (gd > kDrawMaxBlocks) gd = kDrawMaxBlocks;
    const unsigned G = (unsigned)gd;
    mark_kernel<<<G, 256, 0, stream>>>(v, ws.prm);
    // the batch's pairs, sorted as 64-bit indices into S x D (the low word, then the high word if there is one)
    Batch bt{ws.k, ws.v, 0};
    if (batch > 0) {
        batch_keys_kernel<<<grid_for(batch), 256, 0, stream>>>(v, reinterpret_cast<const long long*>(batch_src_dev),
                                                                reinterpret_cast<const long long*>(batch_dst_dev), batch,
                                                                ws.k, ws.v);
        SortBufs b{ws.k, ws.v, ws.k2, ws.v2, ws.hist};
        const Count cb{(int)batch, nullptr};
        const int bits = 2 * s->id_bits + 1 < 64 ? 2 * s->id_bits + 1 : 64;     // |S||D| itself must sort too
        const int total = passes_for_bits(bits);
        sort_passes(b, cb, 0, total < 4 ? total : 4, stream);
        if (total > 4) {            // then stably by the high word, the low word riding along as the value
            SortBufs h{b.v, b.k, b.k2, b.v2, ws.hist};
            sort_passes(h, cb, 0, total - 4, stream);
            bt = Batch{h.v, h.k, batch};
        } else {
            bt = Batch{b.k, b.v, batch};
        }
        batch_count_kernel<<<grid_for(batch), 256, 0, stream>>>(v, bt.lo, bt.hi, batch, ws.prm);
    }
    draw_count_kernel<kNegTagHist><<<G, kDrawThreads, 0, stream>>>(v, ws.prm, bt, call, size, ws.bcount_h);
    draw_write_kernel<kNegTagHist><<<G, kDrawThreads, 0, stream>>>(v, ws.prm, bt, call, size, ws.bcount_h, ws.hist_idx,
                                                                    nullptr);
    draw_count_kernel<kNegTagFill><<<G, kDrawThreads, 0, stream>>>(v, ws.prm, bt, call, size, ws.bcount_f);
    draw_write_kernel<kNegTagFill><<<G, kDrawThreads, 0, stream>>>(v, ws.prm, bt, call, size, ws.bcount_f, nullptr,
                                                                    ws.fill_idx);
    finalize_kernel<<<grid_for(size), 256, 0, stream>>>(v, ws.prm, call, size, ws.hist_idx, ws.fill_idx, osrc, odst);
    unmark_kernel<<<G, 256, 0, stream>>>(v, ws.prm);
    return check_launch();
}

// Stable LSD radix sort of uint32 keys carrying uint32 values, 8-bit digits, two or three launches per pass
// (block histograms, optional prefix over blocks, scatter with warp-match ranking; integer atomics only on
// histogram counts).  Used by tpn_update.cu (messages by target) and tpn_sampler.cu (the streaming sampler's
// pending batch by node).  Each translation unit gets its own copy (anonymous namespace).
#pragma once

#include "tpn_common.cuh"

namespace tpn {
namespace {

constexpr int kRadixThreads = 256;
constexpr int kRadixItems = 8;
constexpr int kRadixTile = kRadixThreads * kRadixItems;   // 2048 keys per block
constexpr int kRadixBins = 256;
constexpr int kRadixDirectBlocks = 16;    // up to this many tiles the scatter sums the block histograms itself

// Number of messages of a call: known on the host (dev == nullptr: `cap` is the count), or produced on the
// device by the routing kernels of a sharded state (tpn_route.cu) and only bounded by `cap` on the host — grids
// are then sized for `cap` and every kernel reads the real count, so no launch depends on a device -> host copy.
struct Count {
    int cap;
    const int* dev;
    __device__ __forceinline__ int get() const {
        if (dev == nullptr) return cap;
        const int v = *dev;
        return v < 0 ? 0 : (v > cap ? cap : v);
    }
};

// one 2048-key tile: digit counts -> hist[tile][digit]  (bins: 256 shared counters)
__device__ __forceinline__ void hist_tile(uint32_t* bins, const uint32_t* __restrict__ key, int E, int shift,
                                          uint32_t* __restrict__ hist, int tile) {
    bins[threadIdx.x] = 0;
    __syncthreads();
    const int base = tile * kRadixTile;
#pragma unroll
    for (int i = 0; i < kRadixItems; ++i) {
        const int idx = base + i * kRadixThreads + threadIdx.x;
        if (idx < E) atomicAdd(&bins[(key[idx] >> shift) & 0xff], 1u);     // integer count: order-independent
    }
    __syncthreads();
    hist[tile * kRadixBins + threadIdx.x] = bins[threadIdx.x];     // [tile][digit]
}

__global__ void __launch_bounds__(kRadixThreads)
radix_hist_kernel(const uint32_t* __restrict__ key, Count count, int shift, uint32_t* __restrict__ hist) {
    __shared__ uint32_t bins[kRadixBins];
    const int E = count.get();
    if ((int)blockIdx.x * kRadixTile >= E) return;       // device-side count: tiles past the end do nothing
    hist_tile(bins, key, E, shift, hist, blockIdx.x);
}

// Many tiles (nblk > kRadixDirectBlocks): per digit, the exclusive prefix over blocks and the digit
// total, one warp per digit, in place ([block][digit] counts -> prefixes; totals in row nblk).
__device__ __forceinline__ void prefix_digit(uint32_t* __restrict__ hist, int nblk, int dgt, int lane) {
    uint32_t carry = 0;
    for (int b0 = 0; b0 < nblk; b0 += 32) {
        const int b = b0 + lane;
        const uint32_t c = b < nblk ? hist[b * kRadixBins + dgt] : 0u;
        uint32_t inc = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t nb = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += nb;
        }
        if (b < nblk) hist[b * kRadixBins + dgt] = carry + inc - c;
        carry += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane == 0) hist[nblk * kRadixBins + dgt] = carry;
}

__global__ void __launch_bounds__(256) radix_prefix_kernel(uint32_t* __restrict__ hist, Count count) {
    const int nblk = (count.get() + kRadixTile - 1) / kRadixTile;
    prefix_digit(hist, nblk, blockIdx.x * 8 + (threadIdx.x >> 5), threadIdx.x & 31);
}

constexpr int kRadixWarps = kRadixThreads / 32;
struct ScatterSmem {
    uint32_t wcount[kRadixWarps][kRadixBins + 1];
    uint32_t wtot[kRadixWarps];
};

// one 2048-key tile of a stable LSD pass
__device__ __forceinline__ void scatter_tile(ScatterSmem& sm, const uint32_t* __restrict__ kin,
                                             const uint32_t* __restrict__ vin, uint32_t* __restrict__ kout,
                                             uint32_t* __restrict__ vout, int E, int shift,
                                             const uint32_t* __restrict__ offs, int nblk, int prefixed, int tile,
                                             uint32_t* __restrict__ hist_next = nullptr) {
    constexpr int kWarps = kRadixWarps;
    uint32_t (&wcount)[kRadixWarps][kRadixBins + 1] = sm.wcount;
    uint32_t (&wtot)[kRadixWarps] = sm.wtot;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    for (int i = tid; i < kWarps * (kRadixBins + 1); i += kRadixThreads) (&wcount[0][0])[i] = 0;
    __syncthreads();
    // warp `wid` owns the contiguous chunk [base, base + 32*items): order inside the
    // tile is (warp, item, lane), which is the input order — the pass is stable.
    const int base = tile * kRadixTile + wid * (32 * kRadixItems);
    uint32_t k[kRadixItems], v[kRadixItems], rank[kRadixItems];
    const uint32_t lt_mask = (1u << lane) - 1u;
#pragma unroll
    for (int i = 0; i < kRadixItems; ++i) {
        const int idx = base + i * 32 + lane;
        const bool valid = idx < E;
        k[i] = valid ? kin[idx] : 0u;
        v[i] = valid ? vin[idx] : 0u;
        const uint32_t dgt = valid ? ((k[i] >> shift) & 0xff) : (uint32_t)kRadixBins;
        const uint32_t peers = __match_any_sync(0xffffffffu, dgt);
        const uint32_t before = wcount[wid][dgt];
        __syncwarp();
        if ((peers & lt_mask) == 0) wcount[wid][dgt] = before + __popc(peers);    // lowest peer lane updates
        __syncwarp();
        rank[i] = before + __popc(peers & lt_mask);
    }
    __syncthreads();
    {   // per digit: global offset of this block + exclusive prefix over warps.  The global offset
        // of (digit, block) = keys with a smaller digit + keys with this digit in earlier blocks,
        // summed here from the [block][digit] histogram (coalesced, L2-resident) — no scan launch.
        const int dgt = tid;    // kRadixThreads == kRadixBins
        uint32_t before = 0, total = 0;
        if (prefixed) {          // radix_prefix_kernel ran: prefixes in place, totals in row nblk
            before = offs[tile * kRadixBins + dgt];
            total = offs[nblk * kRadixBins + dgt];
        } else {
            for (int b0 = 0; b0 < nblk; b0 += 16) {          // 16 independent L2 loads per round
                uint32_t c[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) c[i] = b0 + i < nblk ? offs[(b0 + i) * kRadixBins + dgt] : 0u;
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    total += c[i];
                    before += b0 + i < tile ? c[i] : 0u;
                }
            }
        }
        uint32_t inc = total;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t nb = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += nb;
        }
        if (lane == 31) wtot[wid] = inc;
        __syncthreads();
        uint32_t wbase = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) wbase += w < wid ? wtot[w] : 0u;
        uint32_t run = wbase + inc - total + before;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
            const uint32_t c = wcount[w][dgt];
            wcount[w][dgt] = run;
            run += c;
        }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < kRadixItems; ++i) {
        const int idx = base + i * 32 + lane;
        if (idx < E) {
            const uint32_t dgt = (k[i] >> shift) & 0xff;
            const uint32_t pos = wcount[wid][dgt] + rank[i];
            kout[pos] = k[i];
            vout[pos] = v[i];
            // fused front end: the next pass's histogram of the output tile this key lands in (integer count)
            if (hist_next != nullptr)
                atomicAdd(&hist_next[(pos / kRadixTile) * kRadixBins + ((k[i] >> (shift + 8)) & 0xff)], 1u);
        }
    }
}

__global__ void __launch_bounds__(kRadixThreads)
radix_scatter_kernel(const uint32_t* __restrict__ kin, const uint32_t* __restrict__ vin,
                     uint32_t* __restrict__ kout, uint32_t* __restrict__ vout, Count count, int shift,
                     const uint32_t* __restrict__ offs, int prefixed) {
    __shared__ ScatterSmem sm;
    const int E = count.get();
    if ((int)blockIdx.x * kRadixTile >= E) return;
    const int nblk = (E + kRadixTile - 1) / kRadixTile;
    scatter_tile(sm, kin, vin, kout, vout, E, shift, offs, nblk, prefixed, blockIdx.x);
}

}  // namespace
}  // namespace tpn

// tpn_head_tc — the pair-wise head `self.mlp` on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//     y = W2 · relu(W1 · x + b1) + b2        (models/TPNet.py:64-65 and :125/:129), x: 64 features, 256 hidden
// This is the one dense contraction of the hot path ([n,64] x [64,256] x [256,64]).  The reference computes it in
// fp32; plain TF32 / FP16 would be narrower arithmetic, so every operand is SPLIT into two fp16 numbers,
//     v * 2^s = hi + lo,  hi = fp16(v * 2^s),  lo = fp16(v * 2^s - hi)            (22 significant bits, like 3xTF32)
// with an exact power-of-two scale 2^s (per row for the activations, per matrix for the weights) that keeps hi and lo
// in fp16's normal range, and each product is issued as THREE tensor-core MMAs with fp32 accumulation in TMEM:
//     A·B ≈ A_hi·B_lo + A_lo·B_hi + A_hi·B_hi        (the dropped A_lo·B_lo term is 2^-22 relative)
// The scales are undone exactly in the epilogues.  The tensor core adds each K = 16 block of products to the fp32
// accumulator with TRUNCATION (measured: the error of a plain 48-step accumulation, 1.0e-5, is reproduced exactly by
// an emulation that truncates, 1.1e-5, and not by one that rounds, 2.0e-6), so the number of additions at full
// magnitude is kept small: the two small cross products go first, the hi·hi product last (4 additions per
// accumulator instead of 12), and GEMM2 uses one accumulator per 64-column K chunk, summed in fp32 by the epilogue.
// Measured error against the float64 head: see profiles/r02_head_bench.json (packed-FFMA kernel 2.0e-6, cuBLAS 4.6e-6).
//
// One persistent CTA per SM, 128 pairs per tile:
//   warps 0-3 ("row workers", thread r <-> pair r of the tile <-> TMEM lane r): load and split the X rows into the
//       canonical K-major shared-memory layout; epilogue 1 (TMEM -> bias + ReLU -> split -> shared memory, in 64-column
//       chunks that feed GEMM2 while the next chunk is converted); epilogue 2 (TMEM -> bias -> global).
//   warp 4, one elected thread: issues tcgen05.mma (GEMM1: M128 N256 K16 x 4 k-steps x 3 products into TMEM columns
//       0..255; GEMM2: M128 N64 K16 x 16 k-steps x 3 products into columns 256..511, one 64-column accumulator per
//       K chunk) and tcgen05.commit to mbarriers.
//   Both weight matrices stay in shared memory for the whole launch, split and laid out once per CTA (128 KB).
// Operand layout: UMMA "K-major, no swizzle" canonical form — 8-row x 16-byte core matrices, consecutive along K
// (LBO = 128 B), 8-row groups 1024 B apart (SBO) — described to the tensor core by 64-bit shared-memory descriptors.
// Every mbarrier wait is bounded (a lost arrival traps instead of hanging the GPU).
#include <cuda_fp16.h>
#include <float.h>

#include "tpn_common.cuh"

namespace tpn {

namespace {

constexpr int kF = 64;                 // features in / out
constexpr int kHid = 256;              // hidden units
constexpr int kTile = 128;             // pairs per tile = UMMA M = TMEM lanes
constexpr int kTcThreads = 160;        // 4 row-worker warps + the MMA warp
constexpr uint32_t kTmemCols = 512;    // D1: 256 columns; D2: 4 accumulators (one per K chunk) x 64 columns
constexpr uint32_t kD2Col = 256;
constexpr uint32_t kLbo = 128;         // bytes between the two 16-byte K chunks of one MMA (core matrices along K)
constexpr uint32_t kSbo = 1024;        // bytes between 8-row groups (K = 64 halfs = 8 core matrices of 128 B)
constexpr uint32_t kKStepBytes = 256;  // one MMA consumes K = 16 halfs = 2 core matrices

struct TcSmem {
    __half w1[2][kHid * kF];           // [hi|lo] B of GEMM1: 256 rows (hidden unit) x K = 64          64 KB
    __half w2[2][4][kF * 64];          // [hi|lo][k chunk] B of GEMM2: 64 rows (output) x K = 64        64 KB
    __half x[2][kTile * kF];           // [hi|lo] A of GEMM1: 128 rows (pair) x K = 64                   32 KB
    __half h[2][2][kTile * 64];        // [buffer][hi|lo] A of GEMM2: one 64-column chunk of the hidden   64 KB
    float b1[kHid];
    float b2[kF];
    uint64_t x_full, d1_full, d2_full, h_full[2], h_empty[2];
    uint32_t tmem_base;
    float red[8];
    int w1_exp, w2_exp;                // exponents of the power-of-two scales of W1, W2
};

// element (row, k) of a K = 64 operand in the canonical layout, in halfs
__device__ __forceinline__ int canon(int row, int k) { return (row >> 3) * 512 + (k >> 3) * 64 + (row & 7) * 8 + (k & 7); }

__device__ __forceinline__ uint64_t smem_desc(const void* p) {
    const uint32_t addr = smem_u32(p);
    uint64_t d = (uint64_t)((addr & 0x3FFFFu) >> 4);             // start address, 16-byte units        bits [0,14)
    d |= (uint64_t)(kLbo >> 4) << 16;                            // leading-dimension byte offset        bits [16,30)
    d |= (uint64_t)(kSbo >> 4) << 32;                            // stride-dimension byte offset         bits [32,46)
    d |= (uint64_t)1 << 46;                                      // descriptor version (Blackwell)       bits [46,48)
    return d;                                                    // base offset 0, layout type 0 = no swizzle
}

// kind::f16 instruction descriptor: D = F32, A = B = F16, both K-major, N / 8 at bit 17, M / 16 at bit 24
__device__ __forceinline__ constexpr uint32_t instr_desc(int m, int n) {
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ void mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t* bar) {       // arrives on `bar` when every MMA issued so far is done
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// the same load without the wait: several loads are issued back to back and waited for once (tmem_ld_wait)
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// bounded wait: a lost arrival becomes a trap (an error the host sees), never a hung GPU
__device__ __forceinline__ void mbar_wait_bounded(uint64_t* bar, uint32_t parity) {
    const long long t0 = clock64();
    for (;;) {
        uint32_t done;
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}" : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (done) return;
        if (clock64() - t0 > 4000000000ll) __trap();
    }
}

// 8 consecutive values -> hi / lo fp16 octets (16 bytes each)
__device__ __forceinline__ void split8(const float (&v)[8], uint4& hi, uint4& lo) {
    __half2 h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __half a = __float2half_rn(v[2 * i]), b = __float2half_rn(v[2 * i + 1]);
        h[i] = __halves2half2(a, b);
        l[i] = __halves2half2(__float2half_rn(v[2 * i] - __half2float(a)), __float2half_rn(v[2 * i + 1] - __half2float(b)));
    }
    hi = make_uint4(*reinterpret_cast<uint32_t*>(&h[0]), *reinterpret_cast<uint32_t*>(&h[1]),
                    *reinterpret_cast<uint32_t*>(&h[2]), *reinterpret_cast<uint32_t*>(&h[3]));
    lo = make_uint4(*reinterpret_cast<uint32_t*>(&l[0]), *reinterpret_cast<uint32_t*>(&l[1]),
                    *reinterpret_cast<uint32_t*>(&l[2]), *reinterpret_cast<uint32_t*>(&l[3]));
}

// exponent s of the power-of-two scale 2^s that puts `vmax` into [2^13, 2^14): hi = fp16(v * 2^s) is then far from
// fp16's overflow (2^16) and lo (about 2^-11 of hi) is a normal fp16 for every element within 2^-16 of the row /
// matrix maximum.  s spans -114 (vmax near FLT_MAX) .. 162 (vmax = 2^-149); 0 for a zero, inf or NaN maximum.
__device__ __forceinline__ int pow2_exp(float vmax) {
    if (!(vmax > 0.f) || !(vmax <= FLT_MAX)) return 0;
    int e;
    (void)frexpf(vmax, &e);                                      // vmax = m * 2^e, m in [0.5, 1)
    return 14 - e;
}

// 2^s as two exact power-of-two factors, pre * post.  pre = 1 whenever 2^s is a float itself (s in [-149, 127]), so
// one multiply (or fmaf) by `post` is the whole operation there; otherwise v * pre stays in the normal range whenever
// v * 2^s does.  s is clamped to [-252, 254]: past that every product of the head under- or overflows anyway.
struct Pow2 {
    float pre, post;
};
__device__ __forceinline__ Pow2 pow2(int s) {
    s = s > 254 ? 254 : (s < -252 ? -252 : s);
    const int p = s > 127 ? s - 127 : (s < -149 ? s + 126 : 0);
    return {ldexpf(1.0f, p), ldexpf(1.0f, s - p)};
}

// v *= f over one 64-column chunk (rare: the scale is outside the float range, see pow2)
__device__ __forceinline__ void scale64(float (&d0)[32], float (&d1)[32], float f) {
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        d0[j] *= f;
        d1[j] *= f;
    }
}

__global__ void __launch_bounds__(kTcThreads, 1)
head_tc_kernel(const float* __restrict__ x, long long n, const float* __restrict__ w1, const float* __restrict__ b1,
               const float* __restrict__ w2, const float* __restrict__ b2, float* __restrict__ y,
               const int* __restrict__ n_dev) {
    if (n_dev != nullptr) n = min(n, (long long)max(*n_dev, 0));      // routed calls: the count lives on the device
    extern __shared__ __align__(128) unsigned char tc_raw[];
    TcSmem& sm = *reinterpret_cast<TcSmem*>(tc_raw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long ntiles = (n + kTile - 1) / kTile;

    // ---- one-time set-up: barriers, TMEM, weights
    if (tid == 0) {
        mbar_init(&sm.x_full, kTile);
        mbar_init(&sm.d1_full, 1);
        mbar_init(&sm.d2_full, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&sm.h_full[i], kTile);
            mbar_init(&sm.h_empty[i], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sm.tmem_base)),
                     "r"(kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // weight scales: max |W1|, max |W2| over the whole matrices (every CTA computes the same value)
    {
        float m1 = 0.f, m2 = 0.f;
        for (int i = tid; i < kHid * kF / 4; i += kTcThreads) {
            const float4 a = ld4(w1 + 4 * i), b = ld4(w2 + 4 * i);
            m1 = fmaxf(m1, fmaxf(fmaxf(fabsf(a.x), fabsf(a.y)), fmaxf(fabsf(a.z), fabsf(a.w))));
            m2 = fmaxf(m2, fmaxf(fmaxf(fabsf(b.x), fabsf(b.y)), fmaxf(fabsf(b.z), fabsf(b.w))));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, o));
            m2 = fmaxf(m2, __shfl_xor_sync(0xffffffffu, m2, o));
        }
        if (lane == 0) sm.red[warp] = m1;                  // warps 0..4
        __syncthreads();
        float t1 = 0.f;
        for (int wq = 0; wq < 5; ++wq) t1 = fmaxf(t1, sm.red[wq]);
        __syncthreads();
        if (lane == 0) sm.red[warp] = m2;
        __syncthreads();
        float t2 = 0.f;
        for (int wq = 0; wq < 5; ++wq) t2 = fmaxf(t2, sm.red[wq]);
        const int e1 = pow2_exp(t1), e2 = pow2_exp(t2);
        const Pow2 s1 = pow2(e1), s2 = pow2(e2);
        if (tid == 0) {
            sm.w1_exp = e1;
            sm.w2_exp = e2;
        }
        // split + canonical layout, one 16-byte K chunk (8 values) per step
        for (int c = tid; c < kHid * kF / 8; c += kTcThreads) {        // W1[h][k]: row h, chunk k8
            const int row = c >> 3, k8 = c & 7;
            const float4 a = ld4(w1 + row * kF + k8 * 8), b = ld4(w1 + row * kF + k8 * 8 + 4);
            float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = v[j] * s1.pre * s1.post;
            uint4 hi, lo;
            split8(v, hi, lo);
            *reinterpret_cast<uint4*>(&sm.w1[0][canon(row, k8 * 8)]) = hi;
            *reinterpret_cast<uint4*>(&sm.w1[1][canon(row, k8 * 8)]) = lo;
        }
        for (int c = tid; c < kF * kHid / 8; c += kTcThreads) {        // W2[o][h]: row o, K chunk = h / 64
            const int row = c >> 5, k8 = c & 31;
            const float4 a = ld4(w2 + row * kHid + k8 * 8), b = ld4(w2 + row * kHid + k8 * 8 + 4);
            float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = v[j] * s2.pre * s2.post;
            uint4 hi, lo;
            split8(v, hi, lo);
            const int kc = k8 >> 3, kk = (k8 & 7) * 8;
            *reinterpret_cast<uint4*>(&sm.w2[0][kc][canon(row, kk)]) = hi;
            *reinterpret_cast<uint4*>(&sm.w2[1][kc][canon(row, kk)]) = lo;
        }
        for (int i = tid; i < kHid; i += kTcThreads) sm.b1[i] = b1[i];
        for (int i = tid; i < kF; i += kTcThreads) sm.b2[i] = b2[i];
    }
    fence_proxy_async_smem();             // the weights were written by the generic proxy, the tensor core reads them
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = sm.tmem_base;
    const int w1_exp = sm.w1_exp, w2_exp = sm.w2_exp;

    uint32_t it = 0;                      // tiles done by this CTA (phase of the once-per-tile barriers)
    if (warp < 4) {
        // =================================================================== row workers
        // Software pipeline over the tiles of this CTA: the X rows of tile i+1 are loaded into registers while tile
        // i is in its epilogues, and they are split into shared memory as soon as epilogue 1 of tile i has drained
        // D1 — so GEMM1(i+1) runs on the tensor core while the workers are in epilogue 2 of tile i.
        const int r = tid;                                   // pair of the tile == TMEM lane
        const uint32_t lane_base = (uint32_t)(warp * 32) << 16;      // a warp reaches TMEM lanes [32 * (warp % 4), + 32)
        float4 xn[kF / 4];                                   // X row of the NEXT tile (in flight / waiting to be split)
        auto load_x = [&](long long tile) {
            const long long row = tile * kTile + r;
            const bool ok = tile < ntiles && row < n;
#pragma unroll
            for (int q = 0; q < kF / 4; ++q) xn[q] = ok ? ld4(x + row * kF + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
        };
        // xn -> scaled, split, canonical layout; returns the exponent of 1 / (row scale * W1 scale)
        auto split_x = [&]() -> int {
            float vmax = 0.f;
#pragma unroll
            for (int q = 0; q < kF / 4; ++q)
                vmax = fmaxf(vmax, fmaxf(fmaxf(fabsf(xn[q].x), fabsf(xn[q].y)), fmaxf(fabsf(xn[q].z), fabsf(xn[q].w))));
            const int ex = pow2_exp(vmax);
            const Pow2 p = pow2(ex);
            if (p.pre != 1.0f) {                             // rows below 2^-113: two exact steps
#pragma unroll
                for (int q = 0; q < kF / 4; ++q) scale4(xn[q], p.pre);
            }
            const float sx = p.post;
#pragma unroll
            for (int k8 = 0; k8 < kF / 8; ++k8) {
                const float4 a = xn[2 * k8], b = xn[2 * k8 + 1];
                const float v[8] = {a.x * sx, a.y * sx, a.z * sx, a.w * sx, b.x * sx, b.y * sx, b.z * sx, b.w * sx};
                uint4 hi, lo;
                split8(v, hi, lo);
                *reinterpret_cast<uint4*>(&sm.x[0][canon(r, k8 * 8)]) = hi;
                *reinterpret_cast<uint4*>(&sm.x[1][canon(r, k8 * 8)]) = lo;
            }
            fence_proxy_async_smem();
            tc_fence_before();            // this thread's TMEM reads of the previous tile are ordered before the arrival
            mbar_arrive(&sm.x_full);
            return -(w1_exp + ex);
        };
        long long tile = blockIdx.x;
        load_x(tile);
        int undo1 = split_x();
        load_x(tile + gridDim.x);
        for (; tile < ntiles; tile += gridDim.x, ++it) {
            const long long row = tile * kTile + r;
            const bool valid = row < n;
            // ---- epilogue 1: h = relu(D1 / (sx * s1) + b1), one 64-column chunk at a time; every chunk gets its own
            // power-of-two scale (its own row maximum), undone per chunk in epilogue 2 — no separate maximum pass
            mbar_wait_bounded(&sm.d1_full, it & 1u);
            tc_fence_after();
            const Pow2 u1 = pow2(undo1);
            int undo2[4];
#pragma unroll 1
            for (int c = 0; c < 4; ++c) {
                const int buf = c & 1;
                const uint32_t use = it * 2u + (uint32_t)(c >> 1);
                float d0[32], d1[32];
                tmem_ld32_nowait(tmem + lane_base + (uint32_t)(c * 64), d0);
                tmem_ld32_nowait(tmem + lane_base + (uint32_t)(c * 64 + 32), d1);
                tmem_ld_wait();
                if (u1.pre != 1.0f) scale64(d0, d1, u1.pre);
                float hmax = 0.f;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    d0[j] = relu(fmaf(d0[j], u1.post, sm.b1[c * 64 + j]));
                    d1[j] = relu(fmaf(d1[j], u1.post, sm.b1[c * 64 + 32 + j]));
                    hmax = fmaxf(hmax, fmaxf(d0[j], d1[j]));
                }
                const int eh = pow2_exp(hmax);
                const Pow2 ph = pow2(eh);
                if (ph.pre != 1.0f) scale64(d0, d1, ph.pre);
                const float sh = ph.post;
                undo2[c] = -(w2_exp + eh);
                mbar_wait_bounded(&sm.h_empty[buf], (use & 1u) ^ 1u);       // GEMM2 is done with this buffer
#pragma unroll
                for (int k8 = 0; k8 < 8; ++k8) {
                    float v[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = (k8 < 4 ? d0[k8 * 8 + j] : d1[(k8 - 4) * 8 + j]) * sh;
                    uint4 hi, lo;
                    split8(v, hi, lo);
                    *reinterpret_cast<uint4*>(&sm.h[buf][0][canon(r, k8 * 8)]) = hi;
                    *reinterpret_cast<uint4*>(&sm.h[buf][1][canon(r, k8 * 8)]) = lo;
                }
                fence_proxy_async_smem();
                mbar_arrive(&sm.h_full[buf]);
            }
            // ---- D1 is drained and GEMM1 of this tile completed long ago: hand the next tile's X to the tensor core
            const Pow2 u2_0 = pow2(undo2[0]), u2_1 = pow2(undo2[1]), u2_2 = pow2(undo2[2]), u2_3 = pow2(undo2[3]);
            if (tile + gridDim.x < ntiles) {
                undo1 = split_x();
                load_x(tile + 2 * (long long)gridDim.x);
            }
            // ---- epilogue 2: y = sum over the K chunks of D2_c / (sh_c * s2), + b2
            mbar_wait_bounded(&sm.d2_full, it & 1u);
            tc_fence_after();
#pragma unroll 1
            for (int half = 0; half < 2; ++half) {
                float d[32];
                {   // the four K-chunk accumulators, each with its own scale, summed pairwise in fp32
                    float d1[32], d2[32], d3[32];
                    tmem_ld32_nowait(tmem + lane_base + kD2Col + (uint32_t)(half * 32), d);
                    tmem_ld32_nowait(tmem + lane_base + kD2Col + 64u + (uint32_t)(half * 32), d1);
                    tmem_ld32_nowait(tmem + lane_base + kD2Col + 128u + (uint32_t)(half * 32), d2);
                    tmem_ld32_nowait(tmem + lane_base + kD2Col + 192u + (uint32_t)(half * 32), d3);
                    tmem_ld_wait();
                    if (u2_0.pre != 1.0f || u2_1.pre != 1.0f || u2_2.pre != 1.0f || u2_3.pre != 1.0f) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            d[j] *= u2_0.pre;
                            d1[j] *= u2_1.pre;
                            d2[j] *= u2_2.pre;
                            d3[j] *= u2_3.pre;
                        }
                    }
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        d[j] = (d[j] * u2_0.post + d1[j] * u2_1.post) + (d2[j] * u2_2.post + d3[j] * u2_3.post);
                }
                if (valid) {
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const int o = half * 32 + q * 4;
                        st4(y + row * kF + o, make_float4(d[q * 4] + sm.b2[o], d[q * 4 + 1] + sm.b2[o + 1],
                                                          d[q * 4 + 2] + sm.b2[o + 2], d[q * 4 + 3] + sm.b2[o + 3]));
                    }
                }
            }
            tc_fence_before();            // the TMEM reads of this tile are ordered before the next tile's arrivals
        }
    } else if (lane == 0) {
        // =================================================================== MMA issuer (one thread)
        constexpr uint32_t idesc1 = instr_desc(kTile, kHid), idesc2 = instr_desc(kTile, kF);
        const uint64_t xa[2] = {smem_desc(sm.x[0]), smem_desc(sm.x[1])};
        const uint64_t wb[2] = {smem_desc(sm.w1[0]), smem_desc(sm.w1[1])};
        // GEMM1 of one tile: small cross products first, hi * hi last (only its 4 additions happen at full magnitude)
        auto gemm1 = [&](uint32_t t) {
            mbar_wait_bounded(&sm.x_full, t & 1u);     // X of tile t is in shared memory — and D1 of tile t-1 is drained
            tc_fence_after();
#pragma unroll
            for (int ks = 0; ks < kF / 16; ++ks) {
                const uint64_t adv = (uint64_t)((ks * kKStepBytes) >> 4);
                mma_f16(tmem, xa[0] + adv, wb[1] + adv, idesc1, ks > 0 ? 1u : 0u);       // hi * lo
                mma_f16(tmem, xa[1] + adv, wb[0] + adv, idesc1, 1u);                    // lo * hi
            }
#pragma unroll
            for (int ks = 0; ks < kF / 16; ++ks) {
                const uint64_t adv = (uint64_t)((ks * kKStepBytes) >> 4);
                mma_f16(tmem, xa[0] + adv, wb[0] + adv, idesc1, 1u);                    // hi * hi
            }
            mma_commit(&sm.d1_full);
        };
        long long tile = blockIdx.x;
        if (tile < ntiles) gemm1(0);
        for (; tile < ntiles; tile += gridDim.x, ++it) {
#pragma unroll 1
            for (int c = 0; c < 4; ++c) {
                const int buf = c & 1;
                const uint32_t use = it * 2u + (uint32_t)(c >> 1);
                mbar_wait_bounded(&sm.h_full[buf], use & 1u);
                tc_fence_after();
                const uint64_t ha[2] = {smem_desc(sm.h[buf][0]), smem_desc(sm.h[buf][1])};
                const uint64_t vb[2] = {smem_desc(sm.w2[0][c]), smem_desc(sm.w2[1][c])};
                const uint32_t dacc = tmem + kD2Col + (uint32_t)(c * 64);       // this chunk's own accumulator
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                    const uint64_t adv = (uint64_t)((ks * kKStepBytes) >> 4);
                    mma_f16(dacc, ha[0] + adv, vb[1] + adv, idesc2, ks > 0 ? 1u : 0u);  // hi * lo
                    mma_f16(dacc, ha[1] + adv, vb[0] + adv, idesc2, 1u);                // lo * hi
                }
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                    const uint64_t adv = (uint64_t)((ks * kKStepBytes) >> 4);
                    mma_f16(dacc, ha[0] + adv, vb[0] + adv, idesc2, 1u);                // hi * hi
                }
                mma_commit(&sm.h_empty[buf]);
            }
            mma_commit(&sm.d2_full);
            // GEMM1 of the next tile runs while the workers are in epilogue 2 of this one
            if (tile + gridDim.x < ntiles) gemm1(it + 1u);
        }
    }

    // ---- teardown: every tcgen05 operation of this CTA has completed (the workers waited for their loads)
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols) : "memory");
    }
}

}  // namespace

// Launch of the tensor-core head (tpn_head.cu decides when it is used).  Returns TPN_OK or an error code.
int launch_head_tensor(const float* x, long long n, const int* n_dev, const float* w1, const float* b1, const float* w2,
                       const float* b2, float* y, int dev_slot, cudaStream_t stream) {
    static bool configured_tab[kMaxDevices];
    bool& configured = configured_tab[dev_slot];
    const int smem = (int)sizeof(TcSmem);                    // operands need 16-byte alignment only (no swizzle)
    if (!configured) {
        const cudaError_t e = cudaFuncSetAttribute(head_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) {
            set_cuda_error(e);
            return TPN_ERR_CUDA;
        }
        configured = true;
    }
    const long long ntiles = (n + kTile - 1) / kTile;
    const int sms = device_sm_count();
    const unsigned grid = (unsigned)(ntiles < sms ? ntiles : sms);
    head_tc_kernel<<<grid, kTcThreads, smem, stream>>>(x, n, w1, b1, w2, b2, y, n_dev);
    return TPN_OK;
}

}  // namespace tpn

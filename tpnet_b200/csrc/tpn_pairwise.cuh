// Device helpers shared by the pair-wise encoder kernels (tpn_pairwise.cu, tpn_pairwise_nbr.cu):
// packed-FFMA2 Gram accumulation, the transposing butterfly reduce, the branch-free log of the
// epilogue (TPNet.py:127-128) and the mbarrier / bulk-copy (TMA) wrappers.
#pragma once

#include "tpn_common.cuh"

namespace tpn {
namespace {

constexpr int kPairThreads = 128;

__device__ __forceinline__ float2 lo2(const float4& v) { return make_float2(v.x, v.y); }
__device__ __forceinline__ float2 hi2(const float4& v) { return make_float2(v.z, v.w); }


// log(x) for finite x >= 1 (the epilogue passes NaN and +inf around it): exponent /
// mantissa split with m in [2/3, 4/3) and a minimax polynomial for log1p(m - 1), evaluated
// with FMAs and no special-case branches (inputs are never zero, negative, inf or denormal).
// Checked against float64 log over [1, 1e6]: max error 0.85 ulp (torch's CPU log is <= 1 ulp).
__device__ __forceinline__ float log_ge1(float a) {
    const int ia = __float_as_int(a);
    const int e = (ia - 0x3f2aaaab) & 0xff800000;
    const float fe = (float)e * 1.19209290e-7f;           // unbiased exponent (e / 2^23)
    const float m = __int_as_float(ia - e) - 1.0f;        // exact
    const float s = m * m;
    float r = -0.130310059f, t = 0.140869141f;
    r = fmaf(r, s, -0.121483512f);
    t = fmaf(t, s, 0.139814854f);
    r = fmaf(r, s, -0.166846126f);
    t = fmaf(t, s, 0.200120345f);
    r = fmaf(r, s, -0.249996200f);
    r = fmaf(t, m, r);
    r = fmaf(r, m, 0.333331972f);
    r = fmaf(r, m, -0.500000000f);
    r = fmaf(r, s, m);
    return fmaf(fe, 0.693147182f, r);
}

// unique Gram entry e (row-major over the upper triangle) -> (r << 8 | q)
template <int R>
__device__ __forceinline__ void fill_entry_table(unsigned short* tab, int lane) {
    constexpr int NU = R * (R + 1) / 2;
    for (int e = lane; e < NU; e += 32) {
        int r = 0, rem = e;
        while (rem >= R - r) { rem -= R - r; ++r; }
        tab[e] = (unsigned short)((r << 8) | (r + rem));
    }
}

// One butterfly step over N live values: lanes whose `mask` bit is set keep the upper half.
template <int N>
__device__ __forceinline__ void halve(float (&v)[N], int n, int mask, bool upper) {
#pragma unroll
    for (int i = 0; i < N / 2; ++i) {
        if (i < n / 2) {
            const float send = upper ? v[i] : v[i + n / 2];
            const float keep = upper ? v[i + n / 2] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, mask);
        }
    }
}


template <int R>
__device__ __forceinline__ void gram_step(float2 (&acc)[R * (R + 1) / 2], const float4 (&x)[R]) {
    int e = 0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const float2 rl = lo2(x[r]), rh = hi2(x[r]);
#pragma unroll
        for (int q = r; q < R; ++q) {
            acc[e] = __ffma2_rn(rl, lo2(x[q]), acc[e]);
            acc[e] = __ffma2_rn(rh, hi2(x[q]), acc[e]);
            ++e;
        }
    }
}

// The reference's epilogue (TPNet.py:127-128): rf[rf < 0] = 0; log(rf + 1.0).  The clamp is a compare, not fmaxf,
// so NaN stays NaN, and NaN / +inf skip the polynomial (log_ge1 is finite for them): NaN -> NaN, +inf -> +inf,
// -inf -> 0, as torch gives.  Branch-free; finite inputs take exactly the ops of the polynomial.
__device__ __forceinline__ float epilogue(float g, int apply_log_scale) {
    if (apply_log_scale) {
        const float a = __fadd_rn(g < 0.f ? 0.f : g, 1.0f);       // torch.log(x + 1.0), not log1p
        const float r = log_ge1(a);
        g = a < INFINITY ? r : a;
    }
    return g;
}

// Reduce the partial Gram sums over the G lanes of a group with a transposing butterfly
// (each shuffle step halves the number of live values, so every lane ends up owning NP/G
// finished entries), apply clamp + log(x + 1.0) to just those, and mirror them into the
// group's R x R tile in shared memory.
template <int R, int G>
__device__ __forceinline__ void finish_pair(const float2 (&acc)[R * (R + 1) / 2], int gl, float* mine,
                                            const unsigned short* tab, int apply_log_scale) {
    constexpr int NU = R * (R + 1) / 2;
    constexpr int NP = (NU + G - 1) / G * G;
    float s[NP];
#pragma unroll
    for (int i = 0; i < NP; ++i) s[i] = i < NU ? acc[i].x + acc[i].y : 0.f;
    int first = 0;                         // index of the entry held in s[0] after the reduction
    int nlive = NP;
#pragma unroll
    for (int mask = G / 2; mask >= 1; mask >>= 1) {
        const bool upper = (gl & mask) != 0;
        halve<NP>(s, nlive, mask, upper);
        nlive >>= 1;
        if (upper) first += nlive;
    }
#pragma unroll
    for (int k = 0; k < NP / G; ++k) {
        const int e = first + k;
        if (e < NU) {
            const int rq = tab[e];
            const int r = rq >> 8, q = rq & 0xff;
            const float g = epilogue(s[k], apply_log_scale);
            mine[r * R + q] = g;
            mine[q * R + r] = g;
        }
    }
}

}  // namespace
}  // namespace tpn

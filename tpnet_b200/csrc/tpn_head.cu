// tpn_head — forward of the pair-wise head `self.mlp` for inference (no autograd):
//     y = W2 · relu(W1 · x + b1) + b2        (models/TPNet.py:64-65 and :125/:129)
// for the default 3-layer configuration: x = 64 features per pair, 256 hidden units, 64 outputs.
// Training keeps the head in PyTorch (autograd); this kernel serves the no-grad paths
// (evaluate_link_prediction.py, validation) where cuBLAS' fp32 SIMT GEMM runs the skinny
// [n,64]x[64,256]x[256,64] chain at ~17 TFLOP/s and round-trips the hidden layer through HBM.
//
// One persistent CTA per SM keeps BOTH weight matrices in shared memory (2 x 64 KB, transposed so
// that a k-step reads contiguous rows) and walks over tiles of 64 pairs:
//   phase 1  H[64 pairs][256] = relu(X · W1ᵀ + b1): 256 threads x (8 pairs x 8 hidden units), packed
//            FFMA2 (two hidden units per instruction), operands read as conflict-free 128-bit LDS;
//   phase 2  Y[64 pairs][64]  = H · W2ᵀ + b2: the 256 hidden units are split over 4 thread groups
//            (split-K), each thread again an 8 x 8 tile with FFMA2; the 4 partial tiles are summed
//            through shared memory in a fixed order (deterministic), bias added, stored coalesced.
// The hidden layer never leaves the SM.  fp32 throughout (no TF32): results differ from cuBLAS only
// in summation order.
#include "tpn_common.cuh"

namespace tpn {
namespace {

constexpr int kHeadF = 64;             // features in / out
constexpr int kHeadHid = 256;          // hidden units
constexpr int kHeadTile = 64;          // pairs per tile
constexpr int kHeadThreads = 256;

constexpr int kXStride = kHeadF + 4;        // padded rows: 8 consecutive rows hit 8 different 16-byte bank groups
constexpr int kHStride = kHeadHid + 4;

struct HeadSmem {
    float w1t[kHeadF][kHeadHid];       // W1ᵀ: [k][h]            64 KB
    float w2t[kHeadHid][kHeadF];       // W2ᵀ: [h][o]            64 KB
    float hs[kHeadTile][kHStride];     // H:   [pair][h]         65 KB (then the 4 partial Y tiles, 64 KB)
    float xs[kHeadTile][kXStride];     // X:   [pair][k]         17 KB
    float b1[kHeadHid];
    float b2[kHeadF];
};

__device__ __forceinline__ float2 splat(float v) { return make_float2(v, v); }
__device__ __forceinline__ float pick(const float4& v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w)); }

// acc[p][0..3] += a[p] * (wa.xy, wa.zw, wb.xy, wb.zw) for the 8 rows of the thread's tile
__device__ __forceinline__ void tile_fma(float2 (&acc)[8][4], const float (&a)[8], const float4& wa, const float4& wb) {
    const float2 w0 = make_float2(wa.x, wa.y), w1 = make_float2(wa.z, wa.w);
    const float2 w2 = make_float2(wb.x, wb.y), w3 = make_float2(wb.z, wb.w);
#pragma unroll
    for (int p = 0; p < 8; ++p) {
        const float2 ap = splat(a[p]);
        acc[p][0] = __ffma2_rn(ap, w0, acc[p][0]);
        acc[p][1] = __ffma2_rn(ap, w1, acc[p][1]);
        acc[p][2] = __ffma2_rn(ap, w2, acc[p][2]);
        acc[p][3] = __ffma2_rn(ap, w3, acc[p][3]);
    }
}

__global__ void __launch_bounds__(kHeadThreads, 1)
head_forward_kernel(const float* __restrict__ x, long long n, const float* __restrict__ w1,
                    const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ b2,
                    float* __restrict__ y, const int* __restrict__ n_dev) {
    if (n_dev != nullptr) n = min(n, (long long)max(*n_dev, 0));      // routed calls: the count lives on the device
    extern __shared__ __align__(16) unsigned char head_raw[];
    HeadSmem& sm = *reinterpret_cast<HeadSmem*>(head_raw);
    const int tid = threadIdx.x;
    // weights, transposed once per CTA (W1 is [256][64] row-major as nn.Linear keeps it, W2 is [64][256]);
    // consecutive threads write consecutive shared-memory words
    for (int i = tid; i < kHeadF * kHeadHid; i += kHeadThreads) {
        const int k = i / kHeadHid, h = i - k * kHeadHid;
        sm.w1t[k][h] = w1[h * kHeadF + k];
    }
    for (int i = tid; i < kHeadHid * kHeadF; i += kHeadThreads) {
        const int h = i / kHeadF, o = i - h * kHeadF;
        sm.w2t[h][o] = w2[o * kHeadHid + h];
    }
    if (tid < kHeadHid) sm.b1[tid] = b1[tid];
    if (tid < kHeadF) sm.b2[tid] = b2[tid];

    const long long ntiles = (n + kHeadTile - 1) / kHeadTile;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long p0 = tile * kHeadTile;
        __syncthreads();                                    // weights ready / previous tile fully consumed
        {   // X tile: thread (pair = tid % 64, quarter = tid / 64) copies 16 consecutive features of its pair
            const int p = tid & 63, qd = tid >> 6;
            const long long gp = p0 + p < n ? p0 + p : n - 1;
            const float4* src = reinterpret_cast<const float4*>(x + gp * kHeadF + qd * 16);
#pragma unroll
            for (int j = 0; j < 4; ++j) *reinterpret_cast<float4*>(&sm.xs[p][qd * 16 + 4 * j]) = src[j];
        }
        __syncthreads();
        // ---- phase 1: thread = pairs {ty + 8p} x hidden units {4tx..4tx+3} U {128+4tx..128+4tx+3}
        {
            const int ty = tid >> 5, tx = tid & 31;
            float2 acc[8][4];
            {
                const float4 ba = *reinterpret_cast<const float4*>(&sm.b1[tx * 4]);
                const float4 bb = *reinterpret_cast<const float4*>(&sm.b1[128 + tx * 4]);
#pragma unroll
                for (int p = 0; p < 8; ++p) {
                    acc[p][0] = make_float2(ba.x, ba.y);
                    acc[p][1] = make_float2(ba.z, ba.w);
                    acc[p][2] = make_float2(bb.x, bb.y);
                    acc[p][3] = make_float2(bb.z, bb.w);
                }
            }
#pragma unroll 1
            for (int k = 0; k < kHeadF; k += 4) {
                float4 x4[8];
#pragma unroll
                for (int p = 0; p < 8; ++p) x4[p] = *reinterpret_cast<const float4*>(&sm.xs[ty + 8 * p][k]);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    const float4 wa = *reinterpret_cast<const float4*>(&sm.w1t[k + kk][tx * 4]);
                    const float4 wb = *reinterpret_cast<const float4*>(&sm.w1t[k + kk][128 + tx * 4]);
                    float a[8];
#pragma unroll
                    for (int p = 0; p < 8; ++p) a[p] = pick(x4[p], kk);
                    tile_fma(acc, a, wa, wb);
                }
            }
#pragma unroll
            for (int p = 0; p < 8; ++p) {                   // relu, H[pair][h]
                float* row = &sm.hs[ty + 8 * p][0];
                *reinterpret_cast<float4*>(row + tx * 4) =
                    make_float4(relu(acc[p][0].x), relu(acc[p][0].y), relu(acc[p][1].x), relu(acc[p][1].y));
                *reinterpret_cast<float4*>(row + 128 + tx * 4) =
                    make_float4(relu(acc[p][2].x), relu(acc[p][2].y), relu(acc[p][3].x), relu(acc[p][3].y));
            }
        }
        __syncthreads();
        // ---- phase 2: group g = hidden units [64g, 64g+64); thread = pairs {ty + 8p} x outputs {4tx..} U {32+4tx..}
        {
            const int g = tid >> 6, ty = (tid & 63) >> 3, tx = tid & 7;
            float2 acc[8][4];
#pragma unroll
            for (int p = 0; p < 8; ++p)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[p][j] = make_float2(0.f, 0.f);
#pragma unroll 1
            for (int k = g * (kHeadHid / 4); k < (g + 1) * (kHeadHid / 4); k += 4) {
                float4 h4[8];
#pragma unroll
                for (int p = 0; p < 8; ++p) h4[p] = *reinterpret_cast<const float4*>(&sm.hs[ty + 8 * p][k]);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    const float4 wa = *reinterpret_cast<const float4*>(&sm.w2t[k + kk][tx * 4]);
                    const float4 wb = *reinterpret_cast<const float4*>(&sm.w2t[k + kk][32 + tx * 4]);
                    float a[8];
#pragma unroll
                    for (int p = 0; p < 8; ++p) a[p] = pick(h4[p], kk);
                    tile_fma(acc, a, wa, wb);
                }
            }
            __syncthreads();                                // every group is done reading H: reuse it for the partials
            float* part = &sm.hs[0][0] + (size_t)g * (kHeadTile * kHeadF);      // [pair][out] per group
#pragma unroll
            for (int p = 0; p < 8; ++p) {
                float* row = part + (ty + 8 * p) * kHeadF;
                *reinterpret_cast<float4*>(row + tx * 4) = make_float4(acc[p][0].x, acc[p][0].y, acc[p][1].x, acc[p][1].y);
                *reinterpret_cast<float4*>(row + 32 + tx * 4) = make_float4(acc[p][2].x, acc[p][2].y, acc[p][3].x, acc[p][3].y);
            }
        }
        __syncthreads();
        // ---- sum the 4 partial tiles in a fixed order, add the bias, store: 4096 outputs, 16 per thread
        {
            const float* part = &sm.hs[0][0];
#pragma unroll
            for (int it = 0; it < 4; ++it) {
                const int i4 = it * kHeadThreads + tid;               // float4 index inside the [64][64] tile
                const int p = i4 >> 4, o = (i4 & 15) * 4;
                float4 s = *reinterpret_cast<const float4*>(part + i4 * 4);
#pragma unroll
                for (int g = 1; g < 4; ++g) {
                    const float4 v = *reinterpret_cast<const float4*>(part + g * (kHeadTile * kHeadF) + i4 * 4);
                    s.x += v.x;
                    s.y += v.y;
                    s.z += v.z;
                    s.w += v.w;
                }
                s.x += sm.b2[o];
                s.y += sm.b2[o + 1];
                s.z += sm.b2[o + 2];
                s.w += sm.b2[o + 3];
                if (p0 + p < n) *reinterpret_cast<float4*>(y + (p0 + p) * kHeadF + o) = s;
            }
        }
    }
}

}  // namespace
}  // namespace tpn

extern "C" int tpn_head_forward(const float* x_dev, int64_t n, const int32_t* n_dev, int features, int hidden, const float* w1_dev,
                                const float* b1_dev, const float* w2_dev, const float* b2_dev, float* y_dev,
                                void* stream_v) {
    using namespace tpn;
    if (n < 0 || features < 1 || hidden < 1) return TPN_ERR_INVALID_ARGUMENT;
    if (features != kHeadF || hidden != kHeadHid) return TPN_ERR_UNSUPPORTED;
    if (n == 0) return TPN_OK;
    if (x_dev == nullptr || w1_dev == nullptr || b1_dev == nullptr || w2_dev == nullptr || b2_dev == nullptr ||
        y_dev == nullptr || ((reinterpret_cast<uintptr_t>(x_dev) | reinterpret_cast<uintptr_t>(y_dev)) & 15) != 0)
        return TPN_ERR_INVALID_ARGUMENT;
    DeviceScope scope(x_dev);
    if (!(debug_flags() & TPN_DEBUG_HEAD_FFMA)) {
        const int trc = launch_head_tensor(x_dev, n, reinterpret_cast<const int*>(n_dev), w1_dev, b1_dev, w2_dev, b2_dev,
                                           y_dev, scope.slot(), reinterpret_cast<cudaStream_t>(stream_v));
        return trc != TPN_OK ? trc : check_launch();
    }
    static bool configured_tab[kMaxDevices];
    bool& configured = configured_tab[scope.slot()];
    const int smem = (int)sizeof(HeadSmem);
    if (!configured) {
        const cudaError_t e = cudaFuncSetAttribute(head_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) {
            set_cuda_error(e);
            return TPN_ERR_CUDA;
        }
        configured = true;
    }
    const int sms = device_sm_count();
    const long long ntiles = (n + kHeadTile - 1) / kHeadTile;
    const unsigned grid = (unsigned)(ntiles < sms ? ntiles : sms);
    head_forward_kernel<<<grid, kHeadThreads, smem, reinterpret_cast<cudaStream_t>(stream_v)>>>(
        x_dev, n, w1_dev, b1_dev, w2_dev, b2_dev, y_dev, reinterpret_cast<const int*>(n_dev));
    return check_launch();
}

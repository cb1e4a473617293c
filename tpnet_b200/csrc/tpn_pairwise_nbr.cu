// tpn_pairwise_nbr — the structured encoder call of the pair-wise features for sm_100a.
//
// Reference call site (models/TPNet.py:313-324): for every row n of a batch of m nodes with K
// sampled neighbours, TPNet asks for get_pair_wise_feature(nbr[n,k], src[n]) and
// get_pair_wise_feature(nbr[n,k], dst[n]) by materialising two index lists of 2mK ids
// (np.tile / np.repeat / np.concatenate), runs the generic pair encoder over 2mK pairs and then
// re-splits and concatenates the result into [m, K, 2F].  Here the structure is used directly:
//   * out[n, k, 0, :] = Gram([W; S]) and out[n, k, 1, :] = Gram([W; D]) with W = rows P_0..P_L of
//     nbr[n,k], S of src[n], D of dst[n] — written in place in the final [m, K, 2, F] layout;
//   * the W.W block is shared by both outputs, S.S / D.D by all K neighbours of the row: 42
//     unique dot products per (n, k) instead of 72 (L = 3), and 1 + 2/K node blocks read per
//     (n, k) instead of 4;
//   * one CTA per row n: S and D are fetched once into shared memory (cp.async.bulk + mbarrier),
//     each warp fetches the blocks of 4 neighbours the same way, 8 lanes per neighbour run the
//     packed-FFMA2 accumulation and the transposing butterfly of tpn_pairwise.cuh, the epilogue
//     (clamp, log(x + 1.0), TPNet.py:127-128) is applied once per unique entry and mirrored
//     through a shared-memory tile, and the warp stores its 4 x 2F outputs as coalesced 128-bit
//     streaming stores.
// Padding neighbours (id 0) are ordinary rows, as in the reference (P_0[0] is random, P_{>=1}[0]
// stays zero; the masked_fill at TPNet.py:332 is not in place and has no effect).
#include "tpn_pairwise.cuh"

namespace tpn {
namespace {

thread_local int g_dev_slot = 0;      // device of the call in progress (set by the entry point)


constexpr int kNbrMaxWarps = 5;     // K = 20 (the reference default) = 5 quads: one pass, 3 CTAs per SM
constexpr int kNbrG = 8;            // lanes per neighbour
constexpr int kNbrPPW = 4;          // neighbours per warp pass

__host__ __device__ inline size_t nbr_warp_bytes(size_t block_bytes, int F) {
    const size_t rows = kNbrPPW * block_bytes, tile = (size_t)kNbrPPW * 2 * F * sizeof(float);
    return ((rows > tile ? rows : tile) + 127) / 128 * 128;
}

template <int H>
__device__ __forceinline__ void nbr_step(float2 (&acc)[H * (H + 1) / 2 + 2 * H * H], const float4 (&w)[H],
                                         const float4 (&s)[H], const float4 (&d)[H]) {
    int e = 0;
#pragma unroll
    for (int r = 0; r < H; ++r) {
        const float2 rl = lo2(w[r]), rh = hi2(w[r]);
#pragma unroll
        for (int q = r; q < H; ++q) {
            acc[e] = __ffma2_rn(rl, lo2(w[q]), acc[e]);
            acc[e] = __ffma2_rn(rh, hi2(w[q]), acc[e]);
            ++e;
        }
    }
#pragma unroll
    for (int r = 0; r < H; ++r) {
        const float2 rl = lo2(w[r]), rh = hi2(w[r]);
#pragma unroll
        for (int q = 0; q < H; ++q) {
            acc[e] = __ffma2_rn(rl, lo2(s[q]), acc[e]);
            acc[e] = __ffma2_rn(rh, hi2(s[q]), acc[e]);
            ++e;
        }
    }
#pragma unroll
    for (int r = 0; r < H; ++r) {
        const float2 rl = lo2(w[r]), rh = hi2(w[r]);
#pragma unroll
        for (int q = 0; q < H; ++q) {
            acc[e] = __ffma2_rn(rl, lo2(d[q]), acc[e]);
            acc[e] = __ffma2_rn(rh, hi2(d[q]), acc[e]);
            ++e;
        }
    }
}

template <int LAYERS, bool LAZY>
__global__ void __launch_bounds__(kNbrMaxWarps * 32, LAYERS <= 3 ? 3 : 2)
pairwise_nbr_kernel(StateView st, const long long* __restrict__ nbr, const long long* __restrict__ src,
                    const long long* __restrict__ dst, int K, int apply_log_scale, float* __restrict__ out,
                    int ds4, uint32_t warp_bytes) {
    constexpr int G = kNbrG, PPW = kNbrPPW;
    constexpr int H = LAYERS + 1;
    constexpr int R = 2 * H;
    constexpr int F = R * R;
    constexpr int NH = H * (H + 1) / 2;        // unique entries of a symmetric H x H block
    constexpr int NX = H * H;
    constexpr int NU = NH + 2 * NX;            // W.W (upper triangle), W.S, W.D
    constexpr int NP = (NU + G - 1) / G * G;
    extern __shared__ __align__(128) unsigned char nbr_raw[];
    __shared__ __align__(8) uint64_t mbar[1 + kNbrMaxWarps];
    __shared__ unsigned short tab[NH];
    __shared__ float ssdd[2][NX];              // finished S.S and D.D blocks (after the epilogue)

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int nw = blockDim.x >> 5;
    const int sub = lane / G, gl = lane % G;
    const long long n = blockIdx.x;
    const int rs4 = (int)(st.row_stride >> 2);
    const uint32_t block_bytes = (uint32_t)(H * st.row_stride * 4);
    unsigned char* sd_base = nbr_raw;                                               // S block, then D block
    unsigned char* wbase = nbr_raw + 2 * (size_t)block_bytes + (size_t)warp * warp_bytes;

    if (threadIdx.x == 0) mbar_init(&mbar[0], 1);
    if (lane == 0) mbar_init(&mbar[1 + warp], 1);
    if (warp == 0) fill_entry_table<H>(tab, lane);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();

    auto clamp_id = [&](long long id) { return resolve_id(st, id, true); };
    const long long ids = clamp_id(src[n]), idd = clamp_id(dst[n]);
    if (threadIdx.x == 0) {
        mbar_expect_tx(&mbar[0], 2 * block_bytes);
        bulk_g2s(sd_base, st.data + ids * st.node_stride, block_bytes, &mbar[0]);
        bulk_g2s(sd_base + block_bytes, st.data + idd * st.node_stride, block_bytes, &mbar[0]);
    }

    const int nquads = (K + PPW - 1) / PPW;
    uint64_t* bar = &mbar[1 + warp];
    auto fetch_quad = [&](int q, long long& idw) {
        const int k = q * PPW + sub;
        idw = clamp_id(nbr[n * K + (k < K ? k : K - 1)]);
        if (lane == 0) mbar_expect_tx(bar, (uint32_t)min(PPW, K - q * PPW) * block_bytes);
        __syncwarp();                               // expect_tx is registered before any copy can complete
        if (gl == 0 && k < K) bulk_g2s(wbase + (size_t)sub * block_bytes, st.data + idw * st.node_stride, block_bytes, bar);
    };
    long long idw = 0;
    if (warp < nquads) fetch_quad(warp, idw);

    // S, D: bring rows current in place (lazy), then the S.S / D.D entries, shared by all neighbours
    mbar_wait(&mbar[0], 0);
    if (LAZY) {
        for (int i = threadIdx.x; i < 2 * LAYERS * rs4; i += blockDim.x) {
            const int which = i / (LAYERS * rs4);
            const int rem = i - which * (LAYERS * rs4);
            const int l = rem / rs4;                                    // layer l + 1
            const long long stamp = st.stamps[(which ? idd : ids) * LAYERS + l];
            if (stamp >= 0) {
                float4* p = reinterpret_cast<float4*>(sd_base + (size_t)which * block_bytes) + rs4 + rem;
                float4 v = *p;
                scale4(v, decay_factor(st, l, stamp));
                *p = v;
            }
        }
        __syncthreads();
    }
    for (int e = warp; e < 2 * NH; e += nw) {
        const int which = e >= NH ? 1 : 0;
        const int rq = tab[e - which * NH];
        const int r = rq >> 8, q = rq & 0xff;
        const float4* blk = reinterpret_cast<const float4*>(sd_base + (size_t)which * block_bytes);
        float sum = 0.f;
        for (int c = lane; c < ds4; c += 32) {
            const float4 x = blk[r * rs4 + c], y = blk[q * rs4 + c];
            sum = fmaf(x.x, y.x, sum);
            sum = fmaf(x.y, y.y, sum);
            sum = fmaf(x.z, y.z, sum);
            sum = fmaf(x.w, y.w, sum);
        }
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        if (lane == 0) {
            const float g = epilogue(sum, apply_log_scale);
            ssdd[which][r * H + q] = g;
            ssdd[which][q * H + r] = g;
        }
    }
    __syncthreads();

    const float4* ps = reinterpret_cast<const float4*>(sd_base);
    const float4* pd = reinterpret_cast<const float4*>(sd_base + block_bytes);
    const float4* pw = reinterpret_cast<const float4*>(wbase + (size_t)sub * block_bytes);
    float* tile = reinterpret_cast<float*>(wbase);                      // output staging aliases the row buffers
    uint32_t parity = 0;
    for (int q = warp; q < nquads; q += nw) {
        float fac[H];
        if (LAZY) {
#pragma unroll
            for (int l = 1; l < H; ++l) {
                const long long sw = st.stamps[idw * LAYERS + (l - 1)];
                fac[l] = sw >= 0 ? decay_factor(st, l - 1, sw) : 1.0f;
            }
        }
        float2 acc[NU];
#pragma unroll
        for (int i = 0; i < NU; ++i) acc[i] = make_float2(0.f, 0.f);
        mbar_wait(bar, parity);
        parity ^= 1u;
        if (q * PPW + sub < K) {
            for (int c = gl; c < ds4; c += G) {
                float4 w[H], s[H], d[H];
#pragma unroll
                for (int l = 0; l < H; ++l) {
                    w[l] = pw[l * rs4 + c];
                    s[l] = ps[l * rs4 + c];
                    d[l] = pd[l * rs4 + c];
                }
                if (LAZY) {
#pragma unroll
                    for (int l = 1; l < H; ++l) scale4(w[l], fac[l]);
                }
                nbr_step<H>(acc, w, s, d);
            }
        }
        __syncwarp();                               // every lane is done reading the neighbour buffers

        // transposing butterfly over the 8 lanes of the group: each lane ends up with NP/G finished entries
        float sred[NP];
#pragma unroll
        for (int i = 0; i < NP; ++i) sred[i] = i < NU ? acc[i].x + acc[i].y : 0.f;
        int first = 0, nlive = NP;
#pragma unroll
        for (int mask = G / 2; mask >= 1; mask >>= 1) {
            const bool upper = (gl & mask) != 0;
            halve<NP>(sred, nlive, mask, upper);
            nlive >>= 1;
            if (upper) first += nlive;
        }
        float* t0 = tile + sub * (2 * F);
        float* t1 = t0 + F;
#pragma unroll
        for (int k = 0; k < NP / G; ++k) {
            const int e = first + k;
            if (e < NU) {
                const float g = epilogue(sred[k], apply_log_scale);
                if (e < NH) {                       // W.W: both outputs, mirrored
                    const int rq = tab[e];
                    const int r = rq >> 8, c = rq & 0xff;
                    t0[r * R + c] = g;
                    t0[c * R + r] = g;
                    t1[r * R + c] = g;
                    t1[c * R + r] = g;
                } else {
                    const int x = e - NH;
                    float* t = x >= NX ? t1 : t0;   // W.S -> output 0, W.D -> output 1
                    const int y = x >= NX ? x - NX : x;
                    const int r = y / H, c = y - r * H;
                    t[r * R + H + c] = g;
                    t[(H + c) * R + r] = g;
                }
            }
        }
        for (int i = lane; i < PPW * 2 * NX; i += 32) {     // S.S / D.D corner of every output
            const int p = i / (2 * NX);
            const int rem = i - p * (2 * NX);
            const int which = rem / NX;
            const int y = rem - which * NX;
            const int r = y / H, c = y - r * H;
            tile[p * (2 * F) + which * F + (H + r) * R + H + c] = ssdd[which][y];
        }
        __syncwarp();
        const int valid = min(PPW, K - q * PPW) * (2 * F);              // multiple of 4
        float* dptr = out + ((size_t)n * K + (size_t)q * PPW) * (2 * F);
        for (int i = lane * 4; i < valid; i += 32 * 4)
            __stcs(reinterpret_cast<float4*>(dptr + i), *reinterpret_cast<const float4*>(tile + i));
        if (q + nw < nquads) {
            __syncwarp();
            fence_proxy_async_smem();               // generic accesses of the buffers before the next bulk copies
            fetch_quad(q + nw, idw);
        }
    }
}

template <int LAYERS>
int launch_nbr(const StateView& v, const long long* nbr, const long long* src, const long long* dst, long long m,
               int K, int scale, float* out, cudaStream_t s) {
    constexpr int F = 4 * (LAYERS + 1) * (LAYERS + 1);
    const size_t block_bytes = (size_t)(LAYERS + 1) * v.row_stride * 4;
    const size_t wb = nbr_warp_bytes(block_bytes, F);
    const size_t budget = (LAYERS <= 3 ? 72 : 100) * 1024;      // three (two) CTAs per SM
    if ((block_bytes & 15) != 0 || (v.node_stride & 3) != 0 || 2 * block_bytes + wb > 200 * 1024)
        return TPN_ERR_UNSUPPORTED;                 // rows too wide for the shared-memory staging
    int nw = (K + kNbrPPW - 1) / kNbrPPW;
    if (nw > kNbrMaxWarps) nw = kNbrMaxWarps;
    while (nw > 1 && 2 * block_bytes + nw * wb > budget) --nw;
    const size_t smem = 2 * block_bytes + nw * wb;
    const bool lazy = v.stamps != nullptr;
    auto kernel = lazy ? pairwise_nbr_kernel<LAYERS, true> : pairwise_nbr_kernel<LAYERS, false>;
    static bool configured_tab[kMaxDevices][2];          // per device
    bool* configured = configured_tab[g_dev_slot];
    if (!configured[lazy ? 1 : 0]) {
        const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) {
            set_cuda_error(e);
            return TPN_ERR_CUDA;
        }
        configured[lazy ? 1 : 0] = true;
    }
    kernel<<<(unsigned)m, nw * 32, smem, s>>>(v, nbr, src, dst, K, scale, out, (int)(v.row_stride / 4), (uint32_t)wb);
    return TPN_OK;
}

}  // namespace
}  // namespace tpn

extern "C" int tpn_pairwise_neighbors(const tpn_state_t* st, const int64_t* nbr_dev, const int64_t* src_dev,
                                      const int64_t* dst_dev, int64_t m, int num_neighbors, int apply_log_scale,
                                      float* out_dev, void* stream_v) {
    using namespace tpn;
    int rc = validate_state(st);
    if (rc != TPN_OK) return rc;
    if (m < 0 || m > 0x7fffffffll || num_neighbors < 0 || num_neighbors > (1 << 20)) return TPN_ERR_INVALID_ARGUMENT;
    if (m == 0 || num_neighbors == 0) return TPN_OK;
    if (nbr_dev == nullptr || src_dev == nullptr || dst_dev == nullptr || out_dev == nullptr ||
        (reinterpret_cast<uintptr_t>(out_dev) & 15) != 0)
        return TPN_ERR_INVALID_ARGUMENT;
    DeviceScope scope(st->data);
    g_dev_slot = scope.slot();
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_v);
    const StateView v = make_view(st);
    const long long* nb = reinterpret_cast<const long long*>(nbr_dev);
    const long long* sp = reinterpret_cast<const long long*>(src_dev);
    const long long* dp = reinterpret_cast<const long long*>(dst_dev);
    switch (st->num_layer) {
        case 1: rc = launch_nbr<1>(v, nb, sp, dp, m, num_neighbors, apply_log_scale, out_dev, stream); break;
        case 2: rc = launch_nbr<2>(v, nb, sp, dp, m, num_neighbors, apply_log_scale, out_dev, stream); break;
        case 3: rc = launch_nbr<3>(v, nb, sp, dp, m, num_neighbors, apply_log_scale, out_dev, stream); break;
        case 4: rc = launch_nbr<4>(v, nb, sp, dp, m, num_neighbors, apply_log_scale, out_dev, stream); break;
        default: return TPN_ERR_UNSUPPORTED;
    }
    if (rc != TPN_OK) return rc;
    return check_launch();
}

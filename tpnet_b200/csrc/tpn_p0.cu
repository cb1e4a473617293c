// P_0 from a counter-based generator (tpn_init_projection): the value of (seed, draw, node, column) depends on
// nothing else, so every placement of the rows (one GPU, any number of shards) holds the same bits.
#include "tpn_common.cuh"

namespace tpn {
namespace {

// ((x >> 11) + 0.5) * 2^-53, the add rounded to nearest (exact below 2^52): a uniform in (0, 1]
__device__ __forceinline__ double uniform53(unsigned long long x) {
    return __dmul_rn(__dadd_rn(__ull2double_rn(x >> 11), 0.5), 0x1.0p-53);
}

// Box-Muller of one pair, f64, every product rounded on its own (no FMA contraction)
__device__ __forceinline__ void box_muller(unsigned long long a, unsigned long long b, double& z0, double& z1) {
    const double r = __dsqrt_rn(__dmul_rn(-2.0, log(uniform53(a))));
    const double theta = __dmul_rn(6.283185307179586, uniform53(b));
    double s, c;
    sincos(theta, &s, &c);
    z0 = __dmul_rn(r, c);
    z1 = __dmul_rn(r, s);
}

// One thread per (local row, block of 4 columns); the block's four normals come from one Philox call.
__global__ void __launch_bounds__(256)
init_p0_kernel(float* __restrict__ data, long long rows, int blocks, int dim, long long node_stride,
               long long first_node, long long node_step, unsigned long long seed, unsigned long long draw,
               double scale) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * blocks) return;
    const long long j = i / blocks;
    const int q = (int)(i - j * blocks);
    unsigned long long x[4] = {(unsigned long long)q, (unsigned long long)(first_node + j * node_step), 0ull, 0ull};
    philox4x64_10(x, seed, draw);
    double z[4];
    box_muller(x[0], x[1], z[0], z[1]);
    box_muller(x[2], x[3], z[2], z[3]);
    const int c = 4 * q;
    float4 v;
    v.x = __double2float_rn(__dmul_rn(z[0], scale));
    v.y = c + 1 < dim ? __double2float_rn(__dmul_rn(z[1], scale)) : 0.f;      // pad columns stay zero
    v.z = c + 2 < dim ? __double2float_rn(__dmul_rn(z[2], scale)) : 0.f;
    v.w = c + 3 < dim ? __double2float_rn(__dmul_rn(z[3], scale)) : 0.f;
    st4(data + j * node_stride + c, v);
}

}  // namespace
}  // namespace tpn

extern "C" int tpn_init_projection(const tpn_state_t* st, int64_t rows, int64_t first_node, int64_t node_step,
                                   uint64_t seed, uint64_t draw, void* stream_v) {
    using namespace tpn;
    int rc = validate_state(st);
    if (rc != TPN_OK) return rc;
    if (rows < 0 || rows > st->num_nodes || node_step < 1 || first_node < 0) return TPN_ERR_INVALID_ARGUMENT;
    if (rows == 0) return TPN_OK;
    if ((rows - 1) > (INT64_MAX - first_node) / node_step) return TPN_ERR_INVALID_ARGUMENT;   // node ids fit int64
    DeviceScope scope(st->data);
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_v);
    const int blocks = (st->dim + 3) / 4;
    const long long threads = rows * blocks;
    const double scale = 1.0 / sqrt((double)st->dim);         // host f64: the same bits as Python's 1 / math.sqrt(d)
    init_p0_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(
        st->data, rows, blocks, st->dim, st->node_stride, first_node, node_step, (unsigned long long)seed,
        (unsigned long long)draw, scale);
    return check_launch();
}

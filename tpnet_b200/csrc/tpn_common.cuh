// Shared device helpers for the tpnet_b200 kernels (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "tpnet_b200.h"

namespace tpn {

// Device-side copy of tpn_state_t (passed by value as a kernel argument).
struct StateView {
    float* data;
    long long num_nodes;
    int num_layer;
    int dim;
    long long row_stride;    // floats
    long long node_stride;   // floats
    int* stamps;             // nullptr => eager
    const double* decay_log; // [cap][L] cumulative products of the per-update fp32 factors (row 0 = 1.0)
    long long epoch;         // epoch readers bring rows up to
    int* err;                // optional device int32 error flag (tpn_state_t::err_flag)
};

inline StateView make_view(const tpn_state_t* st) {
    StateView v;
    v.data = st->data;
    v.num_nodes = st->num_nodes;
    v.num_layer = st->num_layer;
    v.dim = st->dim;
    v.row_stride = st->row_stride;
    v.node_stride = st->node_stride;
    v.stamps = st->stamps;
    v.decay_log = st->decay_log;
    v.epoch = st->epoch;
    v.err = st->err_flag;
    return v;
}

// Every entry point runs on the device that OWNS its buffers, whatever the caller's current device is
// (the reference scripts only build the string 'cuda:G' and never call torch.cuda.set_device).
// Restores the caller's device on exit.  `dev` also indexes the per-device "kernel attributes set" tables.
constexpr int kMaxDevices = 64;
struct DeviceScope {
    int prev = -1, dev = -1;
    bool switched = false;
    explicit DeviceScope(const void* device_ptr);
    ~DeviceScope();
    DeviceScope(const DeviceScope&) = delete;
    DeviceScope& operator=(const DeviceScope&) = delete;
    int slot() const { return dev >= 0 && dev < kMaxDevices ? dev : 0; }
};
// SM count of the current device (cached per device; 148 on B200)
int device_sm_count();
// TPN_DEBUG_* flags (tpn_set_debug_flags)
int debug_flags();
// tpn_head_tc.cu: the head on tcgen05 tensor cores
int launch_head_tensor(const float* x, long long n, const int* n_dev, const float* w1, const float* b1, const float* w2,
                       const float* b2, float* y, int dev_slot, cudaStream_t stream);

inline int validate_state(const tpn_state_t* st) {
    if (st == nullptr || st->data == nullptr) return TPN_ERR_INVALID_ARGUMENT;
    if (st->num_layer < 1 || st->num_layer > TPN_MAX_LAYERS) return TPN_ERR_UNSUPPORTED;
    if (st->num_nodes < 1 || st->dim < 1) return TPN_ERR_INVALID_ARGUMENT;
    if (st->row_stride < st->dim || (st->row_stride & 3)) return TPN_ERR_INVALID_ARGUMENT;
    if (st->node_stride < (long long)(st->num_layer + 1) * st->row_stride || (st->node_stride & 3))
        return TPN_ERR_INVALID_ARGUMENT;
    if ((reinterpret_cast<uintptr_t>(st->data) & 15) != 0) return TPN_ERR_INVALID_ARGUMENT;
    if (st->stamps != nullptr && (st->decay_log == nullptr || st->log_capacity < 2 || st->epoch < 0 ||
                                  st->epoch >= st->log_capacity))
        return TPN_ERR_INVALID_ARGUMENT;
    return TPN_OK;
}

void set_cuda_error(cudaError_t e);
int check_launch();

// Device-resident node id -> row.  Indexing calls (pair-wise, gather: TPNet.py:109 indexes tensors, where
// negative ids wrap) pass wrap = true.  An id outside the range is the reference's IndexError: it cannot be
// raised from a kernel, so the flag is set (RandomProjectionModule.check_errors raises) and the id is
// clamped only to keep the access in bounds.
__device__ __forceinline__ long long resolve_id(const StateView& st, long long id, bool wrap) {
    if (wrap && id < 0) id += st.num_nodes;
    if (id < 0 || id >= st.num_nodes) {
        if (st.err != nullptr) *st.err = 1;
        id = id < 0 ? 0 : st.num_nodes - 1;
    }
    return id;
}

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, const float4& v) { *reinterpret_cast<float4*>(p) = v; }

// ReLU of the heads (torch.nn.ReLU): max(v, 0) for every number, NaN stays NaN (fmaxf would turn it into 0).
__device__ __forceinline__ float relu(float v) { return v <= 0.f ? 0.f : v; }

__device__ __forceinline__ void scale4(float4& v, float f) {
    v.x = __fmul_rn(v.x, f);
    v.y = __fmul_rn(v.y, f);
    v.z = __fmul_rn(v.z, f);
    v.w = __fmul_rn(v.w, f);
}

// acc += fl32(x * w): product rounded BEFORE the add (no FMA contraction), as the
// reference materialises `P[idx] * time_weight` before scatter_add_ (TPNet.py:91-96).
__device__ __forceinline__ void axpy4_rn(float4& acc, const float4& x, float w) {
    acc.x = __fadd_rn(acc.x, __fmul_rn(x.x, w));
    acc.y = __fadd_rn(acc.y, __fmul_rn(x.y, w));
    acc.z = __fadd_rn(acc.z, __fmul_rn(x.z, w));
    acc.w = __fadd_rn(acc.w, __fmul_rn(x.w, w));
}

// Lazy decay (TPNet.py:83-85 deferred).  The reference multiplies every row of layer l by the
// fp32 scalar c_l at EVERY update.  Row e of the log holds, per layer, the f64 product
// Q_l[e] = c_l(1) * c_l(2) * ... * c_l(e) of the fp32 factors logged so far (Q[0] = 1), so a row
// last written at epoch `from` is brought to epoch `to` by ONE multiply with
// f32(Q[to] / Q[from]): the product of exactly the factors the reference applied, rounded once
// instead of once per update (|relative difference| <= (to - from + 1) * 2^-24, and exactly
// equal when to - from <= 1).  from == to gives exactly 1.0f.
__device__ __forceinline__ float decay_factor(const double* __restrict__ log, int L, int li, long long from,
                                              long long to) {
    if (from == to) return 1.0f;            // also keeps a zero product (f32 factor underflow) harmless
    return (float)(__ldg(log + to * L + li) / __ldg(log + from * L + li));
}
__device__ __forceinline__ float decay_factor(const StateView& st, int li, long long from) {
    return decay_factor(st.decay_log, st.num_layer, li, from, st.epoch);
}

// Two columns per lane: acc += fl32(x * w) per column.  The product is one packed FMUL2, the adds
// are SCALAR on purpose: ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 even with explicit
// .rn modifiers and --fmad=false (seen in SASS, CUDA 12.9), which would skip the rounding of the
// product that the reference performs (TPNet.py:91-96).  Scalar add.rn.f32 is never contracted.
__device__ __forceinline__ float2 mul2_rn(const float2& a, float b) { return __fmul2_rn(a, make_float2(b, b)); }
__device__ __forceinline__ void axpy2_rn(float2& acc, const float2& x, float w) {
    const float2 p = __fmul2_rn(x, make_float2(w, w));
    acc.x = __fadd_rn(acc.x, p.x);
    acc.y = __fadd_rn(acc.y, p.y);
}

// ---------------------------------------------------------------- mbarrier / bulk-copy (TMA) wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// one non-blocking test of a phase (acquire): true = complete
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// orders prior generic-proxy accesses of shared memory before later async-proxy (bulk copy) writes
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}


// ---------------------------------------------------------------- cp.async (LDGSTS) wrappers
__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src_gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async4(void* dst_smem, const void* src_gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() {      // at most N committed groups of this thread still in flight
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
// the mbarrier receives one arrival (pre-counted in its init count) once every cp.async this
// thread issued so far has landed
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint64_t* bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

}  // namespace tpn

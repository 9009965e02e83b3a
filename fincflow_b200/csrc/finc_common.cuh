// finc_common.cuh -- shared device helpers for the sm_100a FInC kernels.
//
// Data model (see include/fincflow_b200.h): fp32 NCHW [B, G*C, H, W]; tile (n, g) is the
// contiguous block of C*H*W floats at ((n*G + g) * C*H*W).  Because a tile is contiguous
// it is moved global<->shared with 1-D TMA bulk copies (cp.async.bulk, SASS UBLKCP)
// completing on an mbarrier -- no tensor map needed.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/fincflow_b200.h"

namespace finc {

struct Shape {
    int B, G, C, H, W, kH, kW;
    unsigned orders;
};

__host__ __device__ __forceinline__ int order_of(unsigned orders, int g) { return (orders >> (2 * g)) & 3; }
// tap (a,b) reads x[h + row_off(a)][w + col_off(b)]   (reference: layers/conv.py:41-55)
__host__ __device__ __forceinline__ int row_off(int order, int a, int kH) { return (order & 2) ? a : a - (kH - 1); }
__host__ __device__ __forceinline__ int col_off(int order, int b, int kW) { return (order & 1) ? b : b - (kW - 1); }
__host__ __device__ __forceinline__ int corner_a(int order, int kH) { return (order & 2) ? 0 : kH - 1; }
__host__ __device__ __forceinline__ int corner_b(int order, int kW) { return (order & 1) ? 0 : kW - 1; }

// ---------------------------------------------------------------------------------------
// PTX wrappers: mbarrier + 1-D bulk async copies (TMA engine, no descriptor).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// generic-proxy accesses to shared memory -> visible to / ordered before the async proxy (TMA)
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// try_wait suspends the thread in hardware for a bounded time; the spin bound turns a
// protocol bug into a trap (launch error) instead of a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    for (uint32_t spins = 0; !mbar_try_wait(bar, parity); ++spins) {
        if (spins > (1u << 24)) __trap();
    }
}
// global -> shared bulk copy; bytes % 16 == 0, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
// shared -> global bulk copy (bulk async-group completion)
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem),
                 "r"(smem_u32(src_smem)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until all committed bulk stores have finished READING their shared-memory source
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }


// Cooperative gather of `n` contiguous weights starting at `src` with all loads of a batch in
// flight before the first scatter: f(e, value) places element e.  (The dependent
// load -> index math -> store loop costs one global round trip per iteration.)
template <typename F>
__device__ __forceinline__ void stage_weights(const float* __restrict__ src, int n, F&& f) {
    const int tid = threadIdx.x, nthr = blockDim.x;
    if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
        const int n4 = n >> 2;
        const float4* src4 = reinterpret_cast<const float4*>(src);
        for (int base = 0; base < n4; base += 4 * nthr) {
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e4 = base + u * nthr + tid;
                if (e4 < n4) v[u] = __ldg(src4 + e4);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e4 = base + u * nthr + tid;
                if (e4 < n4) { f(4 * e4, v[u].x); f(4 * e4 + 1, v[u].y); f(4 * e4 + 2, v[u].z); f(4 * e4 + 3, v[u].w); }
            }
        }
        for (int e = (n4 << 2) + tid; e < n; e += nthr) f(e, __ldg(src + e));
    } else {
        for (int base = 0; base < n; base += 8 * nthr) {
            float v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int e = base + u * nthr + tid;
                if (e < n) v[u] = __ldg(src + e);
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int e = base + u * nthr + tid;
                if (e < n) f(e, v[u]);
            }
        }
    }
}

// ---- debug timestamps (FINC_DEBUG_TS=1): per-CTA %globaltimer marks, read back with
// finc_debug_timestamps(); never enabled in normal operation --------------------------------
constexpr int kDbgSlots = 8;
constexpr int kDbgCtas = 1024;
__device__ __forceinline__ void dbg_mark(unsigned long long* buf, int slot) {
    if (buf) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
        const int cta = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
        if (cta < kDbgCtas) buf[cta * kDbgSlots + slot] = t;
    }
}
unsigned long long* debug_ts_buffer();  // device pointer, or nullptr when disabled

// Programmatic dependent launch (PDL): a kernel launched with the attribute may start while
// its stream predecessor is still draining.  pdl_wait() blocks until the predecessor has
// completed and its memory is visible -- it must precede the first global access; everything
// before it (barrier init, index math) overlaps the predecessor's tail.  pdl_trigger() lets the
// successor start launching.  Both are no-ops for ordinary launches.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

int pdl_enabled();  // FINC_PDL=0 disables (default on)

// kernel launch with the PDL attribute (plain launch when disabled)
template <typename Kern, typename Args>
inline int launch_kernel(Kern kern, dim3 grid, int threads, size_t smem, cudaStream_t st, const Args& a) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = dim3((unsigned)threads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return (int)cudaLaunchKernelEx(&cfg, kern, a);
}

__device__ __forceinline__ bool is_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---------------------------------------------------------------------------------------
// host-side launch helpers (defined in finc_api.cu)
// ---------------------------------------------------------------------------------------
int sm_count_cached();
size_t max_optin_smem_cached();

// launchers implemented by the per-kernel translation units; all return cudaError_t as int
int launch_conv_fast(const float* x, const float* w, float* y, float* logdet, bool logdet_acc, const Shape& s,
                     bool transpose, bool prepared, int sm_div, cudaStream_t st, bool* handled);
size_t conv_prepared_floats(const Shape& s);
int launch_conv_prepare(const float* w, float* out, int n_units, size_t w_stride, size_t out_stride, const Shape& s,
                        bool transpose, cudaStream_t st);
int launch_inverse_fast(const float* z, const float* w, float* x, const Shape& s, cudaStream_t st, bool* handled);
int launch_inverse_wave(const float* z, const float* w, float* x, const Shape& s, bool prepared, cudaStream_t st,
                        bool* handled);
int launch_inverse_rw(const float* z, const float* w, float* x, const Shape& s, bool prepared, cudaStream_t st,
                      bool* handled);
int launch_inverse_rw_adjoint(const float* dx, const float* w, float* dz, const Shape& s, cudaStream_t st,
                              bool* handled);
int launch_inverse_rw_chain(const float* z, const float* w, float* x, const Shape& s, bool prepared, int n_units,
                            int u_first, int u_step, long unit_stride, cudaStream_t st, bool* handled);
// one level of launch_inverse_rw_multi: the arguments of launch_inverse_rw_chain (prepared tables)
struct RwChainLevel {
    const float* z;
    const float* w;
    float* x;
    Shape s;
    int n_units, u_first, u_step;
    long unit_stride;
};
constexpr int kInverseMultiMaxLevels = 4;
int launch_inverse_rw_multi(const RwChainLevel* levels, int n, cudaStream_t st);
bool rw_shape_supported(const Shape& s);
size_t wave_prepared_floats(const Shape& s);
int launch_wave_prepare(const float* w, float* out, int n_units, size_t w_stride, size_t out_stride, const Shape& s,
                        cudaStream_t st);
constexpr int kPrepHeaderFloats = 32;  // 128-byte header in front of a prepared table
int launch_wgrad_fast(const float* dz, const float* x, float* dw, float* workspace, size_t ws_floats, const Shape& s,
                      unsigned flags, cudaStream_t st, bool* handled);
size_t wgrad_workspace_floats(const Shape& s);
size_t wgrad_batched_workspace_floats(const Shape& s, int n_units);
int launch_wgrad_batched(const float* dz, const float* x, float* dw, float* workspace, size_t ws_floats, const Shape& s,
                         unsigned flags, int n_units, long dz_ustride, long x_ustride, long dw_ustride,
                         cudaStream_t st, bool* handled);

int launch_conv_naive(const float* x, const float* w, float* y, const Shape& s, bool transpose, cudaStream_t st);
int launch_inverse_naive(const float* z, const float* w, float* x, const Shape& s, cudaStream_t st);
int launch_inverse_adjoint_naive(const float* dx, const float* w, float* dz, const Shape& s, cudaStream_t st);
int launch_wgrad_naive(const float* dz, const float* x, float* dw, const Shape& s, unsigned flags, cudaStream_t st);
int launch_mask(float* dw, const Shape& s, cudaStream_t st);
int launch_logdet(const float* w, float* logdet, bool accumulate, const Shape& s, cudaStream_t st);
int launch_squeeze(const float* x, float* y, int B, int C, int H, int W, bool inverse, cudaStream_t st);
int launch_affine1x1(const float* x, const float* A, const float* bias, float* y, int B, int C, long HW, cudaStream_t st);
size_t affine1x1_wgrad_workspace_floats(int B, int C, long HW);
int launch_affine1x1_wgrad(const float* dy, const float* x, float* dA, float* db, float* workspace, size_t ws_floats,
                           int B, int C, long HW, cudaStream_t st);
int launch_slogdet_inverse(const float* W, float* logabsdet, float* Winv, int n, int C, cudaStream_t st);
int launch_preprocess(const float* x, const float* u, float* y, float* logdet, int B, long D, float alpha, int reverse,
                      cudaStream_t st);
int launch_adam(float* p, const float* g, float* m, float* v, float* step, float lr, float b1, float b2, float eps,
                long n, cudaStream_t st);
int launch_allreduce_adam(const void* peer_grad, const void* peer_signal, void* local, float* param, float* m, float* v,
                          float* step, float lr, float b1, float b2, float eps, float grad_scale, long n, int rank,
                          int world, cudaStream_t st);
int launch_gaussian_logp(const float* z, const float* logdet, float* logp, float* dz, float dz_scale, int B, long D,
                         cudaStream_t st);

}  // namespace finc

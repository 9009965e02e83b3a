// finc_api.cu -- extern "C" entry points declared in include/fincflow_b200.h.
//
// Argument checking + dispatch: tiled sm_100a kernels when the shape is covered, generic
// GPU kernels otherwise.  There is no CPU path.
#include "finc_common.cuh"

#include <cstdlib>

namespace finc {

__device__ unsigned long long g_finc_dbg[kDbgCtas * kDbgSlots];

unsigned long long* debug_ts_buffer() {
    static int enabled = -1;
    if (enabled < 0) {
        const char* e = getenv("FINC_DEBUG_TS");
        enabled = (e && e[0] == '1') ? 1 : 0;
    }
    if (!enabled) return nullptr;
    void* p = nullptr;
    if (cudaGetSymbolAddress(&p, g_finc_dbg) != cudaSuccess) return nullptr;
    return static_cast<unsigned long long*>(p);
}

int pdl_enabled() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("FINC_PDL");
        v = (e && e[0] == '0') ? 0 : 1;
    }
    return v;
}

static int g_sm_count[64];
static size_t g_smem_optin[64];

static int current_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    return dev < 0 || dev >= 64 ? 0 : dev;
}

int sm_count_cached() {
    const int dev = current_device();
    if (g_sm_count[dev] == 0) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
        g_sm_count[dev] = v;
    }
    return g_sm_count[dev];
}

size_t max_optin_smem_cached() {
    const int dev = current_device();
    if (g_smem_optin[dev] == 0) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess || v <= 0)
            v = 48 * 1024;
        g_smem_optin[dev] = (size_t)v;
    }
    return g_smem_optin[dev];
}

static bool shape_ok(int B, int G, int C, int H, int W, int kH, int kW) {
    return B >= 0 && G >= 1 && G <= 16 && C >= 1 && H >= 1 && W >= 1 && kH >= 1 && kW >= 1 &&
           (long)G * C <= (1L << 20) && (long)H * W <= (1L << 28);
}

static Shape mk(int B, int G, int C, int H, int W, int kH, int kW, unsigned orders) {
    Shape s;
    s.B = B; s.G = G; s.C = C; s.H = H; s.W = W; s.kH = kH; s.kW = kW; s.orders = orders;
    return s;
}

}  // namespace finc

using namespace finc;

extern "C" {

int finc_abi_version(void) { return FINC_ABI_VERSION; }

const char* finc_error_string(int code) {
    switch (code) {
        case FINC_OK: return "ok";
        case FINC_E_BADARG: return "finc: bad argument (null pointer, non-positive dimension or G > 16)";
        case FINC_E_WORKSPACE: return "finc: workspace too small (see finc_backward_weight_workspace_bytes)";
        case FINC_E_UNSUPPORTED: return "finc: unsupported configuration";
        default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "finc: unknown error";
    }
}

int finc_set_device(int device) { return (int)cudaSetDevice(device); }

int finc_sm_count(void) {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return -1;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
    return v;
}

int finc_forward_f32(const float* x, const float* w, float* z, float* logdet, int B, int G, int C, int H, int W,
                     int kH, int kW, unsigned orders, unsigned flags, void* stream) {
    if (!shape_ok(B, G, C, H, W, kH, kW) || !w) return FINC_E_BADARG;
    if (B == 0) return FINC_OK;
    if (!x || !z || x == z) return FINC_E_BADARG;
    const Shape s = mk(B, G, C, H, W, kH, kW, orders);
    cudaStream_t st = (cudaStream_t)stream;
    int rc = 0;
    bool handled = false;
    const bool prep = (flags & FINC_FLAG_PREPARED) != 0;
    if (prep && (flags & FINC_FLAG_NAIVE)) return FINC_E_BADARG;
    if (!(flags & FINC_FLAG_NAIVE)) rc = launch_conv_fast(x, w, z, logdet, (flags & FINC_FLAG_LOGDET_ACCUMULATE) != 0, s, false, prep, (flags & FINC_FLAG_HALF_GPU) ? 2 : 1, st, &handled);
    if (rc) return rc;
    if (handled) return FINC_OK;  // logdet was written by the fused epilogue
    if (prep) return FINC_E_UNSUPPORTED;  // the generic kernels need the raw weights
    rc = launch_conv_naive(x, w, z, s, false, st);
    if (rc) return rc;
    if (logdet) rc = launch_logdet(w, logdet, (flags & FINC_FLAG_LOGDET_ACCUMULATE) != 0, s, st);
    return rc;
}

int finc_backward_input_f32(const float* dz, const float* w, float* dx, int B, int G, int C, int H, int W, int kH,
                            int kW, unsigned orders, unsigned flags, void* stream) {
    if (!shape_ok(B, G, C, H, W, kH, kW) || !w) return FINC_E_BADARG;
    if (B == 0) return FINC_OK;
    if (!dz || !dx || dz == dx) return FINC_E_BADARG;
    const Shape s = mk(B, G, C, H, W, kH, kW, orders);
    cudaStream_t st = (cudaStream_t)stream;
    int rc = 0;
    bool handled = false;
    const bool prep = (flags & FINC_FLAG_PREPARED) != 0;
    if (prep && (flags & FINC_FLAG_NAIVE)) return FINC_E_BADARG;
    if (!(flags & FINC_FLAG_NAIVE)) rc = launch_conv_fast(dz, w, dx, nullptr, false, s, true, prep, (flags & FINC_FLAG_HALF_GPU) ? 2 : 1, st, &handled);
    if (rc) return rc;
    if (prep && !handled) return FINC_E_UNSUPPORTED;
    if (!handled) rc = launch_conv_naive(dz, w, dx, s, true, st);
    return rc;
}

size_t finc_backward_weight_workspace_bytes(int B, int G, int C, int H, int W, int kH, int kW) {
    if (!shape_ok(B, G, C, H, W, kH, kW)) return 0;
    return wgrad_workspace_floats(mk(B, G, C, H, W, kH, kW, 0)) * sizeof(float);
}

int finc_backward_weight_f32(const float* dz, const float* x, float* dw, void* workspace, size_t workspace_bytes,
                             int B, int G, int C, int H, int W, int kH, int kW, unsigned orders, unsigned flags,
                             void* stream) {
    if (!shape_ok(B, G, C, H, W, kH, kW) || !dw) return FINC_E_BADARG;
    const Shape s = mk(B, G, C, H, W, kH, kW, orders);
    cudaStream_t st = (cudaStream_t)stream;
    if (B > 0 && (!dz || !x)) return FINC_E_BADARG;
    int rc = 0;
    bool handled = false;
    if (!(flags & FINC_FLAG_NAIVE) && B > 0) {
        if (!workspace) return FINC_E_WORKSPACE;
        rc = launch_wgrad_fast(dz, x, dw, (float*)workspace, workspace_bytes / sizeof(float), s, flags, st, &handled);
        if (rc) return rc;
    }
    if (!handled) rc = launch_wgrad_naive(dz, x, dw, s, flags, st);  // B == 0 writes zeros
    return rc;
}

size_t finc_backward_weight_batched_workspace_bytes(int B, int G, int C, int H, int W, int kH, int kW, int n_units) {
    if (!shape_ok(B, G, C, H, W, kH, kW) || n_units < 1) return 0;
    return wgrad_batched_workspace_floats(mk(B, G, C, H, W, kH, kW, 0), n_units) * (size_t)n_units * sizeof(float);
}

int finc_backward_weight_batched_f32(const float* dz, const float* x, float* dw, void* workspace, size_t workspace_bytes,
                                     int B, int G, int C, int H, int W, int kH, int kW, unsigned orders, unsigned flags,
                                     int n_units, long dz_unit_stride, long x_unit_stride, long dw_unit_stride,
                                     void* stream) {
    if (!shape_ok(B, G, C, H, W, kH, kW) || !dw || !dz || !x || n_units < 1 || B < 1) return FINC_E_BADARG;
    if (!workspace) return FINC_E_WORKSPACE;
    const Shape s = mk(B, G, C, H, W, kH, kW, orders);
    bool handled = false;
    const int rc = launch_wgrad_batched(dz, x, dw, (float*)workspace, workspace_bytes / sizeof(float), s, flags, n_units,
                                        dz_unit_stride, x_unit_stride, dw_unit_stride, (cudaStream_t)stream, &handled);
    if (rc) return rc;
    return handled ? FINC_OK : FINC_E_UNSUPPORTED;
}

int finc_inverse_f32(const float* z, const float* w, float* x, int B, int G, int C, int H, int W, int kH, int kW,
                     unsigned orders, unsigned flags, void* stream) {
    if (!shape_ok(B, G, C, H, W, kH, kW) || !w) return FINC_E_BADARG;
    if (B == 0) return FINC_OK;
    if (!z || !x) return FINC_E_BADARG;
    const Shape s = mk(B, G, C, H, W, kH, kW, orders);
    cudaStream_t st = (cudaStream_t)stream;
    int rc = 0;
    bool handled = false;
    if (!(flags & FINC_FLAG_NAIVE)) {
        const bool prep = (flags & FINC_FLAG_PREPARED) != 0;
        if (!(flags & (FINC_FLAG_GENERIC_TILED | FINC_FLAG_WAVE_SMEM))) rc = launch_inverse_rw(z, w, x, s, prep, st, &handled);
        if (rc) return rc;
        if (!handled && !(flags & FINC_FLAG_GENERIC_TILED)) rc = launch_inverse_wave(z, w, x, s, prep, st, &handled);
        if (rc) return rc;
        if (prep && !handled) return FINC_E_UNSUPPORTED;
        if (!handled) rc = launch_inverse_fast(z, w, x, s, st, &handled);
    }
    if (rc) return rc;
    if (!handled) rc = launch_inverse_naive(z, w, x, s, st);
    return rc;
}

int finc_inverse_adjoint_f32(const float* dx, const float* w, float* dz, int B, int G, int C, int H, int W, int kH,
                             int kW, unsigned orders, unsigned flags, void* stream) {
    if (!shape_ok(B, G, C, H, W, kH, kW) || !w) return FINC_E_BADARG;
    if (flags & FINC_FLAG_PREPARED) return FINC_E_UNSUPPORTED;
    if (B == 0) return FINC_OK;
    if (!dx || !dz) return FINC_E_BADARG;
    // A^T is the inverse swept from the opposite corner: flip both order bits of every group
    const unsigned flip = G >= 16 ? 0xFFFFFFFFu : (1u << (2 * G)) - 1u;
    const Shape s = mk(B, G, C, H, W, kH, kW, orders ^ flip);
    cudaStream_t st = (cudaStream_t)stream;
    int rc = 0;
    bool handled = false;
    if (!(flags & FINC_FLAG_NAIVE)) rc = launch_inverse_rw_adjoint(dx, w, dz, s, st, &handled);
    if (rc) return rc;
    if (!handled) rc = launch_inverse_adjoint_naive(dx, w, dz, s, st);
    return rc;
}

int finc_inverse_chain_f32(const float* z, const void* prepared, size_t prepared_stride_bytes, float* x, int B, int G,
                           int C, int H, int W, int kH, int kW, unsigned orders, int n_units, int u_first, int u_step,
                           void* stream) {
    if (!shape_ok(B, G, C, H, W, kH, kW) || !prepared || n_units < 1 || prepared_stride_bytes % 16 != 0) return FINC_E_BADARG;
    if (B == 0) return FINC_OK;
    if (!z || !x) return FINC_E_BADARG;
    const Shape s = mk(B, G, C, H, W, kH, kW, orders);
    bool handled = false;
    const int rc = launch_inverse_rw_chain(z, (const float*)prepared, x, s, true, n_units, u_first, u_step,
                                           (long)(prepared_stride_bytes / 4), (cudaStream_t)stream, &handled);
    if (rc) return rc;
    return handled ? FINC_OK : FINC_E_UNSUPPORTED;
}

int finc_inverse_chain_multi_f32(const FincInverseLevel* levels, int n_levels, void* stream) {
    if (!levels || n_levels < 1) return FINC_E_BADARG;
    if (n_levels > kInverseMultiMaxLevels) return FINC_E_UNSUPPORTED;
    RwChainLevel lv[kInverseMultiMaxLevels];
    for (int i = 0; i < n_levels; ++i) {
        const FincInverseLevel& l = levels[i];
        if (!shape_ok(l.B, l.G, l.C, l.H, l.W, l.kH, l.kW) || !l.prepared || l.n_units < 1 ||
            l.prepared_stride_bytes % 16 != 0)
            return FINC_E_BADARG;
        if (l.B > 0 && (!l.z || !l.x)) return FINC_E_BADARG;
        lv[i] = RwChainLevel{l.z, (const float*)l.prepared, l.x, mk(l.B, l.G, l.C, l.H, l.W, l.kH, l.kW, l.orders),
                             l.n_units, l.u_first, l.u_step, (long)(l.prepared_stride_bytes / 4)};
    }
    return launch_inverse_rw_multi(lv, n_levels, (cudaStream_t)stream);
}

int finc_apply_grad_mask_f32(float* dw, int G, int C, int kH, int kW, unsigned orders, void* stream) {
    if (!shape_ok(1, G, C, 1, 1, kH, kW) || !dw) return FINC_E_BADARG;
    return launch_mask(dw, mk(1, G, C, 1, 1, kH, kW, orders), (cudaStream_t)stream);
}

int finc_logdet_f32(const float* w, float* logdet, int B, int G, int C, int H, int W, int kH, int kW,
                    unsigned orders, void* stream) {
    if (!shape_ok(B, G, C, H, W, kH, kW) || !w) return FINC_E_BADARG;
    if (B == 0) return FINC_OK;
    if (!logdet) return FINC_E_BADARG;
    return launch_logdet(w, logdet, false, mk(B, G, C, H, W, kH, kW, orders), (cudaStream_t)stream);
}

int finc_gaussian_logp_f32(const float* z, const float* logdet, float* logp, float* dz, float dz_scale, int B,
                           long D, void* stream) {
    if (B < 0 || D < 1) return FINC_E_BADARG;
    if (B == 0) return FINC_OK;
    if (!z || !logp) return FINC_E_BADARG;
    return launch_gaussian_logp(z, logdet, logp, dz, dz_scale, B, D, (cudaStream_t)stream);
}

int finc_adam_step_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, float* step, float lr,
                       float beta1, float beta2, float eps, long n, void* stream) {
    if (n < 0 || (n > 0 && (!param || !grad || !exp_avg || !exp_avg_sq || !step))) return FINC_E_BADARG;
    if (n == 0) return FINC_OK;
    return launch_adam(param, grad, exp_avg, exp_avg_sq, step, lr, beta1, beta2, eps, n, (cudaStream_t)stream);
}

int finc_allreduce_adam_f32(const void* peer_grad, const void* peer_signal, void* local, float* param, float* exp_avg,
                            float* exp_avg_sq, float* step, float lr, float beta1, float beta2, float eps,
                            float grad_scale, long n, int rank, int world, void* stream) {
    if (!peer_grad || !peer_signal || !local || !param || !exp_avg || !exp_avg_sq || !step || n < 1 || rank < 0 ||
        rank >= world)
        return FINC_E_BADARG;
    return launch_allreduce_adam(peer_grad, peer_signal, local, param, exp_avg, exp_avg_sq, step, lr, beta1, beta2, eps,
                                 grad_scale, n, rank, world, (cudaStream_t)stream);
}

int finc_squeeze_f32(const float* x, float* y, int B, int C, int H, int W, void* stream) {
    if (B < 0 || C < 1 || H < 2 || W < 2 || (H & 1) || (W & 1)) return FINC_E_BADARG;
    if (B == 0) return FINC_OK;
    if (!x || !y || x == y || (reinterpret_cast<uintptr_t>(x) & 7)) return FINC_E_BADARG;
    return launch_squeeze(x, y, B, C, H, W, false, (cudaStream_t)stream);
}

int finc_unsqueeze_f32(const float* x, float* y, int B, int C4, int H, int W, void* stream) {
    if (B < 0 || C4 < 4 || (C4 & 3) || H < 1 || W < 1) return FINC_E_BADARG;
    if (B == 0) return FINC_OK;
    if (!x || !y || x == y || (reinterpret_cast<uintptr_t>(y) & 7)) return FINC_E_BADARG;
    return launch_squeeze(x, y, B, C4 / 4, 2 * H, 2 * W, true, (cudaStream_t)stream);
}

int finc_affine1x1_f32(const float* x, const float* A, const float* bias, float* y, int B, int C, long HW, void* stream) {
    if (B < 0 || C < 1 || C > 4096 || HW < 1) return FINC_E_BADARG;
    if (B == 0) return FINC_OK;
    if (!x || !A || !y || x == y) return FINC_E_BADARG;
    return launch_affine1x1(x, A, bias, y, B, C, HW, (cudaStream_t)stream);
}

int finc_slogdet_inverse_f32(const float* W, float* logabsdet, float* Winv, int n, int C, void* stream) {
    if (n < 0 || C < 1 || C > 128) return FINC_E_BADARG;
    if (n == 0) return FINC_OK;
    if (!W || !logabsdet || !Winv) return FINC_E_BADARG;
    return launch_slogdet_inverse(W, logabsdet, Winv, n, C, (cudaStream_t)stream);
}

int finc_preprocess_f32(const float* x, const float* noise, float* y, float* logdet, int B, long D, float alpha,
                        int reverse, void* stream) {
    if (B < 0 || D < 1 || !(alpha >= 0.f && alpha < 0.5f)) return FINC_E_BADARG;
    if (B == 0) return FINC_OK;
    if (!x || !y) return FINC_E_BADARG;
    return launch_preprocess(x, noise, y, logdet, B, D, alpha, reverse, (cudaStream_t)stream);
}

size_t finc_affine1x1_backward_weight_workspace_bytes(int B, int C, long HW) {
    if (B < 0 || C < 1 || C > 4096 || HW < 1) return 0;
    return affine1x1_wgrad_workspace_floats(B, C, HW) * sizeof(float);
}

int finc_affine1x1_backward_weight_f32(const float* dy, const float* x, float* dA, float* dbias, void* workspace,
                                       size_t workspace_bytes, int B, int C, long HW, void* stream) {
    if (B < 0 || C < 1 || C > 4096 || HW < 1 || !dA) return FINC_E_BADARG;
    if (B > 0 && (!dy || !x)) return FINC_E_BADARG;
    if (B > 0 && !workspace) return FINC_E_WORKSPACE;
    if (B == 0) {
        cudaError_t e = cudaMemsetAsync(dA, 0, (size_t)C * C * sizeof(float), (cudaStream_t)stream);
        if (e == cudaSuccess && dbias) e = cudaMemsetAsync(dbias, 0, (size_t)C * sizeof(float), (cudaStream_t)stream);
        return (int)e;
    }
    return launch_affine1x1_wgrad(dy, x, dA, dbias, static_cast<float*>(workspace), workspace_bytes / sizeof(float), B, C, HW,
                                  (cudaStream_t)stream);
}

size_t finc_prepared_weights_bytes(int kind, int B, int G, int C, int H, int W, int kH, int kW) {
    if (!shape_ok(B, G, C, H, W, kH, kW) || B < 1) return 0;
    const Shape s = mk(B, G, C, H, W, kH, kW, 0);
    size_t f = 0;
    if (kind == FINC_PREP_FORWARD || kind == FINC_PREP_BACKWARD_INPUT) f = conv_prepared_floats(s);
    else if (kind == FINC_PREP_INVERSE) f = wave_prepared_floats(s);
    return ((f * sizeof(float) + 127) / 128) * 128;
}

int finc_prepare_weights_f32(const float* w, void* prepared, int kind, int n_units, size_t w_stride_floats,
                             size_t prepared_stride_bytes, int B, int G, int C, int H, int W, int kH, int kW,
                             unsigned orders, void* stream) {
    if (!shape_ok(B, G, C, H, W, kH, kW) || !w || !prepared || n_units < 1 || prepared_stride_bytes % 16 != 0 ||
        (reinterpret_cast<uintptr_t>(prepared) & 15) != 0)
        return FINC_E_BADARG;
    const Shape s = mk(B, G, C, H, W, kH, kW, orders);
    float* out = static_cast<float*>(prepared);
    const size_t ostride = prepared_stride_bytes / sizeof(float);
    if (kind == FINC_PREP_FORWARD) return launch_conv_prepare(w, out, n_units, w_stride_floats, ostride, s, false, (cudaStream_t)stream);
    if (kind == FINC_PREP_BACKWARD_INPUT) return launch_conv_prepare(w, out, n_units, w_stride_floats, ostride, s, true, (cudaStream_t)stream);
    if (kind == FINC_PREP_INVERSE) return launch_wave_prepare(w, out, n_units, w_stride_floats, ostride, s, (cudaStream_t)stream);
    return FINC_E_BADARG;
}

/* debug only (FINC_DEBUG_TS=1): copy the per-CTA timestamp marks of the last launch (synchronises) */
int finc_debug_timestamps(unsigned long long* host_out, int n) {
    if (!host_out || n <= 0) return FINC_E_BADARG;
    if (n > kDbgCtas * kDbgSlots) n = kDbgCtas * kDbgSlots;
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return (int)e;
    e = cudaMemcpyFromSymbol(host_out, g_finc_dbg, sizeof(unsigned long long) * n);
    if (e != cudaSuccess) return (int)e;
    void* p = nullptr;
    if (cudaGetSymbolAddress(&p, g_finc_dbg) == cudaSuccess) cudaMemset(p, 0, sizeof(g_finc_dbg));  // fresh marks next time
    return 0;
}

}  // extern "C"

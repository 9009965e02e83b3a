// tc_api.cu -- host side of the tensor-core path: TMA tensor maps, weight preparation (hi / lo
// TF32 split), im2col for the small-channel first convolution, and the extern "C" entry points
// finc_tc_conv_* / finc_coupling_* declared in include/fincflow_b200.h.
//
// Reference layer: fastflow/layers/coupling.py:9-105 (Conv2dZero, Coupling) -- 3x3 C/2 -> width,
// ReLU, 1x1 width -> width, ReLU, 3x3 width -> C (zero-init, * exp(3 logs)), then
// log_s = 2 tanh(h[::2] / 2), t = h[1::2], z2 = x2 * exp(log_s) + t.
#include "tc_host.cuh"
#include "tc_wgrad.cuh"

#include <cudaTypedefs.h>

#include <cstdlib>

namespace finc {
namespace tc {

#define FINC_TC_DECL(P, CL)                                                                                      \
    int launch_igemm_nhwc_p##P##_c##CL(int BN, const CUtensorMap&, const CUtensorMap&, const CUtensorMap&, const Geom&, \
                                       const EpiArgs&, cudaStream_t);
FINC_TC_DECL(1, 1) FINC_TC_DECL(1, 2) FINC_TC_DECL(1, 4) FINC_TC_DECL(3, 1) FINC_TC_DECL(3, 2) FINC_TC_DECL(3, 4)
#undef FINC_TC_DECL
int launch_igemm_rows_p1(int BN, const CUtensorMap&, const CUtensorMap&, const Geom&, const EpiArgs&, cudaStream_t);
int launch_igemm_rows_p3(int BN, const CUtensorMap&, const CUtensorMap&, const Geom&, const EpiArgs&, cudaStream_t);

int launch_igemm_nhwc(int BN, int npass, int cluster, const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& o,
                      const Geom& g, const EpiArgs& e, cudaStream_t st) {
    if (npass == 1)
        return cluster == 4   ? launch_igemm_nhwc_p1_c4(BN, a, b, o, g, e, st)
               : cluster == 2 ? launch_igemm_nhwc_p1_c2(BN, a, b, o, g, e, st)
                              : launch_igemm_nhwc_p1_c1(BN, a, b, o, g, e, st);
    return cluster == 4   ? launch_igemm_nhwc_p3_c4(BN, a, b, o, g, e, st)
           : cluster == 2 ? launch_igemm_nhwc_p3_c2(BN, a, b, o, g, e, st)
                          : launch_igemm_nhwc_p3_c1(BN, a, b, o, g, e, st);
}
int launch_igemm_rows(int BN, int npass, const CUtensorMap& a, const CUtensorMap& b, const Geom& g, const EpiArgs& e,
                      cudaStream_t st) {
    return npass == 1 ? launch_igemm_rows_p1(BN, a, b, g, e, st) : launch_igemm_rows_p3(BN, a, b, g, e, st);
}

// CTAs per cluster for the channels-last GEMMs: FINC_TC_CLUSTER = 1 | 2 | 4 (experiments), read on every call like
// the FInC plan knobs; a size the kernel cannot take is lowered below
static int cluster_size(int BN, int m_tiles) {
    const char* v = getenv("FINC_TC_CLUSTER");
    const int env = v ? atoi(v) : 0;
    int cl = env > 4 ? 4 : env > 0 ? env : 1;   // measured on B200: 1 and 2 tie (the layer is not L2-bound), 4 loses
    // (more than 4 would pass the divisibility rule at BN = 128 and launch the CL = 1 kernel with a weight box of
    // BN / cl rows, whose `full` barrier then never completes)
    while (cl > 1 && ((BN / cl) % 8 != 0 || BN % cl != 0 || m_tiles < cl || (BN == 32 && cl == 4))) cl >>= 1;
    return cl;
}

// ---- tensor maps ------------------------------------------------------------------------------
static PFN_cuTensorMapEncodeTiled_v12000 encoder() {
    static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
    }
    return fn;
}

// channels-last activation [B, H, W, C] (C % 4 == 0), box = (32 channels, wb, hb, nb) pixels, 128-byte swizzle;
// coordinates outside the tensor read as zero (= conv padding) and are dropped on stores
static int map_nhwc(CUtensorMap* m, const float* base, int C, int W, int H, int B, int wb, int hb, int nb, long ld = 0) {
    auto enc = encoder();
    if (enc == nullptr) return FINC_E_UNSUPPORTED;
    if (ld == 0) ld = C;   // floats between consecutive pixels
    cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
    cuuint64_t strides[3] = {(cuuint64_t)ld * 4, (cuuint64_t)W * ld * 4, (cuuint64_t)H * W * ld * 4};
    cuuint32_t box[4] = {(cuuint32_t)kBK, (cuuint32_t)wb, (cuuint32_t)hb, (cuuint32_t)nb};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : FINC_E_BADARG;
}
// weight matrix [rows, K] row-major, box = (32, BN)
static int map_weights(CUtensorMap* m, const float* base, long rows, int K, int BN) {
    auto enc = encoder();
    if (enc == nullptr) return FINC_E_UNSUPPORTED;
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)K * 4};
    cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)BN};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : FINC_E_BADARG;
}

// plain 2-D map over a row-major [rows, ld] matrix: box = (box_cols, box_rows), optional 128-byte swizzle
static int map_2d(CUtensorMap* m, const float* base, long rows, int cols, int ld, int box_cols, int box_rows, bool swizzle) {
    auto enc = encoder();
    if (enc == nullptr) return FINC_E_UNSUPPORTED;
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : FINC_E_BADARG;
}

static int pow2ceil(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}
static int round_up(int v, int m) { return (v + m - 1) / m * m; }

static Geom make_geom(int B, int H, int W, int taps, int Cpad, int Npad, int BN) {
    Geom g;
    g.W = W; g.H = H; g.B = B;
    g.wb = pow2ceil(W) < kBM ? pow2ceil(W) : kBM;
    g.hb = pow2ceil(H) < kBM / g.wb ? pow2ceil(H) : kBM / g.wb;
    g.nb = kBM / (g.wb * g.hb);
    g.tiles_w = (W + g.wb - 1) / g.wb;
    g.tiles_h = (H + g.hb - 1) / g.hb;
    g.tiles_n = (B + g.nb - 1) / g.nb;
    g.taps = taps;
    g.kb_per_tap = Cpad / kBK;
    g.n_tiles = Npad / BN;
    g.n_rows = Npad;
    g.group_n = 0;
    return g;
}

static int pick_bn_nhwc(int Npad) {
    return Npad % 128 == 0 ? 128 : Npad % 64 == 0 ? 64 : 32;
}

// ---- small kernels ----------------------------------------------------------------------------
// out[part][tap][n][c] (Npad x Cpad per tap, zero padded), part 0 = tf32(w), part 1 = tf32(w - tf32(w)).
//   mode 0: w is OIHW [N, Cin, kh, kw], taps = kh*kw, row n = output channel, c = input channel
//   mode 1: im2col form of a 3x3 conv: ONE tap, c = tap9 * Cin + cin          (first coupling conv)
//   mode 2: transposed + flipped (backward-data): row = input channel, c = output channel, tap -> taps-1-tap
__global__ void split_weights_kernel(const float* __restrict__ w, float* __restrict__ out, int N, int Cin, int taps,
                                     int Npad, int Cpad, int mode) {
    const int out_taps = mode == 1 ? 1 : taps;
    const long per_part = (long)out_taps * Npad * Cpad;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < per_part; idx += (long)gridDim.x * blockDim.x) {
        const int c = (int)(idx % Cpad);
        const int n = (int)((idx / Cpad) % Npad);
        const int tap = (int)(idx / ((long)Cpad * Npad));
        float v = 0.f;
        if (mode == 0) {
            if (n < N && c < Cin) v = w[((long)n * Cin + c) * taps + tap];
        } else if (mode == 1) {
            if (n < N && c < taps * Cin) v = w[((long)n * Cin + c % Cin) * taps + c / Cin];
        } else {
            if (n < Cin && c < N) v = w[((long)c * Cin + n) * taps + (taps - 1 - tap)];
        }
        const float hi = tf32_rn(v);
        out[idx] = hi;
        out[per_part + idx] = tf32_rn(v - hi);
    }
}

// A1[pixel][k] = x[n, k % Cin, h + (k / Cin) / 3 - 1, w + (k / Cin) % 3 - 1], zero outside the image and for
// k >= 9 Cin; x is NCHW with `Ctot` channels of which the first Cin are read
__global__ void im2col3x3_kernel(const float* __restrict__ x, float* __restrict__ out, int B, int Ctot, int Cin, int H,
                                 int W, int Kpad) {
    const long total = (long)B * H * W * Kpad;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int k = (int)(idx % Kpad);
        long p = idx / Kpad;
        const int pw = (int)(p % W);
        p /= W;
        const int ph = (int)(p % H);
        const int n = (int)(p / H);
        float v = 0.f;
        if (k < 9 * Cin) {
            const int tap = k / Cin, c = k - tap * Cin;
            const int hh = ph + tap / 3 - 1, ww = pw + tap % 3 - 1;
            if (hh >= 0 && hh < H && ww >= 0 && ww < W) v = __ldg(x + (((long)n * Ctot + c) * H + hh) * W + ww);
        }
        out[idx] = v;
    }
}

// logdet[n] (+)= sum_p rowsum[n, p]  in a fixed order (deterministic)
__global__ void rowsum_reduce_kernel(const float* __restrict__ rowsum, float* __restrict__ logdet, int HW,
                                     int accumulate) {
    __shared__ float red[128];
    const int n = blockIdx.x;
    float s = 0.f;
    for (int p = threadIdx.x; p < HW; p += 128) s += rowsum[(long)n * HW + p];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) logdet[n] = (accumulate ? logdet[n] : 0.f) + red[0];
}

// Last step of the coupling layer.  The 3x3 convolution width -> C ran as ONE plain GEMM
//   Y[pixel, tap * N3pad + n] = sum_c h2[pixel, c] * W3[n, c, tap]
// (the activation tile is read once, not nine times, and the MMAs are 9x wider than N = C); here
// every pixel gathers its nine neighbours' tap columns, h[n] = sum_tap Y[pixel + offset(tap), tap, n],
// and applies the coupling (layers/coupling.py:73-99): h = (h + bias) * exp(3 logs),
// log_s = 2 tanh(h[2j] / 2), t = h[2j+1], y2 = x2 * exp(log_s) + t  (reverse: (x2 - t) * exp(-log_s)).
// rowsum (nullable) gets the pixel's log-det term: sum_j log_s, or -sum_j log_s in reverse.
__global__ void coupling_gather_kernel(const float* __restrict__ Y, const float* __restrict__ bias,
                                       const float* __restrict__ scale, const float* x, float* y,
                                       float* __restrict__ rowsum, int B, int C, int H, int W, int N3pad, int reverse) {
    const long np = (long)B * H * W;
    const long pix = blockIdx.x * (long)blockDim.x + threadIdx.x;
    if (pix >= np) return;
    const int pw = (int)(pix % W), ph = (int)((pix / W) % H);
    const long n = pix / ((long)W * H);
    const int half = C / 2, ldy = 9 * N3pad;
    const size_t plane = (size_t)H * W;
    const size_t base = (size_t)n * C * plane + (size_t)ph * W + pw;
    const float* rows[9];
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
        const int hh = ph + tap / 3 - 1, ww = pw + tap % 3 - 1;
        rows[tap] = (hh >= 0 && hh < H && ww >= 0 && ww < W) ? Y + (pix + (long)(tap / 3 - 1) * W + (tap % 3 - 1)) * ldy + tap * N3pad
                                                             : nullptr;
    }
    float rs = 0.f;
    for (int jc = 0; jc < half; ++jc) {
        float hs = 0.f, tt = 0.f;
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
            if (rows[tap] != nullptr) {
                const float2 v = __ldg(reinterpret_cast<const float2*>(rows[tap]) + jc);
                hs += v.x;
                tt += v.y;
            }
        }
        hs = (hs + __ldg(bias + 2 * jc)) * __ldg(scale + 2 * jc);
        tt = (tt + __ldg(bias + 2 * jc + 1)) * __ldg(scale + 2 * jc + 1);
        const float log_s = 2.0f * tanhf(hs * 0.5f);
        const size_t o2 = base + (size_t)(half + jc) * plane;
        const float x2 = x[o2];
        y[o2] = reverse ? (x2 - tt) * expf(-log_s) : x2 * expf(log_s) + tt;
        rs += log_s;
        if (y != x) {
            const size_t o1 = base + (size_t)jc * plane;
            y[o1] = x[o1];
        }
    }
    if (rowsum != nullptr) rowsum[pix] = reverse ? -rs : rs;
}

// Backward-data forms of the three coupling weights, hi / lo split (part 1 follows part 0):
//   w2t[i][o] = w2[o][i]
//   w1t[k][o] = w1[o][c][tap],  k = tap * Cin + c      (zero rows for k >= 9 Cin)
//   w3t[c][k] = w3[n][c][tap],  k = tap * N3pad + n    (zero columns elsewhere, ld = ldY)
__global__ void coupling_bwd_weights_kernel(const float* __restrict__ w1, const float* __restrict__ w2,
                                            const float* __restrict__ w3, float* __restrict__ w2t,
                                            float* __restrict__ w1t, float* __restrict__ w3t, int C, int Cin, int width,
                                            int K1pad, int N3pad, int ldY) {
    const long n2 = (long)width * width, n1 = (long)K1pad * width, n3 = (long)width * ldY;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < n2 + n1 + n3; idx += (long)gridDim.x * blockDim.x) {
        float v = 0.f;
        float* dst;
        long part;
        if (idx < n2) {
            const int o = (int)(idx % width), i = (int)(idx / width);
            v = w2[(long)o * width + i];
            dst = w2t + idx; part = n2;
        } else if (idx < n2 + n1) {
            const long j = idx - n2;
            const int o = (int)(j % width), k = (int)(j / width);
            if (k < 9 * Cin) v = w1[((long)o * Cin + k % Cin) * 9 + k / Cin];
            dst = w1t + j; part = n1;
        } else {
            const long j = idx - n2 - n1;
            const int k = (int)(j % ldY), c = (int)(j / ldY);
            const int tap = k / N3pad, n = k % N3pad;
            if (tap < 9 && n < C) v = w3[((long)n * width + c) * 9 + tap];
            dst = w3t + j; part = n3;
        }
        const float hi = tf32_rn(v);
        dst[0] = hi;
        dst[part] = tf32_rn(v - hi);
    }
}

// Backward of the coupling's pointwise part (thread = pixel).  Recomputes h from the saved tap GEMM output Y
// (same gather as the forward), then with e = exp(log_s), log_s = 2 tanh(hs / 2):
//   forward  (y2 = x2 * e + t, logdet = sum log_s):
//     dx2 = dy2 * e;   dlog_s = dy2 * x2 * e + dlogdet[n];  dt = dy2
//   reverse  (y2 = (x2 - t) / e, logdet = -sum log_s; x is the reverse's input):
//     dx2 = dy2 / e;   dlog_s = -dy2 * y2 - dlogdet[n];     dt = -dy2 / e
//   dhs = dlog_s * (1 - tanh^2(hs / 2))
//   G3[pixel, 2j] = dhs * s3[2j],  G3[pixel, 2j+1] = dt * s3[2j+1]      (gradient at the conv output, before bias)
// and the per-pixel terms of db3 = sum G3 and dlogs3 = factor * sum G3 * (acc + b3) go to `red` [pixel][2 * N3pad]
// for a fixed-order column sum.  dx1 is initialised with dy1 (the col2im pass adds the network's part).
__global__ void coupling_bwd_pointwise_kernel(const float* __restrict__ Y, const float* __restrict__ bias,
                                              const float* __restrict__ scale, const float* __restrict__ x,
                                              const float* __restrict__ dy, const float* __restrict__ dlogdet,
                                              float* __restrict__ dx, float* __restrict__ G3, float* __restrict__ red,
                                              int B, int C, int H, int W, int N3pad, const float* __restrict__ header,
                                              int reverse) {
    const float factor = __ldg(header);   // logscale_factor of the last conv, written by finc_coupling_prepare_f32
    const long np = (long)B * H * W;
    const long pix = blockIdx.x * (long)blockDim.x + threadIdx.x;
    if (pix >= np) return;
    const int pw = (int)(pix % W), ph = (int)((pix / W) % H);
    const long n = pix / ((long)W * H);
    const int half = C / 2, ldy = 9 * N3pad;
    const size_t plane = (size_t)H * W;
    const size_t base = (size_t)n * C * plane + (size_t)ph * W + pw;
    const float* rows[9];
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
        const int hh = ph + tap / 3 - 1, ww = pw + tap % 3 - 1;
        rows[tap] = (hh >= 0 && hh < H && ww >= 0 && ww < W) ? Y + (pix + (long)(tap / 3 - 1) * W + (tap % 3 - 1)) * ldy + tap * N3pad
                                                             : nullptr;
    }
    const float dld = dlogdet != nullptr ? dlogdet[n] : 0.f;
    float* g3 = G3 + pix * N3pad;
    float* rd = red + pix * 2 * N3pad;
    for (int jc = 0; jc < N3pad / 2; ++jc) {
        float gs = 0.f, gt = 0.f, as = 0.f, at = 0.f;
        if (jc < half) {
            float hs = 0.f, tt = 0.f;
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
                if (rows[tap] != nullptr) {
                    const float2 v = __ldg(reinterpret_cast<const float2*>(rows[tap]) + jc);
                    hs += v.x;
                    tt += v.y;
                }
            }
            as = hs + __ldg(bias + 2 * jc);
            at = tt + __ldg(bias + 2 * jc + 1);
            const float s0 = __ldg(scale + 2 * jc), s1 = __ldg(scale + 2 * jc + 1);
            const float th = tanhf(as * s0 * 0.5f);
            const size_t o2 = base + (size_t)(half + jc) * plane, o1 = base + (size_t)jc * plane;
            const float d2 = dy[o2], x2 = x[o2];
            float dlog_s;
            if (reverse) {
                const float ei = expf(-2.0f * th);
                const float y2 = (x2 - at * s1) * ei;
                dx[o2] = d2 * ei;
                dx[o1] = dy[o1];
                dlog_s = -d2 * y2 - dld;
                gt = -d2 * ei * s1;
            } else {
                const float e = expf(2.0f * th);
                dx[o2] = d2 * e;
                dx[o1] = dy[o1];
                dlog_s = d2 * x2 * e + dld;
                gt = d2 * s1;
            }
            gs = dlog_s * (1.f - th * th) * s0;
        }
        g3[2 * jc] = gs;
        g3[2 * jc + 1] = gt;
        rd[2 * jc] = gs;
        rd[2 * jc + 1] = gt;
        rd[N3pad + 2 * jc] = factor * gs * as;
        rd[N3pad + 2 * jc + 1] = factor * gt * at;
    }
}

// dY[q, tap * N3pad + n] = G3[q - offset(tap), n] (zero outside the image and in the pad columns): the gradient of
// the nine-neighbour gather  h[p] = sum_tap Y[p + offset(tap), tap]
__global__ void coupling_bwd_expand_kernel(const float* __restrict__ G3, float* __restrict__ dY, int B, int H, int W,
                                           int N3pad, int ldY) {
    const long total = (long)B * H * W * (ldY / 4);
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int k4 = (int)(idx % (ldY / 4)) * 4;
        const long q = idx / (ldY / 4);
        const int qw = (int)(q % W), qh = (int)((q / W) % H);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        const int tap = k4 / N3pad, n = k4 % N3pad;   // N3pad % 16 == 0: a float4 never straddles taps
        if (tap < 9) {
            const int hh = qh - (tap / 3 - 1), ww = qw - (tap % 3 - 1);
            if (hh >= 0 && hh < H && ww >= 0 && ww < W)
                v = __ldg(reinterpret_cast<const float4*>(G3 + (q - (long)(tap / 3 - 1) * W - (tap % 3 - 1)) * N3pad + n));
        }
        *reinterpret_cast<float4*>(dY + q * ldY + k4) = v;
    }
}

// dx1[n, c, h, w] += sum_tap dA1[pixel - offset(tap), tap * Cin + c]     (col2im of the first conv's patch gradient)
__global__ void coupling_bwd_col2im_kernel(const float* __restrict__ dA1, float* __restrict__ dx, int B, int C, int Cin,
                                           int H, int W, int K1pad) {
    const long total = (long)B * Cin * H * W;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int pw = (int)(idx % W), ph = (int)((idx / W) % H);
        const int c = (int)((idx / ((long)W * H)) % Cin);
        const long n = idx / ((long)W * H * Cin);
        float s = 0.f;
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
            // patch element (pixel p, tap) holds x[p + offset(tap)]: x[q] appears in pixel q - offset(tap)
            const int hh = ph - (tap / 3 - 1), ww = pw - (tap % 3 - 1);
            if (hh >= 0 && hh < H && ww >= 0 && ww < W)
                s += __ldg(dA1 + ((n * H + hh) * W + ww) * K1pad + tap * Cin + c);
        }
        dx[((n * C + c) * H + ph) * W + pw] += s;
    }
}

// deterministic column sums of a [rows, ld] matrix.  Stage 1: block b sums rows [64 b, 64 b + 64) -- thread =
// column (coalesced), four independent accumulators; stage 2: a tree over the block partials in a fixed order.
constexpr int kColsumRows = 64;
__global__ void colsum_partial_kernel(const float* __restrict__ a, float* __restrict__ partial, long rows, int cols, int ld) {
    const long r0 = (long)blockIdx.x * kColsumRows;
    const int nr = (int)(r0 + kColsumRows < rows ? kColsumRows : rows - r0);
    for (int c = threadIdx.x; c < cols; c += blockDim.x) {
        const float* p = a + r0 * ld + c;
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
        int r = 0;
        for (; r + 4 <= nr; r += 4) {
            s0 += p[(long)r * ld];
            s1 += p[(long)(r + 1) * ld];
            s2 += p[(long)(r + 2) * ld];
            s3 += p[(long)(r + 3) * ld];
        }
        for (; r < nr; ++r) s0 += p[(long)r * ld];
        partial[(long)blockIdx.x * cols + c] = (s0 + s1) + (s2 + s3);
    }
}
// out[c] = sum_b partial[b][c]: one block per 32 columns, 8 row-lanes per column, fixed-order combination
__global__ void colsum_final_kernel(const float* __restrict__ partial, float* __restrict__ out, int nblocks, int cols) {
    __shared__ float red[8][33];
    const int c = blockIdx.x * 32 + (threadIdx.x & 31), lane_r = threadIdx.x >> 5;
    float s = 0.f;
    if (c < cols)
        for (int b = lane_r; b < nblocks; b += 8) s += partial[(long)b * cols + c];
    red[lane_r][threadIdx.x & 31] = s;
    __syncthreads();
    if (lane_r == 0 && c < cols) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x & 31];
        out[c] = t;
    }
}
static int colsum(const float* a, float* out, float* partial, long rows, int cols, int ld, cudaStream_t st) {
    const int nb = (int)((rows + kColsumRows - 1) / kColsumRows);
    colsum_partial_kernel<<<nb, 256, 0, st>>>(a, partial, rows, cols, ld);
    colsum_final_kernel<<<(cols + 31) / 32, 256, 0, st>>>(partial, out, nb, cols);
    return (int)cudaGetLastError();
}
static size_t colsum_partial_floats(long rows, int cols) { return (size_t)((rows + kColsumRows - 1) / kColsumRows) * cols; }

// dW (OIHW [N, Cin, 3, 3]) from the GEMM-form gradient: mode 1: src[o][tap * Cin + c] (ld), mode 3: src[c][tap * N3pad + n] (ld)
__global__ void wgrad_unpack_kernel(const float* __restrict__ src, float* __restrict__ dw, int N, int Cin, int ld, int N3pad,
                                    int mode) {
    const long total = (long)N * Cin * 9;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int tap = (int)(idx % 9), c = (int)((idx / 9) % Cin), n = (int)(idx / (9L * Cin));
        dw[idx] = mode == 1 ? src[(long)n * ld + tap * Cin + c] : src[(long)c * ld + tap * N3pad + n];
    }
}

// bias / scale vectors of the zero-initialised last conv: scale = exp(logscale_factor * logs)
__global__ void coupling_vectors_kernel(const float* __restrict__ b1, const float* __restrict__ b2,
                                        const float* __restrict__ b3, const float* __restrict__ logs3, float factor,
                                        float* __restrict__ o1, float* __restrict__ o2, float* __restrict__ o3,
                                        float* __restrict__ s3, int width, int C, int N3pad, float* __restrict__ header) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) header[0] = factor;
    if (i < width) {
        o1[i] = b1[i];
        o2[i] = b2[i];
    }
    if (i < N3pad) {
        o3[i] = i < C ? b3[i] : 0.f;
        s3[i] = i < C ? expf(factor * logs3[i]) : 0.f;
    }
}

// ---- prepared coupling blob ----------------------------------------------------------------------
struct CouplingLayout {
    int C, width, Cin, K1pad, N3pad, ldY;
    size_t w1, b1, w2, b2, w3, b3, s3;          // forward sections (float offsets)
    size_t w2t, w1t, w3t;                       // backward-data weights (transposed forms)
    size_t total_fwd, total;
};
static CouplingLayout coupling_layout(int C, int width) {
    CouplingLayout L;
    L.C = C; L.width = width; L.Cin = C / 2;
    L.K1pad = round_up(9 * L.Cin, 64);       // im2col width of the first conv (64: the weight-gradient GEMM's N granule)
    L.N3pad = round_up(C, 16);
    L.ldY = round_up(9 * L.N3pad, 160);      // tap-expanded gradient of the last conv: K of its backward-data GEMM
    size_t o = 32;  // header: [0] = logscale_factor
    L.w1 = o; o += (size_t)2 * width * L.K1pad;
    L.b1 = o; o += round_up(width, 32);
    L.w2 = o; o += (size_t)2 * width * width;
    L.b2 = o; o += round_up(width, 32);
    L.w3 = o; o += (size_t)2 * 9 * L.N3pad * width;
    L.b3 = o; o += round_up(L.N3pad, 32);
    L.s3 = o; o += round_up(L.N3pad, 32);
    L.total_fwd = o;
    L.w2t = o; o += (size_t)2 * width * width;        // [part][i][o]       = w2[o, i]
    L.w1t = o; o += (size_t)2 * L.K1pad * width;      // [part][k][o]       = w1[o, c, tap],  k = tap * Cin + c
    L.w3t = o; o += (size_t)2 * width * L.ldY;        // [part][c][k]       = w3[n, c, tap],  k = tap * N3pad + n
    L.total = o;
    return L;
}
static bool coupling_supported(int C, int width) {
    if (C < 2 || (C & 1) || width < 32 || width % 32 != 0 || width > 4096) return false;
    const int n3 = round_up(C, 16);
    return n3 == 16 || n3 == 32 || n3 == 48 || n3 == 64 || n3 == 96;
}

struct Workspace {
    size_t a1, h1, h2, y3, rowsum, total;  // float offsets
};
static Workspace coupling_workspace(int B, int C, int H, int W, int width) {
    const CouplingLayout L = coupling_layout(C, width);
    const size_t np = (size_t)B * H * W;
    Workspace w;
    size_t o = 0;
    w.a1 = o; o += np * L.K1pad;
    w.h1 = o; o += np * width;
    w.h2 = o; o += np * width;
    w.y3 = o; o += np * 9 * L.N3pad;
    w.rowsum = o; o += (np + 31) / 32 * 32;
    w.total = o;
    return w;
}

static int grid_for(long total, int threads) {
    long b = (total + threads - 1) / threads;
    const long cap = (long)sm_count_cached() * 16;
    return (int)(b < 1 ? 1 : b > cap ? cap : b);
}

// one channels-last convolution on the tensor cores
static int conv_nhwc(const float* x, const float* wsplit, const float* bias, const float* mask, float* y, int B, int H,
                     int W, int Cpad, int Npad, int taps, int relu, int npass, cudaStream_t st) {
    const int BN = pick_bn_nhwc(Npad);
    const Geom g = make_geom(B, H, W, taps, Cpad, Npad, BN);
    const int cl = cluster_size(BN, g.tiles_w * g.tiles_h * g.tiles_n);
    CUtensorMap mA, mB, mO;
    int rc = map_nhwc(&mA, x, Cpad, W, H, B, g.wb, g.hb, g.nb);
    if (rc) return rc;
    rc = map_weights(&mB, wsplit, (long)2 * taps * Npad, Cpad, BN / cl);
    if (rc) return rc;
    rc = map_nhwc(&mO, y, Npad, W, H, B, g.wb, g.hb, g.nb);
    if (rc) return rc;
    EpiArgs e{};
    e.bias = bias;
    e.relu = relu;
    e.mask = mask;
    e.y = y;
    e.ld_out = Npad;
    return launch_igemm_nhwc(BN, npass, cl, mA, mB, mO, g, e, st);
}

// ---- weight-gradient GEMM: dst[m, n] (+)= sum_p P[p, m] * Q[p, n] ---------------------------------------------
static int pick_bn_wgrad(int N) { return N % 160 == 0 ? 160 : N % 128 == 0 ? 128 : N % 64 == 0 ? 64 : 0; }

struct WgradPlan {
    int BN, m_tiles, n_tiles, slices, kb_per_slice;
    size_t slice_floats;
};
static WgradPlan wgrad_plan(long np, int M, int N) {
    WgradPlan p{};
    p.BN = pick_bn_wgrad(N);
    if (p.BN == 0) return p;
    p.m_tiles = (M + kBM - 1) / kBM;
    p.n_tiles = N / p.BN;
    const long kblocks = (np + kBK - 1) / kBK;
    int slices = sm_count_cached() / (p.m_tiles * p.n_tiles);
    if (slices < 1) slices = 1;
    if (slices > kblocks) slices = (int)kblocks;
    p.kb_per_slice = (int)((kblocks + slices - 1) / slices);
    p.slices = (int)((kblocks + p.kb_per_slice - 1) / p.kb_per_slice);
    p.slice_floats = (size_t)p.m_tiles * kBM * N;
    return p;
}

static int wgrad_gemm(const float* P, const float* Q, float* dst, float* workspace, long np, int M, int N, int ldP,
                      int ldQ, int ld_dst, int accumulate, int npass, cudaStream_t st) {
    const WgradPlan p = wgrad_plan(np, M, N);
    if (p.BN == 0) return FINC_E_UNSUPPORTED;
    CUtensorMap mP, mQ;
    int rc = map_2d(&mP, P, np, M, ldP, kBM, kBK, false);
    if (rc) return rc;
    rc = map_2d(&mQ, Q, np, N, ldQ, p.BN, kBK, false);
    if (rc) return rc;
    WgradGeom g{};
    g.np = (int)np;
    g.m_tiles = p.m_tiles;
    g.n_tiles = p.n_tiles;
    g.slices = p.slices;
    g.kb_per_slice = p.kb_per_slice;
    g.ld_out = N;
    g.slice_stride = p.slice_floats;
    rc = launch_wgrad(p.BN, npass, mP, mQ, workspace, g, st);
    if (rc) return rc;
    return launch_wgrad_reduce(workspace, dst, M, N, N, p.slice_floats, p.slices, ld_dst, accumulate, st);
}

}  // namespace tc
}  // namespace finc

using namespace finc;
using namespace finc::tc;

extern "C" {

size_t finc_tc_conv_weights_bytes(int N, int Cin, int taps, int mode) {
    if (N < 1 || Cin < 1 || (taps != 1 && taps != 9)) return 0;
    const int rows = mode == 2 ? Cin : N, cols = mode == 2 ? N : mode == 1 ? taps * Cin : Cin;
    const int out_taps = mode == 1 ? 1 : taps;
    return (size_t)2 * out_taps * round_up(rows, 32) * round_up(cols, kBK) * sizeof(float);
}

int finc_tc_conv_prepare_weights_f32(const float* w, void* out, int N, int Cin, int taps, int mode, void* stream) {
    if (!w || !out || N < 1 || Cin < 1 || (taps != 1 && taps != 9) || mode < 0 || mode > 2) return FINC_E_BADARG;
    const int rows = mode == 2 ? Cin : N, cols = mode == 2 ? N : mode == 1 ? taps * Cin : Cin;
    const int Npad = round_up(rows, 32), Cpad = round_up(cols, kBK);
    const long per_part = (long)(mode == 1 ? 1 : taps) * Npad * Cpad;
    split_weights_kernel<<<grid_for(per_part, 256), 256, 0, (cudaStream_t)stream>>>(w, (float*)out, N, Cin, taps, Npad,
                                                                                    Cpad, mode);
    return (int)cudaGetLastError();
}

int finc_tc_conv_nhwc_f32(const float* x, const void* wprep, const float* bias, const float* relu_mask, float* y, int B,
                          int H, int W, int Cin_pad, int Npad, int taps, int relu, unsigned flags, void* stream) {
    if (!x || !wprep || !bias || !y || B < 1 || H < 1 || W < 1 || Cin_pad < kBK || Cin_pad % kBK || Npad < 32 ||
        Npad % 32 || (taps != 1 && taps != 9))
        return FINC_E_BADARG;
    return conv_nhwc(x, (const float*)wprep, bias, relu_mask, y, B, H, W, Cin_pad, Npad, taps, relu,
                     (flags & FINC_FLAG_TF32_1PASS) ? 1 : 3, (cudaStream_t)stream);
}

size_t finc_tc_wgrad_workspace_bytes(long np, int M, int N) {
    if (np < 1 || M < 1 || N < 1) return 0;
    const WgradPlan p = wgrad_plan(np, M, N);
    return p.BN == 0 ? 0 : p.slice_floats * p.slices * sizeof(float);
}

int finc_tc_wgrad_f32(const float* P, const float* Q, float* dW, void* workspace, size_t workspace_bytes, long np, int M,
                      int N, int ldP, int ldQ, int ld_dW, unsigned flags, void* stream) {
    if (!P || !Q || !dW || !workspace || np < 1 || M < 1 || N < 1 || ldP < M || ldQ < N || ld_dW < N || (ldP & 3) ||
        (ldQ & 3))
        return FINC_E_BADARG;
    const size_t need = finc_tc_wgrad_workspace_bytes(np, M, N);
    if (need == 0) return FINC_E_UNSUPPORTED;
    if (workspace_bytes < need) return FINC_E_WORKSPACE;
    return wgrad_gemm(P, Q, dW, (float*)workspace, np, M, N, ldP, ldQ, ld_dW, (flags & FINC_FLAG_ACCUMULATE) ? 1 : 0,
                      (flags & FINC_FLAG_TF32_1PASS) ? 1 : 3, (cudaStream_t)stream);
}

size_t finc_coupling_prepared_bytes(int C, int width, int with_backward) {
    if (!coupling_supported(C, width) || (with_backward && width % 128 != 0)) return 0;
    const CouplingLayout L = coupling_layout(C, width);
    return (with_backward ? L.total : L.total_fwd) * sizeof(float);
}

size_t finc_coupling_workspace_bytes(int B, int C, int H, int W, int width) {
    if (!coupling_supported(C, width) || B < 1 || H < 1 || W < 1) return 0;
    return coupling_workspace(B, C, H, W, width).total * sizeof(float);
}

int finc_coupling_prepare_f32(const float* w1, const float* b1, const float* w2, const float* b2, const float* w3,
                              const float* b3, const float* logs3, float logscale_factor, void* prepared, int C,
                              int width, int with_backward, void* stream) {
    if (!w1 || !b1 || !w2 || !b2 || !w3 || !b3 || !logs3 || !prepared) return FINC_E_BADARG;
    if (!coupling_supported(C, width)) return FINC_E_UNSUPPORTED;
    const CouplingLayout L = coupling_layout(C, width);
    float* p = (float*)prepared;
    cudaStream_t st = (cudaStream_t)stream;
    split_weights_kernel<<<grid_for((long)width * L.K1pad, 256), 256, 0, st>>>(w1, p + L.w1, width, L.Cin, 9, width,
                                                                               L.K1pad, 1);
    split_weights_kernel<<<grid_for((long)width * width, 256), 256, 0, st>>>(w2, p + L.w2, width, width, 1, width, width,
                                                                             0);
    split_weights_kernel<<<grid_for((long)9 * L.N3pad * width, 256), 256, 0, st>>>(w3, p + L.w3, C, width, 9, L.N3pad,
                                                                                   width, 0);
    const int nv = width > L.N3pad ? width : L.N3pad;
    coupling_vectors_kernel<<<(nv + 127) / 128, 128, 0, st>>>(b1, b2, b3, logs3, logscale_factor, p + L.b1, p + L.b2,
                                                              p + L.b3, p + L.s3, width, C, L.N3pad, p);
    if (with_backward) {
        const long nb = (long)width * width + (long)L.K1pad * width + (long)width * L.ldY;
        coupling_bwd_weights_kernel<<<grid_for(nb, 256), 256, 0, st>>>(w1, w2, w3, p + L.w2t, p + L.w1t, p + L.w3t, C, L.Cin,
                                                                       width, L.K1pad, L.N3pad, L.ldY);
    }
    return (int)cudaGetLastError();
}

int finc_coupling_apply_f32(const float* x, float* y, float* logdet, const void* prepared, void* workspace,
                            size_t workspace_bytes, int B, int C, int H, int W, int width, int reverse, unsigned flags,
                            void* stream) {
    if (!x || !y || !prepared || !workspace || B < 1 || H < 1 || W < 1) return FINC_E_BADARG;
    if (!coupling_supported(C, width)) return FINC_E_UNSUPPORTED;
    const CouplingLayout L = coupling_layout(C, width);
    const Workspace ws = coupling_workspace(B, C, H, W, width);
    if (workspace_bytes < ws.total * sizeof(float)) return FINC_E_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const float* p = (const float*)prepared;
    float* wsp = (float*)workspace;
    const int npass = (flags & FINC_FLAG_TF32_1PASS) ? 1 : 3;
    const long np = (long)B * H * W;

    im2col3x3_kernel<<<grid_for(np * L.K1pad, 256), 256, 0, st>>>(x, wsp + ws.a1, B, C, L.Cin, H, W, L.K1pad);
    int rc = (int)cudaGetLastError();
    if (rc) return rc;
    rc = conv_nhwc(wsp + ws.a1, p + L.w1, p + L.b1, nullptr, wsp + ws.h1, B, H, W, L.K1pad, width, 1, 1, npass, st);
    if (rc) return rc;
    rc = conv_nhwc(wsp + ws.h1, p + L.w2, p + L.b2, nullptr, wsp + ws.h2, B, H, W, width, width, 1, 1, npass, st);
    if (rc) return rc;

    // third convolution as one GEMM over all nine taps (weight rows [tap][n] are already contiguous) ...
    const int n3 = 9 * L.N3pad;   // a multiple of 144
    const int BN = 144;
    const Geom g = make_geom(B, H, W, 1, width, n3, BN);
    CUtensorMap mA, mB;
    rc = map_nhwc(&mA, wsp + ws.h2, width, W, H, B, g.wb, g.hb, g.nb);
    if (rc) return rc;
    rc = map_weights(&mB, p + L.w3, (long)2 * n3, width, BN);
    if (rc) return rc;
    EpiArgs e{};
    e.y = wsp + ws.y3;
    e.ld_out = n3;
    rc = launch_igemm_rows(BN, npass, mA, mB, g, e, st);
    if (rc) return rc;
    // ... then the nine-neighbour gather + coupling math
    float* rowsum = logdet != nullptr ? wsp + ws.rowsum : nullptr;
    coupling_gather_kernel<<<(unsigned)((np + 127) / 128), 128, 0, st>>>(wsp + ws.y3, p + L.b3, p + L.s3, x, y, rowsum, B,
                                                                        C, H, W, L.N3pad, reverse);
    rc = (int)cudaGetLastError();
    if (rc) return rc;
    if (rowsum != nullptr) {
        rowsum_reduce_kernel<<<B, 128, 0, st>>>(wsp + ws.rowsum, logdet, H * W,
                                               (flags & FINC_FLAG_LOGDET_ACCUMULATE) ? 1 : 0);
        rc = (int)cudaGetLastError();
    }
    return rc;
}


// ---- backward of the coupling layer ---------------------------------------------------------------------------
struct BwdScratch {
    size_t g3, red, dY, dh2, dh1, dA1, wcat, part, ws, total;  // float offsets
};
static BwdScratch coupling_bwd_scratch(int B, int C, int H, int W, int width) {
    const CouplingLayout L = coupling_layout(C, width);
    const size_t np = (size_t)B * H * W;
    BwdScratch b;
    size_t o = 0;
    b.g3 = o; o += np * L.N3pad;
    b.red = o; o += np * 2 * L.N3pad;
    b.dY = o; o += np * L.ldY;
    b.dh2 = o; o += np * width;
    b.dh1 = o; o += np * width;
    b.dA1 = o; o += np * L.K1pad;
    b.wcat = o; o += (size_t)width * (L.ldY > L.K1pad ? L.ldY : L.K1pad);
    b.part = o; o += colsum_partial_floats((long)np, width > 2 * L.N3pad ? width : 2 * L.N3pad);
    size_t ws = finc_tc_wgrad_workspace_bytes((long)np, width, width);
    const size_t w3 = finc_tc_wgrad_workspace_bytes((long)np, width, L.ldY), w1 = finc_tc_wgrad_workspace_bytes((long)np, width, L.K1pad);
    ws = ws > w3 ? ws : w3;
    ws = ws > w1 ? ws : w1;
    b.ws = o; o += ws / sizeof(float) + 32;
    b.total = o;
    return b;
}

size_t finc_coupling_backward_workspace_bytes(int B, int C, int H, int W, int width) {
    if (!coupling_supported(C, width) || width % 128 != 0 || B < 1 || H < 1 || W < 1) return 0;
    return coupling_bwd_scratch(B, C, H, W, width).total * sizeof(float);
}

int finc_coupling_backward_f32(const float* x, const float* dy, const float* dlogdet, const void* prepared,
                               const void* forward_workspace, void* scratch, size_t scratch_bytes, float* dx,
                               float* dw1, float* db1, float* dw2, float* db2, float* dw3, float* db3, float* dlogs3,
                               int B, int C, int H, int W, int width, unsigned flags, void* stream) {
    if (!x || !dy || !prepared || !forward_workspace || !scratch || !dx || !dw1 || !db1 || !dw2 || !db2 || !dw3 || !db3 ||
        !dlogs3 || B < 1 || H < 1 || W < 1 || dx == x || dx == dy)
        return FINC_E_BADARG;
    if (!coupling_supported(C, width) || width % 128 != 0) return FINC_E_UNSUPPORTED;
    const CouplingLayout L = coupling_layout(C, width);
    const Workspace fw = coupling_workspace(B, C, H, W, width);
    const BwdScratch sc = coupling_bwd_scratch(B, C, H, W, width);
    if (scratch_bytes < sc.total * sizeof(float)) return FINC_E_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const float* p = (const float*)prepared;
    const float* fws = (const float*)forward_workspace;
    float* s = (float*)scratch;
    const int npass = (flags & FINC_FLAG_TF32_1PASS) ? 1 : 3;
    const long np = (long)B * H * W;
    const float* A1 = fws + fw.a1;
    const float* h1 = fws + fw.h1;
    const float* h2 = fws + fw.h2;
    const float* Y = fws + fw.y3;

    // 1. pointwise part: dx2, dx1 = dy1, gradient at the last conv's output, per-pixel terms of db3 / dlogs3 (the only
    //    step that depends on the direction: the network h = net(x1) is the same in both)
    coupling_bwd_pointwise_kernel<<<(unsigned)((np + 127) / 128), 128, 0, st>>>(
        Y, p + L.b3, p + L.s3, x, dy, dlogdet, dx, s + sc.g3, s + sc.red, B, C, H, W, L.N3pad, p,
        (flags & FINC_FLAG_COUPLING_REVERSE) ? 1 : 0);
    int rc = colsum(s + sc.red, s + sc.wcat, s + sc.part, np, 2 * L.N3pad, 2 * L.N3pad, st);
    if (rc) return rc;
    cudaMemcpyAsync(db3, s + sc.wcat, C * sizeof(float), cudaMemcpyDeviceToDevice, st);
    cudaMemcpyAsync(dlogs3, s + sc.wcat + L.N3pad, C * sizeof(float), cudaMemcpyDeviceToDevice, st);
    // 2. expand over the nine taps; dW3 = h2^T dY; dh2 = (dY W3t) * (h2 > 0)
    coupling_bwd_expand_kernel<<<grid_for(np * (L.ldY / 4), 256), 256, 0, st>>>(s + sc.g3, s + sc.dY, B, H, W, L.N3pad, L.ldY);
    rc = wgrad_gemm(h2, s + sc.dY, s + sc.wcat, s + sc.ws, np, width, L.ldY, width, L.ldY, L.ldY, 0, npass, st);
    if (rc) return rc;
    wgrad_unpack_kernel<<<grid_for((long)C * width * 9, 256), 256, 0, st>>>(s + sc.wcat, dw3, C, width, L.ldY, L.N3pad, 3);
    rc = conv_nhwc(s + sc.dY, p + L.w3t, nullptr, h2, s + sc.dh2, B, H, W, L.ldY, width, 1, 0, npass, st);
    if (rc) return rc;
    // 3. middle 1x1: db2, dW2 = dh2^T h1, dh1 = (dh2 W2) * (h1 > 0)
    rc = colsum(s + sc.dh2, db2, s + sc.part, np, width, width, st);
    if (rc) return rc;
    rc = wgrad_gemm(s + sc.dh2, h1, dw2, s + sc.ws, np, width, width, width, width, width, 0, npass, st);
    if (rc) return rc;
    rc = conv_nhwc(s + sc.dh2, p + L.w2t, nullptr, h1, s + sc.dh1, B, H, W, width, width, 1, 0, npass, st);
    if (rc) return rc;
    // 4. first 3x3 (im2col form): db1, dW1 = dh1^T A1, dA1 = dh1 W1, dx1 += col2im(dA1)
    rc = colsum(s + sc.dh1, db1, s + sc.part, np, width, width, st);
    if (rc) return rc;
    rc = wgrad_gemm(s + sc.dh1, A1, s + sc.wcat, s + sc.ws, np, width, L.K1pad, width, L.K1pad, L.K1pad, 0, npass, st);
    if (rc) return rc;
    wgrad_unpack_kernel<<<grid_for((long)width * L.Cin * 9, 256), 256, 0, st>>>(s + sc.wcat, dw1, width, L.Cin, L.K1pad, 0, 1);
    {
        const Geom g = make_geom(B, H, W, 1, width, L.K1pad, 64);
        CUtensorMap mA, mB;
        rc = map_nhwc(&mA, s + sc.dh1, width, W, H, B, g.wb, g.hb, g.nb);
        if (rc) return rc;
        rc = map_weights(&mB, p + L.w1t, (long)2 * L.K1pad, width, 64);
        if (rc) return rc;
        EpiArgs e{};
        e.y = s + sc.dA1;
        e.ld_out = L.K1pad;
        rc = launch_igemm_rows(64, npass, mA, mB, g, e, st);
        if (rc) return rc;
    }
    coupling_bwd_col2im_kernel<<<grid_for((long)B * L.Cin * H * W, 256), 256, 0, st>>>(s + sc.dA1, dx, B, C, L.Cin, H, W, L.K1pad);
    return (int)cudaGetLastError();
}


// ---- dense form of the FInC inverse for small tiles -----------------------------------------------------------
// The inverse of a FInC convolution is x = L^-1 z with L the (unit lower-triangular after reordering) matrix of
// the convolution over the n = C*H*W unknowns of one (image, group).  For the deep, small levels (4x4, 8x8
// tiles: n <= 1024) L^-1 is small and the same for every image, so a batch is ONE GEMM X = Z (L^-1)^T per group on
// the tensor cores instead of a wavefront recurrence whose parallelism is a diagonal of 4 .. 8 pixels:
// [2048,96,4,4] k=5: 298 us on the wavefront kernel (FP32-pipe bound, 17 % of its peak); [2048,48,8,8] k=5: 224 us.
// L^-1 is obtained by running the wavefront kernel itself on the identity (n unit images), once per weight update.

// prepared[part][g][i][j] = X[j][g][i] (hi / lo split): row i of L_g^-1, K-major; all groups' rows stacked per part
__global__ void dense_inverse_weights_kernel(const float* __restrict__ X, float* __restrict__ out, int G, int n) {
    const long per_part = (long)n * n;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < per_part * G; idx += (long)gridDim.x * blockDim.x) {
        const int g = (int)(idx / per_part);
        const long r = idx - g * per_part;
        const int j = (int)(r % n), i = (int)(r / n);
        const float v = X[((long)j * G + g) * n + i];
        const float hi = tf32_rn(v);
        float* o = out + (long)g * per_part + r;
        o[0] = hi;
        o[per_part * G] = tf32_rn(v - hi);
    }
}
// identity batch: image j of group g is the unit vector e_j  ->  Z[j][g][i] = (i == j)
__global__ void dense_identity_kernel(float* __restrict__ Z, int G, int n) {
    const long total = (long)n * G * n;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int i = (int)(idx % n);
        const int j = (int)(idx / ((long)G * n));
        Z[idx] = i == j ? 1.f : 0.f;
    }
}

static int dense_n(int C, int H, int W) {
    const long n = (long)C * H * W;
    return (n >= 64 && n <= 1024 && n % 64 == 0) ? (int)n : 0;
}

size_t finc_inverse_dense_bytes(int G, int C, int H, int W) {
    const int n = dense_n(C, H, W);
    return (n == 0 || G < 1 || G > 16) ? 0 : (size_t)G * 2 * n * n * sizeof(float);
}
size_t finc_inverse_dense_scratch_bytes(int G, int C, int H, int W) {
    const int n = dense_n(C, H, W);
    return (n == 0 || G < 1 || G > 16) ? 0 : (size_t)2 * n * G * n * sizeof(float);
}

int finc_inverse_dense_prepare_f32(const float* w, void* prepared, void* scratch, size_t scratch_bytes, int G, int C, int H,
                                   int W, int kH, int kW, unsigned orders, void* stream) {
    const int n = dense_n(C, H, W);
    if (!w || !prepared || !scratch) return FINC_E_BADARG;
    if (n == 0 || G < 1 || G > 16) return FINC_E_UNSUPPORTED;
    if (scratch_bytes < finc_inverse_dense_scratch_bytes(G, C, H, W)) return FINC_E_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    float* Z = (float*)scratch;
    float* X = Z + (size_t)n * G * n;
    dense_identity_kernel<<<grid_for((long)n * G * n, 256), 256, 0, st>>>(Z, G, n);
    int rc = finc_inverse_f32(Z, w, X, n, G, C, H, W, kH, kW, orders, 0, stream);   // column j of L_g^-1 = inverse(e_j)
    if (rc) return rc;
    dense_inverse_weights_kernel<<<grid_for((long)n * n * G, 256), 256, 0, st>>>(X, (float*)prepared, G, n);
    return (int)cudaGetLastError();
}

int finc_inverse_dense_f32(const float* z, const void* prepared, float* x, int B, int G, int C, int H, int W, unsigned flags,
                           void* stream) {
    const int n = dense_n(C, H, W);
    if (!z || !prepared || !x || B < 0 || z == x) return FINC_E_BADARG;
    if (n == 0 || G < 1 || G > 16) return FINC_E_UNSUPPORTED;
    if (B == 0) return FINC_OK;
    const int npass = (flags & FINC_FLAG_TF32_1PASS) ? 1 : 3;
    const int BN = n % 128 == 0 ? 128 : 64;
    // ONE block-diagonal GEMM: "pixels" = images, output columns = the G*n unknowns, each group reading its own n inputs
    Geom g = make_geom(1, 1, B, 1, n, G * n, BN);
    g.group_n = n;
    CUtensorMap mA, mB;
    int rc = map_nhwc(&mA, z, G * n, B, 1, 1, g.wb, g.hb, g.nb);
    if (rc) return rc;
    rc = map_weights(&mB, (const float*)prepared, (long)2 * G * n, n, BN);
    if (rc) return rc;
    EpiArgs e{};
    e.y = x;
    e.ld_out = G * n;
    return launch_igemm_rows(BN, npass, mA, mB, g, e, (cudaStream_t)stream);
}

}  // extern "C"

// finc_affine.cu -- per-pixel channel affine map y[n,:,p] = A x[n,:,p] + b, sm_100a.
//
// First "next" row of the scope table (SURVEY.md 8f): the glue that follows every FastFlowUnit
// in the reference's flow step is ActNorm (layers/actnorm.py:14-52: (x - t) * exp(-log_s) per
// channel) and Conv1x1 (layers/conv1x1.py:18-43: z = W x per pixel).  Both are per-pixel affine
// maps over the channel axis, so their composition is ONE such map with A = W diag(exp(-log_s)),
// b = -A t (and the reverse is the map with A^-1, +t): one HBM round trip instead of two, no
// per-call torch.inverse.  The same kernel with A^T is the backward-data pass.
//
// HBM-bound streaming kernel (2*C flop per 8 bytes): a thread owns VEC consecutive pixels of one
// image, reads its C channel vectors with coalesced vector loads (NCHW: channel stride = H*W),
// keeps them in registers and produces the C outputs four at a time with the rows of A^T as
// 128-bit shared-memory broadcasts (one LDS.128 feeds 4*VEC FMAs).
#include "finc_common.cuh"

namespace finc {

namespace {

template <int VEC>
struct VecT;
template <>
struct VecT<4> { using type = float4; };
template <>
struct VecT<2> { using type = float2; };
template <>
struct VecT<1> { using type = float; };

template <int VEC>
__device__ __forceinline__ void ldv(const float* p, float* out) {
    if constexpr (VEC == 4) {
        const float4 v = __ldcs(reinterpret_cast<const float4*>(p));
        out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
    } else if constexpr (VEC == 2) {
        const float2 v = __ldcs(reinterpret_cast<const float2*>(p));
        out[0] = v.x; out[1] = v.y;
    } else {
        out[0] = __ldcs(p);
    }
}
template <int VEC>
__device__ __forceinline__ void stv(float* p, const float* v) {
    if constexpr (VEC == 4) *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    else if constexpr (VEC == 2) *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
    else p[0] = v[0];
}

template <int C, int VEC>
__global__ void __launch_bounds__(256) affine1x1_kernel(const float* __restrict__ x, const float* __restrict__ A,
                                                        const float* __restrict__ bias, float* __restrict__ y,
                                                        long n_items, int hwv, long HW) {
    constexpr int CP = (C + 3) & ~3;
    __shared__ __align__(16) float At[C * CP];  // At[i][o] = A[o][i]
    __shared__ __align__(16) float bs[CP];
    for (int e = threadIdx.x; e < C * CP; e += blockDim.x) {
        const int i = e / CP, o = e - i * CP;
        At[e] = o < C ? __ldg(A + o * C + i) : 0.f;
    }
    for (int o = threadIdx.x; o < CP; o += blockDim.x) bs[o] = (bias != nullptr && o < C) ? __ldg(bias + o) : 0.f;
    __syncthreads();
    for (long item = (long)blockIdx.x * blockDim.x + threadIdx.x; item < n_items; item += (long)gridDim.x * blockDim.x) {
        const long n = item / hwv;
        const long off = n * C * HW + (item - n * hwv) * VEC;
        float xv[C][VEC];
#pragma unroll
        for (int i = 0; i < C; ++i) ldv<VEC>(x + off + i * HW, xv[i]);
#pragma unroll
        for (int ob = 0; ob < CP / 4; ++ob) {
            float acc[4][VEC];
            const float4 b4 = *reinterpret_cast<const float4*>(bs + 4 * ob);
#pragma unroll
            for (int v = 0; v < VEC; ++v) { acc[0][v] = b4.x; acc[1][v] = b4.y; acc[2][v] = b4.z; acc[3][v] = b4.w; }
#pragma unroll
            for (int i = 0; i < C; ++i) {
                const float4 a = *reinterpret_cast<const float4*>(At + i * CP + 4 * ob);
#pragma unroll
                for (int v = 0; v < VEC; ++v) {
                    acc[0][v] = fmaf(a.x, xv[i][v], acc[0][v]);
                    acc[1][v] = fmaf(a.y, xv[i][v], acc[1][v]);
                    acc[2][v] = fmaf(a.z, xv[i][v], acc[2][v]);
                    acc[3][v] = fmaf(a.w, xv[i][v], acc[3][v]);
                }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (4 * ob + k < C) stv<VEC>(y + off + (4 * ob + k) * HW, acc[k]);
        }
    }
}

// Small problems (a few thousand pixels: the 4x4 and 8x8 levels at batch 256): the kernel above has one thread
// per VEC pixels computing ALL C outputs -- C*C*VEC dependent FMAs per thread on a grid of a few CTAs
// ([256,48,4,4]: 8 CTAs, 15.9 us = 1.5 % of the HBM peak).  Here a thread computes FOUR outputs of ONE pixel:
// C/4 times more threads, a C-long critical path, the re-read inputs come from L1.  Pixel index fastest, so a
// warp reads / writes 128 contiguous bytes per channel and its A^T vector is a shared-memory broadcast.
template <int C>
__global__ void __launch_bounds__(256) affine1x1_split_kernel(const float* __restrict__ x, const float* __restrict__ A,
                                                              const float* __restrict__ bias, float* __restrict__ y,
                                                              long npix, long HW) {
    constexpr int CP = (C + 3) & ~3;
    __shared__ __align__(16) float At[C * CP];
    __shared__ __align__(16) float bs[CP];
    for (int e = threadIdx.x; e < C * CP; e += blockDim.x) {
        const int i = e / CP, o = e - i * CP;
        At[e] = o < C ? __ldg(A + o * C + i) : 0.f;
    }
    for (int o = threadIdx.x; o < CP; o += blockDim.x) bs[o] = (bias != nullptr && o < C) ? __ldg(bias + o) : 0.f;
    __syncthreads();
    const long total = npix * (CP / 4);
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const long p = idx % npix;
        const int ob = (int)(idx / npix);
        const long n = p / HW;
        const long off = n * C * HW + (p - n * HW);
        const float4 b4 = *reinterpret_cast<const float4*>(bs + 4 * ob);
        float a0 = b4.x, a1 = b4.y, a2 = b4.z, a3 = b4.w;
#pragma unroll
        for (int i = 0; i < C; ++i) {
            const float xv = __ldg(x + off + i * HW);
            const float4 a = *reinterpret_cast<const float4*>(At + i * CP + 4 * ob);
            a0 = fmaf(a.x, xv, a0); a1 = fmaf(a.y, xv, a1); a2 = fmaf(a.z, xv, a2); a3 = fmaf(a.w, xv, a3);
        }
        float* yp = y + off + (long)(4 * ob) * HW;
        yp[0] = a0;
        if (4 * ob + 1 < C) yp[HW] = a1;
        if (4 * ob + 2 < C) yp[2 * HW] = a2;
        if (4 * ob + 3 < C) yp[3 * HW] = a3;
    }
}

template <int C>
int launch_split(const float* x, const float* A, const float* bias, float* y, int B, long HW, cudaStream_t st) {
    const long npix = (long)B * HW;
    const long total = npix * ((C + 3) / 4);
    const long blocks = (total + 255) / 256;
    const long cap = (long)sm_count_cached() * 8;
    affine1x1_split_kernel<C><<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, st>>>(x, A, bias, y, npix, HW);
    return (int)cudaGetLastError();
}

// any C: one thread per output element (coalesced along the pixels)
__global__ void affine1x1_generic_kernel(const float* __restrict__ x, const float* __restrict__ A,
                                         const float* __restrict__ bias, float* __restrict__ y, long total, int C,
                                         long HW) {
    for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long)gridDim.x * blockDim.x) {
        const long p = e % HW;
        const long no = e / HW;
        const int o = (int)(no % C);
        const long n = no / C;
        float acc = bias ? __ldg(bias + o) : 0.f;
        const float* xp = x + n * C * HW + p;
        for (int i = 0; i < C; ++i) acc = fmaf(__ldg(A + o * C + i), xp[i * HW], acc);
        y[e] = acc;
    }
}

template <int C, int VEC>
int launch_inst(const float* x, const float* A, const float* bias, float* y, int B, long HW, cudaStream_t st) {
    const long n_items = (long)B * (HW / VEC);
    const long blocks = (n_items + 255) / 256;
    const long cap = (long)sm_count_cached() * 8;
    affine1x1_kernel<C, VEC><<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, st>>>(x, A, bias, y, n_items, (int)(HW / VEC), HW);
    return (int)cudaGetLastError();
}

template <int C, int VMAX>
int dispatch_vec(int vec, const float* x, const float* A, const float* bias, float* y, int B, long HW, cudaStream_t st) {
    if constexpr (VMAX >= 4) { if (vec == 4) return launch_inst<C, 4>(x, A, bias, y, B, HW, st); }
    if constexpr (VMAX >= 2) { if (vec >= 2) return launch_inst<C, 2>(x, A, bias, y, B, HW, st); }
    return launch_inst<C, 1>(x, A, bias, y, B, HW, st);
}

// ---- weight gradient of the per-pixel affine map ------------------------------------------------
//   dA[o, i] = sum_{n,p} dy[n, o, p] * x[n, i, p],   db[o] = sum_{n,p} dy[n, o, p]
// A C x C outer-product accumulation over all B*HW pixels (the autograd of ActNorm + Conv1x1:
// dW, dlog_scale and dtranslation follow from dA / db by the chain rule on the host).  CTAs stride
// over tiles of PT pixels; a tile of x and dy is staged channel-major in shared memory, thread
// (4x4 block of (o, i), pixel slice) accumulates 16 products per pixel from 128-bit loads; slices
// meet in shared memory in fixed order, CTAs write partials, a second launch sums them in CTA order
// (deterministic, no floating-point atomics).
constexpr int kAwPT = 64;       // pixels per tile
constexpr int kAwPitch = kAwPT + 4;
constexpr int kAwRounds = 3;    // 4x4 blocks per thread: (C/4)^2 <= 3 * 256  <=>  C <= 108

__global__ void __launch_bounds__(256) affine1x1_wgrad_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                              float* __restrict__ partial, int C, long HW,
                                                              long npix, long ntiles, int slices) {
    extern __shared__ __align__(16) float sm[];
    float* xs = sm;                       // [C][kAwPitch]
    float* ds = sm + (size_t)C * kAwPitch;  // [C][kAwPitch]
    const int nib = C >> 2, nblk = nib * nib;
    const int tid = threadIdx.x;
    float acc[kAwRounds][4][4];
    float dsum[kAwRounds][4];
#pragma unroll
    for (int r = 0; r < kAwRounds; ++r)
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            dsum[r][a] = 0.f;
#pragma unroll
            for (int b = 0; b < 4; ++b) acc[r][a][b] = 0.f;
        }
    // thread -> (block, slice) for round r: unit = tid + r * 256; block = unit / slices
    const bool vec = (HW % 4 == 0) && ((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(x)) & 15) == 0;
    for (long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long P0 = tile * kAwPT;
        __syncthreads();  // previous tile fully consumed
        if (vec) {
            for (int e = tid; e < C * (kAwPT / 4); e += blockDim.x) {
                const int c = e / (kAwPT / 4), q = (e - c * (kAwPT / 4)) * 4;
                const long P = P0 + q;
                float4 vx = make_float4(0.f, 0.f, 0.f, 0.f), vd = vx;
                if (P < npix) {
                    const long n = P / HW, pp = P - n * HW;
                    const long off = (n * C + c) * HW + pp;
                    vx = __ldcs(reinterpret_cast<const float4*>(x + off));
                    vd = __ldcs(reinterpret_cast<const float4*>(dy + off));
                }
                *reinterpret_cast<float4*>(xs + c * kAwPitch + q) = vx;
                *reinterpret_cast<float4*>(ds + c * kAwPitch + q) = vd;
            }
        } else {
            for (int e = tid; e < C * kAwPT; e += blockDim.x) {
                const int c = e / kAwPT, q = e - c * kAwPT;
                const long P = P0 + q;
                float vx = 0.f, vd = 0.f;
                if (P < npix) {
                    const long n = P / HW, pp = P - n * HW;
                    const long off = (n * C + c) * HW + pp;
                    vx = x[off];
                    vd = dy[off];
                }
                xs[c * kAwPitch + q] = vx;
                ds[c * kAwPitch + q] = vd;
            }
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < kAwRounds; ++r) {
            const int unit = tid + r * 256;
            const int blk = unit / slices, sl = unit - blk * slices;
            if (blk < nblk) {
                const int ob = blk / nib, ib = blk - ob * nib;
                const float* dp = ds + (ob * 4) * kAwPitch;
                const float* xp = xs + (ib * 4) * kAwPitch;
                for (int q = sl * 4; q < kAwPT; q += slices * 4) {
                    float4 d4[4], x4[4];
#pragma unroll
                    for (int a = 0; a < 4; ++a) {
                        d4[a] = *reinterpret_cast<const float4*>(dp + a * kAwPitch + q);
                        x4[a] = *reinterpret_cast<const float4*>(xp + a * kAwPitch + q);
                    }
#pragma unroll
                    for (int a = 0; a < 4; ++a) {
#pragma unroll
                        for (int b = 0; b < 4; ++b) {
                            acc[r][a][b] = fmaf(d4[a].x, x4[b].x, acc[r][a][b]);
                            acc[r][a][b] = fmaf(d4[a].y, x4[b].y, acc[r][a][b]);
                            acc[r][a][b] = fmaf(d4[a].z, x4[b].z, acc[r][a][b]);
                            acc[r][a][b] = fmaf(d4[a].w, x4[b].w, acc[r][a][b]);
                        }
                        if (ib == 0) dsum[r][a] += (d4[a].x + d4[a].y) + (d4[a].z + d4[a].w);
                    }
                }
            }
        }
    }
    // slices of a block meet in shared memory in slice order, then the CTA writes its partial
    __syncthreads();
    float* part = sm;  // [C*C + C], the staging buffers are free now
    for (int s_ = 0; s_ < slices; ++s_) {
#pragma unroll
        for (int r = 0; r < kAwRounds; ++r) {
            const int unit = tid + r * 256;
            const int blk = unit / slices, sl = unit - blk * slices;
            if (blk < nblk && sl == s_) {
                const int ob = blk / nib, ib = blk - ob * nib;
#pragma unroll
                for (int a = 0; a < 4; ++a) {
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        float* dst = part + (ob * 4 + a) * C + ib * 4 + b;
                        *dst = (s_ == 0 ? 0.f : *dst) + acc[r][a][b];
                    }
                    if (ib == 0) {
                        float* dst = part + C * C + ob * 4 + a;
                        *dst = (s_ == 0 ? 0.f : *dst) + dsum[r][a];
                    }
                }
            }
        }
        __syncthreads();
    }
    const int nout = C * C + C;
    for (int e = tid; e < nout; e += blockDim.x) partial[(size_t)blockIdx.x * nout + e] = part[e];
}

__global__ void affine1x1_wgrad_finish_kernel(const float* __restrict__ partial, float* __restrict__ dA,
                                              float* __restrict__ db, int C, int nctas) {
    const int nout = C * C + C;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < nout; e += gridDim.x * blockDim.x) {
        float v = 0.f;
        for (int c = 0; c < nctas; ++c) v += partial[(size_t)c * nout + e];
        if (e < C * C) dA[e] = v;
        else if (db != nullptr) db[e - C * C] = v;
    }
}

// any C: one thread per output, fixed summation order
__global__ void affine1x1_wgrad_generic_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                               float* __restrict__ dA, float* __restrict__ db, int B, int C, long HW) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= C * C + C) return;
    const bool bias = e >= C * C;
    const int o = bias ? e - C * C : e / C, i = bias ? 0 : e - o * C;
    float v = 0.f;
    for (int n = 0; n < B; ++n) {
        const float* dp = dy + ((long)n * C + o) * HW;
        const float* xp = x + ((long)n * C + i) * HW;
        for (long p = 0; p < HW; ++p) v += bias ? dp[p] : dp[p] * xp[p];
    }
    if (!bias) dA[e] = v;
    else if (db != nullptr) db[o] = v;
}

int affine_wgrad_ctas(int B, long HW) {
    const long ntiles = ((long)B * HW + kAwPT - 1) / kAwPT;
    const long cap = (long)sm_count_cached() * 2;
    return (int)(ntiles < cap ? ntiles : cap);
}

}  // namespace

size_t affine1x1_wgrad_workspace_floats(int B, int C, long HW) {
    if (C % 4 != 0 || (C / 4) * (C / 4) > kAwRounds * 256) return 16;  // generic kernel: no partials
    return (size_t)affine_wgrad_ctas(B, HW) * ((size_t)C * C + C) + 16;
}

int launch_affine1x1_wgrad(const float* dy, const float* x, float* dA, float* db, float* workspace, size_t ws_floats,
                           int B, int C, long HW, cudaStream_t st) {
    if (C % 4 != 0 || (C / 4) * (C / 4) > kAwRounds * 256) {
        const int nout = C * C + C;
        affine1x1_wgrad_generic_kernel<<<(nout + 127) / 128, 128, 0, st>>>(dy, x, dA, db, B, C, HW);
        return (int)cudaGetLastError();
    }
    if (ws_floats < affine1x1_wgrad_workspace_floats(B, C, HW)) return FINC_E_WORKSPACE;
    const int nblk = (C / 4) * (C / 4);
    int slices = 256 / nblk;
    if (slices < 1) slices = 1;
    if (slices > kAwPT / 4) slices = kAwPT / 4;
    const int nctas = affine_wgrad_ctas(B, HW);
    const long npix = (long)B * HW;
    const long ntiles = (npix + kAwPT - 1) / kAwPT;
    size_t smem = (size_t)2 * C * kAwPitch * sizeof(float);
    const size_t need_part = ((size_t)C * C + C) * sizeof(float);
    if (smem < need_part) smem = need_part;
    cudaError_t e = cudaFuncSetAttribute(affine1x1_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    affine1x1_wgrad_kernel<<<nctas, 256, smem, st>>>(dy, x, workspace, C, HW, npix, ntiles, slices);
    e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
    const int nout = C * C + C;
    affine1x1_wgrad_finish_kernel<<<(nout + 255) / 256, 256, 0, st>>>(workspace, dA, db, C, nctas);
    return (int)cudaGetLastError();
}

int launch_affine1x1(const float* x, const float* A, const float* bias, float* y, int B, int C, long HW, cudaStream_t st) {
    // widest vector the layout allows: rows start at multiples of HW floats from 16-byte aligned bases
    int vec = 1;
    const uintptr_t al = reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y);
    if (HW % 4 == 0 && (al & 15) == 0) vec = 4;
    else if (HW % 2 == 0 && (al & 7) == 0) vec = 2;
    // fewer pixel-vectors than ~2 waves of threads: split the output channels over threads instead
    const int vmax = C >= 96 ? 1 : C >= 32 ? 2 : 4;
    const long items = (long)B * (HW / (vec < vmax ? vec : vmax));
    if (items < (long)sm_count_cached() * 512) {
        switch (C) {
            case 4: return launch_split<4>(x, A, bias, y, B, HW, st);
            case 8: return launch_split<8>(x, A, bias, y, B, HW, st);
            case 12: return launch_split<12>(x, A, bias, y, B, HW, st);
            case 16: return launch_split<16>(x, A, bias, y, B, HW, st);
            case 24: return launch_split<24>(x, A, bias, y, B, HW, st);
            case 32: return launch_split<32>(x, A, bias, y, B, HW, st);
            case 48: return launch_split<48>(x, A, bias, y, B, HW, st);
            case 96: return launch_split<96>(x, A, bias, y, B, HW, st);
            default: break;
        }
    }
    switch (C) {
        case 4: return dispatch_vec<4, 4>(vec, x, A, bias, y, B, HW, st);
        case 8: return dispatch_vec<8, 4>(vec, x, A, bias, y, B, HW, st);
        case 12: return dispatch_vec<12, 4>(vec, x, A, bias, y, B, HW, st);
        case 16: return dispatch_vec<16, 4>(vec, x, A, bias, y, B, HW, st);
        case 24: return dispatch_vec<24, 4>(vec, x, A, bias, y, B, HW, st);
        case 32: return dispatch_vec<32, 2>(vec, x, A, bias, y, B, HW, st);
        case 48: return dispatch_vec<48, 2>(vec, x, A, bias, y, B, HW, st);
        case 96: return dispatch_vec<96, 1>(vec, x, A, bias, y, B, HW, st);
        default: break;
    }
    const long total = (long)B * C * HW;
    const long blocks = (total + 255) / 256;
    const long cap = (long)sm_count_cached() * 16;
    affine1x1_generic_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, st>>>(x, A, bias, y, total, C, HW);
    return (int)cudaGetLastError();
}

}  // namespace finc

// ---------------------------------------------------------------------------------------------
// Preprocess (fastflow_cifar_multi_gpu.py:162-186): Dequantization (layers/dequantize.py:13-19),
// Normalization(0, 256), Normalization(-alpha, 1 / (1 - 2 alpha)) (layers/normalize.py:18-31) and
// LogitTransform (layers/transforms.py:11-18) with their four log-determinants, as ONE pass:
//   p = ((x + u) / 256 + alpha) * (1 - 2 alpha);   y = log p - log(1 - p)
//   logdet[n] = D * (log(1 - 2 alpha) - log 256) + sum_d (-log p - log(1 - p))
// reverse: x = floor((sigmoid(y) / (1 - 2 alpha) - alpha) * 256).  One CTA per image, fixed-order sum.
// ---------------------------------------------------------------------------------------------
namespace finc {

__global__ void preprocess_kernel(const float* __restrict__ x, const float* __restrict__ u, float* __restrict__ y,
                                  float* __restrict__ logdet, long D, float alpha, int reverse) {
    __shared__ float red[256];
    const long base = (long)blockIdx.x * D;
    const float s = 1.f - 2.f * alpha;
    float acc = 0.f;
    for (long d = threadIdx.x; d < D; d += blockDim.x) {
        if (reverse) {
            const float p = 1.f / (1.f + expf(-x[base + d]));
            y[base + d] = floorf((p / s - alpha) * 256.f);
        } else {
            const float v = x[base + d] + (u != nullptr ? u[base + d] : 0.f);
            const float p = (v / 256.f + alpha) * s;
            const float lp = logf(p), lq = logf(1.f - p);
            y[base + d] = lp - lq;
            acc += -lp - lq;
        }
    }
    if (reverse || logdet == nullptr) return;
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) logdet[blockIdx.x] = red[0] + (float)D * (logf(s) - logf(256.f));
}

int launch_preprocess(const float* x, const float* u, float* y, float* logdet, int B, long D, float alpha, int reverse,
                      cudaStream_t st) {
    if (B == 0) return 0;
    preprocess_kernel<<<B, 256, 0, st>>>(x, u, y, logdet, D, alpha, reverse);
    return (int)cudaGetLastError();
}

}  // namespace finc

// ---------------------------------------------------------------------------------------------
// log|det W| and W^-1 of a batch of small matrices (the Conv1x1 weights of a flow: C = 4 ... 128) in ONE
// launch, one CTA per matrix: Gauss-Jordan with partial pivoting on the augmented [C, 2C] matrix in shared
// memory.  Replaces torch.slogdet (conv1x1.py:22: one cuSOLVER LU + host round trip per layer per forward)
// and torch.inverse (conv1x1.py:36, per reverse call); the inverse is also what the backward needs:
// d log|det W| / dW = W^-T.
// ---------------------------------------------------------------------------------------------
namespace finc {

__global__ void slogdet_inverse_kernel(const float* __restrict__ W, float* __restrict__ logabsdet,
                                       float* __restrict__ Winv, int C) {
    extern __shared__ float sm[];
    const int ld = 2 * C + 1;                 // +1: rows start on different banks
    float* aug = sm;                          // [C][ld]
    float* fac = sm + (size_t)C * ld;         // [C] elimination factors
    __shared__ float s_val[4];
    __shared__ int s_idx[4];
    __shared__ int s_piv;
    const float* w = W + (size_t)blockIdx.x * C * C;
    const int tid = threadIdx.x, nthr = blockDim.x;
    for (int e = tid; e < C * 2 * C; e += nthr) {
        const int r = e / (2 * C), c = e % (2 * C);
        aug[r * ld + c] = c < C ? w[r * C + c] : (c - C == r ? 1.f : 0.f);
    }
    __syncthreads();
    float ldsum = 0.f;
    for (int k = 0; k < C; ++k) {
        // pivot: largest |aug[r][k]| over r >= k (ties: smallest r) -- warp shuffles, then across the warps
        float v = (tid >= k && tid < C) ? fabsf(aug[tid * ld + k]) : -1.f;
        int idx = tid;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, v, o);
            const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
            if (ov > v || (ov == v && oi < idx)) { v = ov; idx = oi; }
        }
        if ((tid & 31) == 0) { s_val[tid >> 5] = v; s_idx[tid >> 5] = idx; }
        __syncthreads();
        if (tid == 0) {
            float bv = s_val[0];
            int bi = s_idx[0];
            for (int wi = 1; wi < (nthr >> 5); ++wi)
                if (s_val[wi] > bv || (s_val[wi] == bv && s_idx[wi] < bi)) { bv = s_val[wi]; bi = s_idx[wi]; }
            s_piv = bi;
        }
        __syncthreads();
        const int p = s_piv;
        if (p != k)
            for (int c = tid; c < 2 * C; c += nthr) {
                const float t = aug[k * ld + c];
                aug[k * ld + c] = aug[p * ld + c];
                aug[p * ld + c] = t;
            }
        __syncthreads();
        const float piv = aug[k * ld + k];
        ldsum += logf(fabsf(piv));
        if (tid < C) fac[tid] = aug[tid * ld + k];
        __syncthreads();
        const float inv = 1.f / piv;
        for (int c = tid; c < 2 * C; c += nthr) {
            const float rk = aug[k * ld + c] * inv;
            for (int r = 0; r < C; ++r)
                if (r != k) aug[r * ld + c] -= fac[r] * rk;
            aug[k * ld + c] = rk;
        }
        __syncthreads();
    }
    if (tid == 0) logabsdet[blockIdx.x] = ldsum;
    float* out = Winv + (size_t)blockIdx.x * C * C;
    for (int e = tid; e < C * C; e += nthr) out[e] = aug[(e / C) * ld + C + e % C];
}

int launch_slogdet_inverse(const float* W, float* logabsdet, float* Winv, int n, int C, cudaStream_t st) {
    if (n == 0) return 0;
    const size_t smem = ((size_t)C * (2 * C + 1) + C) * sizeof(float);
    // the opt-in limit is a function attribute of the device's context: raise it once per device, not per process
    static bool configured[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = -1;
    if (smem > 48 * 1024 && (dev < 0 || !configured[dev])) {
        cudaError_t err = cudaFuncSetAttribute(slogdet_inverse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (err != cudaSuccess) return (int)err;
        if (dev >= 0) configured[dev] = true;
    }
    slogdet_inverse_kernel<<<n, 128, smem, st>>>(W, logabsdet, Winv, C);
    return (int)cudaGetLastError();
}

}  // namespace finc

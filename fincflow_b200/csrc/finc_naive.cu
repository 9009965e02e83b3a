// finc_naive.cu -- generic kernels: any C, kernel size, image size, alignment.
//
// These are the universal fall-back for shapes the tiled kernels do not cover (tiles larger
// than shared memory, exotic kernel sizes) and the on-device cross-check used by the tests
// (FINC_FLAG_NAIVE).  They are still GPU code: there is no CPU fallback anywhere.
#include "finc_common.cuh"

namespace finc {

// one thread per output element, grid-stride.  transpose=false: forward
// (reference layers/conv.py:102-107); transpose=true: backward wrt input.
__global__ void conv_naive_kernel(const float* __restrict__ x, const float* __restrict__ w, float* __restrict__ y,
                                  Shape s, bool transpose) {
    const long HW = (long)s.H * s.W;
    const long total = (long)s.B * s.G * s.C * HW;
    for (long e = blockIdx.x * (long)blockDim.x + threadIdx.x; e < total; e += (long)gridDim.x * blockDim.x) {
        const int ww = (int)(e % s.W);
        const int h = (int)((e / s.W) % s.H);
        const int oc = (int)((e / HW) % s.C);
        const long tile = e / (HW * s.C);  // n*G + g
        const int g = (int)(tile % s.G);
        const int ord = order_of(s.orders, g);
        const float* xt = x + tile * s.C * HW;
        const float* wg = w + (long)g * s.C * s.C * s.kH * s.kW;
        float acc = 0.f;
        for (int ic = 0; ic < s.C; ++ic)
            for (int a = 0; a < s.kH; ++a) {
                const int ro = row_off(ord, a, s.kH);
                const int hh = transpose ? h - ro : h + ro;
                if (hh < 0 || hh >= s.H) continue;
                for (int b = 0; b < s.kW; ++b) {
                    const int co = col_off(ord, b, s.kW);
                    const int wc = transpose ? ww - co : ww + co;
                    if (wc < 0 || wc >= s.W) continue;
                    const float wv = transpose ? wg[((ic * s.C + oc) * s.kH + a) * s.kW + b]
                                               : wg[((oc * s.C + ic) * s.kH + a) * s.kW + b];
                    acc = fmaf(wv, xt[ic * HW + hh * s.W + wc], acc);
                }
            }
        y[e] = acc;
    }
}

// one CTA per tile (n,g); anti-diagonal wavefront with two block barriers per diagonal,
// operating in place on the output in global memory.
// reference: utils/fastflow_cuda_inverse/cinc_cuda_kernel_level2.cu:49-72,98-132.
// ADJ: the adjoint solve of finc_inverse_adjoint_f32 -- the same sweep with `s.orders` flipped by the host, the
// weights w''[o][i][a][b] = w[C-1-i][C-1-o][kH-1-a][kW-1-b] and channel c of the system at channel C-1-c.
template <bool ADJ>
__global__ void inverse_naive_kernel(const float* z, const float* __restrict__ w, float* x, Shape s) {
    const long HW = (long)s.H * s.W;
    const int H = s.H, W = s.W, C = s.C, kH = s.kH, kW = s.kW;
    for (long tile = blockIdx.x; tile < (long)s.B * s.G; tile += gridDim.x) {
        const int g = (int)(tile % s.G);
        const int ord = order_of(s.orders, g);
        const bool bot = ord & 2, right = ord & 1;
        const float* zt = z + tile * C * HW;
        volatile float* xt = x + tile * C * HW;
        const float* wg = w + (long)g * C * C * kH * kW;
        const int ca = corner_a(ord, kH), cb = corner_b(ord, kW);
        auto wt = [&](int o, int i, int a, int b) -> float {
            return ADJ ? wg[(((C - 1 - i) * C + (C - 1 - o)) * kH + (kH - 1 - a)) * kW + (kW - 1 - b)]
                       : wg[((o * C + i) * kH + a) * kW + b];
        };
        auto ch = [&](int c) -> int { return ADJ ? C - 1 - c : c; };
        for (int d = 0; d < H + W - 1; ++d) {
            const int hs_lo = max(0, d - (W - 1));
            const int hs_hi = min(H - 1, d);
            const int npix = hs_hi - hs_lo + 1;
            // phase A: everything except the corner tap (depends on earlier diagonals only)
            for (int it = threadIdx.x; it < npix * C; it += blockDim.x) {
                const int o = it % C;
                const int hs = hs_lo + it / C, ws = d - hs;
                const int h = bot ? H - 1 - hs : hs, ww = right ? W - 1 - ws : ws;
                float acc = zt[ch(o) * HW + h * W + ww];
                for (int k_h = 0; k_h < kH && k_h <= hs; ++k_h) {
                    const int hh = bot ? h + k_h : h - k_h;
                    const int a = bot ? k_h : kH - 1 - k_h;
                    for (int k_w = 0; k_w < kW && k_w <= ws; ++k_w) {
                        if (k_h == 0 && k_w == 0) continue;
                        const int wc = right ? ww + k_w : ww - k_w;
                        const int b = right ? k_w : kW - 1 - k_w;
                        for (int i = 0; i < C; ++i)
                            acc = fmaf(-xt[ch(i) * HW + hh * W + wc], wt(o, i, a, b), acc);
                    }
                }
                xt[ch(o) * HW + h * W + ww] = acc;
            }
            __syncthreads();
            // phase B: channel-triangular corner tap, sequential in o inside one thread
            for (int p = threadIdx.x; p < npix; p += blockDim.x) {
                const int hs = hs_lo + p, ws = d - hs;
                const int h = bot ? H - 1 - hs : hs, ww = right ? W - 1 - ws : ws;
                for (int o = 1; o < C; ++o) {
                    float acc = xt[ch(o) * HW + h * W + ww];
                    for (int i = 0; i < o; ++i)
                        acc = fmaf(-xt[ch(i) * HW + h * W + ww], wt(o, i, ca, cb), acc);
                    xt[ch(o) * HW + h * W + ww] = acc;
                }
            }
            __syncthreads();
        }
    }
}

// one warp per dw element; lanes stride over (n,h,w); shuffle reduction (deterministic).
__global__ void wgrad_naive_kernel(const float* __restrict__ dz, const float* __restrict__ x, float* __restrict__ dw,
                                   Shape s, unsigned flags) {
    const int lane = threadIdx.x & 31;
    const long warp = (blockIdx.x * (long)blockDim.x + threadIdx.x) >> 5;
    const long nwarps = ((long)gridDim.x * blockDim.x) >> 5;
    const long nout = (long)s.G * s.C * s.C * s.kH * s.kW;
    const long HW = (long)s.H * s.W;
    for (long e = warp; e < nout; e += nwarps) {
        const int b = (int)(e % s.kW);
        const int a = (int)((e / s.kW) % s.kH);
        const int i = (int)((e / (s.kW * s.kH)) % s.C);
        const int o = (int)((e / ((long)s.kW * s.kH * s.C)) % s.C);
        const int g = (int)(e / ((long)s.kW * s.kH * s.C * s.C));
        const int ord = order_of(s.orders, g);
        const int ro = row_off(ord, a, s.kH), co = col_off(ord, b, s.kW);
        float acc = 0.f;
        for (long p = lane; p < (long)s.B * HW; p += 32) {
            const int ww = (int)(p % s.W);
            const int h = (int)((p / s.W) % s.H);
            const long n = p / HW;
            const int hh = h + ro, wc = ww + co;
            if (hh < 0 || hh >= s.H || wc < 0 || wc >= s.W) continue;
            acc = fmaf(dz[((n * s.G + g) * s.C + o) * HW + h * s.W + ww], x[((n * s.G + g) * s.C + i) * HW + hh * s.W + wc],
                       acc);
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
        if (lane == 0) {
            const bool masked = !(flags & FINC_FLAG_NO_MASK) && a == corner_a(ord, s.kH) && b == corner_b(ord, s.kW) && i >= o;
            if (masked) acc = 0.f;
            else if (flags & FINC_FLAG_NEGATE) acc = -acc;
            if (flags & FINC_FLAG_ACCUMULATE) acc += dw[e];
            dw[e] = acc;
        }
    }
}

// PaddedConv2d.reset_gradients (layers/conv.py:98-99) without the H2D mask copy.
__global__ void mask_kernel(float* dw, Shape s) {
    const int total = s.G * s.C * s.C;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        const int i = e % s.C, o = (e / s.C) % s.C, g = e / (s.C * s.C);
        if (i < o) continue;
        const int ord = order_of(s.orders, g);
        dw[(((long)g * s.C + o) * s.C + i) * s.kH * s.kW + corner_a(ord, s.kH) * s.kW + corner_b(ord, s.kW)] = 0.f;
    }
}

// logdet[n] = H*W*sum log|diag corner tap|; one CTA, fixed-order reduction.
__global__ void logdet_kernel(const float* __restrict__ w, float* __restrict__ logdet, Shape s, bool accumulate) {
    __shared__ float red[32];
    float acc = 0.f;
    for (int e = threadIdx.x; e < s.G * s.C; e += blockDim.x) {
        const int o = e % s.C, g = e / s.C;
        const int ord = order_of(s.orders, g);
        acc += logf(fabsf(w[(((long)g * s.C + o) * s.C + o) * s.kH * s.kW + corner_a(ord, s.kH) * s.kW + corner_b(ord, s.kW)]));
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    float tot = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += red[i];
    tot *= (float)s.H * (float)s.W;
    for (int n = threadIdx.x; n < s.B; n += blockDim.x) logdet[n] = accumulate ? logdet[n] + tot : tot;
}

// one CTA per image: logp[n] = -0.5*|z_n|^2 - 0.5*D*log(2pi) + logdet[n]; dz = dz_scale*z.
// fixed-order reduction (deterministic).  reference: train/losses.py:17-45, flowsequential.py:41-44
__global__ void gaussian_logp_kernel(const float* __restrict__ z, const float* __restrict__ logdet,
                                     float* __restrict__ logp, float* __restrict__ dz, float dz_scale, int B, long D) {
    __shared__ float red[32];
    for (int n = blockIdx.x; n < B; n += gridDim.x) {
        const float* zn = z + (long)n * D;
        float acc = 0.f;
        for (long d = threadIdx.x; d < D; d += blockDim.x) {
            const float v = zn[d];
            acc = fmaf(v, v, acc);
            if (dz) dz[(long)n * D + d] = dz_scale * v;
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            float tot = 0.f;
            for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += red[i];
            logp[n] = -0.5f * tot - 0.5f * (float)D * 1.8378770664093453f + (logdet ? logdet[n] : 0.f);
        }
        __syncthreads();
    }
}

int launch_gaussian_logp(const float* z, const float* logdet, float* logp, float* dz, float dz_scale, int B, long D,
                         cudaStream_t st) {
    gaussian_logp_kernel<<<B < 148 * 8 ? B : 148 * 8, 256, 0, st>>>(z, logdet, logp, dz, dz_scale, B, D);
    return (int)cudaGetLastError();
}

// space-to-depth / depth-to-space (reference layers/squeeze.py:5-24).  One thread per pair of
// horizontally adjacent un-squeezed pixels: a float2 on the un-squeezed side, two scalars on
// the squeezed side (lanes run along w on both sides -> coalesced).  C, H, W describe the
// UN-squeezed tensor [B, C, H, W]; the squeezed one is [B, 4C, H/2, W/2].
__global__ void squeeze_kernel(const float* __restrict__ src, float* __restrict__ dst, int B, int C, int H, int W,
                               bool inverse) {
    const int W2 = W >> 1, H2 = H >> 1;
    const long total = (long)B * C * H * W2;
    for (long e = blockIdx.x * (long)blockDim.x + threadIdx.x; e < total; e += (long)gridDim.x * blockDim.x) {
        const int j = (int)(e % W2);
        const int hh = (int)((e / W2) % H);
        const long nc = e / ((long)W2 * H);  // n*C + c
        const int c = (int)(nc % C);
        const long n = nc / C;
        const long big = (nc * H + hh) * W + 2 * j;                                   // [n][c][hh][2j]
        const long small0 = (((n * C + c) * 4 + (hh & 1) * 2) * H2 + (hh >> 1)) * W2 + j;  // dw = 0
        const long small1 = small0 + (long)H2 * W2;                                     // dw = 1
        if (!inverse) {
            const float2 v = *reinterpret_cast<const float2*>(src + big);
            dst[small0] = v.x;
            dst[small1] = v.y;
        } else {
            *reinterpret_cast<float2*>(dst + big) = make_float2(src[small0], src[small1]);
        }
    }
}

int launch_squeeze(const float* x, float* y, int B, int C, int H, int W, bool inverse, cudaStream_t st) {
    const long total = (long)B * C * H * (W / 2);
    if (total == 0) return 0;
    const long blocks = (total + 255) / 256;
    squeeze_kernel<<<(unsigned)(blocks > 148L * 32 ? 148L * 32 : blocks), 256, 0, st>>>(x, y, B, C, H, W, inverse);
    return (int)cudaGetLastError();
}

// Adam on a flat buffer; the step counter lives on the device so the launch is graph-replayable.
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, float* step, float lr, float b1, float b2, float eps, long n) {
    const float t = *step + 1.f;
    const float c1 = 1.f - powf(b1, t), c2 = 1.f - powf(b2, t);
    for (long e = blockIdx.x * (long)blockDim.x + threadIdx.x; e < n; e += (long)gridDim.x * blockDim.x) {
        const float ge = g[e];
        const float me = b1 * m[e] + (1.f - b1) * ge;
        const float ve = b2 * v[e] + (1.f - b2) * ge * ge;
        m[e] = me;
        v[e] = ve;
        p[e] -= lr * (me / c1) / (sqrtf(ve / c2) + eps);
    }
    // the counter is bumped by a second tiny kernel (adam_tick_kernel) after all blocks have read it
}
__global__ void adam_tick_kernel(float* step) { *step += 1.f; }

int launch_adam(float* p, const float* g, float* m, float* v, float* step, float lr, float b1, float b2, float eps,
                long n, cudaStream_t st) {
    const long blocks = (n + 255) / 256;
    adam_kernel<<<(unsigned)(blocks > 148L * 8 ? 148L * 8 : blocks), 256, 0, st>>>(p, g, m, v, step, lr, b1, b2, eps, n);
    adam_tick_kernel<<<1, 1, 0, st>>>(step);
    return (int)cudaGetLastError();
}

int launch_conv_naive(const float* x, const float* w, float* y, const Shape& s, bool transpose, cudaStream_t st) {
    const long total = (long)s.B * s.G * s.C * s.H * s.W;
    const int threads = 256;
    const long blocks = (total + threads - 1) / threads;
    conv_naive_kernel<<<(unsigned)(blocks > 148L * 64 ? 148L * 64 : blocks), threads, 0, st>>>(x, w, y, s, transpose);
    return (int)cudaGetLastError();
}

int launch_inverse_naive(const float* z, const float* w, float* x, const Shape& s, cudaStream_t st) {
    const long tiles = (long)s.B * s.G;
    inverse_naive_kernel<false><<<(unsigned)(tiles > 148L * 32 ? 148L * 32 : tiles), 128, 0, st>>>(z, w, x, s);
    return (int)cudaGetLastError();
}

int launch_inverse_adjoint_naive(const float* dx, const float* w, float* dz, const Shape& s, cudaStream_t st) {
    const long tiles = (long)s.B * s.G;
    inverse_naive_kernel<true><<<(unsigned)(tiles > 148L * 32 ? 148L * 32 : tiles), 128, 0, st>>>(dx, w, dz, s);
    return (int)cudaGetLastError();
}

int launch_wgrad_naive(const float* dz, const float* x, float* dw, const Shape& s, unsigned flags, cudaStream_t st) {
    const long nout = (long)s.G * s.C * s.C * s.kH * s.kW;
    const int threads = 256;
    const long blocks = (nout * 32 + threads - 1) / threads;
    wgrad_naive_kernel<<<(unsigned)(blocks > 148L * 32 ? 148L * 32 : blocks), threads, 0, st>>>(dz, x, dw, s, flags);
    return (int)cudaGetLastError();
}

int launch_mask(float* dw, const Shape& s, cudaStream_t st) {
    const int total = s.G * s.C * s.C;
    mask_kernel<<<(total + 255) / 256, 256, 0, st>>>(dw, s);
    return (int)cudaGetLastError();
}

int launch_logdet(const float* w, float* logdet, bool accumulate, const Shape& s, cudaStream_t st) {
    logdet_kernel<<<1, 256, 0, st>>>(w, logdet, s, accumulate);
    return (int)cudaGetLastError();
}

}  // namespace finc

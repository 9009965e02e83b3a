/*
 * finc_oracle_impl.h -- type-generic body of the CPU oracle (TEST INFRASTRUCTURE ONLY).
 *
 * Included twice by finc_oracle.c with
 *     REAL   = float  / double      (storage + accumulation type)
 *     SUFFIX = f32    / f64
 *
 * Every function restates one piece of the reference's algorithm for the FInC
 * hot path in the *stored* weight orientation (no flips), citing the reference
 * file:line it follows (paths relative to the reference checkout).
 *
 * Layout everywhere: contiguous NCHW.  A tensor is [B, G*C, H, W]; group g owns
 * channels [g*C, (g+1)*C) and has its own weight [C, C, kH, kW] (OIHW) and its
 * own padding order orders[g] in {0:TL, 1:TR, 2:BL, 3:BR}
 * (bit0 = padded on the right, bit1 = padded at the bottom).
 * A reference PaddedConv2d is G=1; a reference FastFlowUnit is G=4 with
 * orders (TL,TR,BL,BR)  (fastflow/fastflow.py:24-27,32-48).
 */

#define CAT_(a, b) a##_##b
#define CAT(a, b) CAT_(a, b)
#define FN(name) CAT(name, SUFFIX)

/* Row / column offset of tap (a,b) relative to the output pixel.
 * fastflow/layers/conv.py:41-55: F.pad(left,right,top,bottom) followed by a
 * valid cross-correlation, so tap a reads padded row h+a = original row
 * h + a - pad_top. */
static inline int FN(row_off)(int order, int a, int kH) { return (order & 2) ? a : a - (kH - 1); }
static inline int FN(col_off)(int order, int b, int kW) { return (order & 1) ? b : b - (kW - 1); }

/* ---------------------------------------------------------------------------
 * forward:  z[n,o,h,w] = sum_{i,a,b} Ws[o,i,a,b] * x[n,i,h+r(a),w+c(b)]
 * fastflow/layers/conv.py:102-107 (F.pad + nn.Conv2d, bias=False, raw weight);
 * fastflow/fastflow.py:31-50 (chunk into 4, TL/TR/BL/BR, cat).
 * ------------------------------------------------------------------------- */
void FN(finc_oracle_forward)(const REAL* x, const REAL* w, REAL* z, int B, int G, int C, int H,
                             int W, int kH, int kW, const int* orders) {
    const long HW = (long)H * W;
#pragma omp parallel for collapse(2) schedule(static)
    for (int n = 0; n < B; ++n)
        for (int g = 0; g < G; ++g) {
            const int ord = orders[g];
            const REAL* xg = x + ((long)n * G + g) * C * HW;
            REAL* zg = z + ((long)n * G + g) * C * HW;
            const REAL* wg = w + (long)g * C * C * kH * kW;
            for (int o = 0; o < C; ++o)
                for (int h = 0; h < H; ++h)
                    for (int ww = 0; ww < W; ++ww) {
                        REAL acc = 0;
                        for (int i = 0; i < C; ++i)
                            for (int a = 0; a < kH; ++a) {
                                const int hh = h + FN(row_off)(ord, a, kH);
                                if (hh < 0 || hh >= H) continue;
                                for (int b = 0; b < kW; ++b) {
                                    const int wc = ww + FN(col_off)(ord, b, kW);
                                    if (wc < 0 || wc >= W) continue;
                                    acc += wg[((o * C + i) * kH + a) * kW + b] * xg[i * HW + hh * W + wc];
                                }
                            }
                        zg[o * HW + h * W + ww] = acc;
                    }
        }
}

/* ---------------------------------------------------------------------------
 * backward wrt input (what autograd/cuDNN dgrad computes for conv.py:102-105):
 *   dx[n,i,p,q] = sum_{o,a,b} Ws[o,i,a,b] * dz[n,o,p-r(a),q-c(b)]
 * ------------------------------------------------------------------------- */
void FN(finc_oracle_backward_input)(const REAL* dz, const REAL* w, REAL* dx, int B, int G, int C,
                                    int H, int W, int kH, int kW, const int* orders) {
    const long HW = (long)H * W;
#pragma omp parallel for collapse(2) schedule(static)
    for (int n = 0; n < B; ++n)
        for (int g = 0; g < G; ++g) {
            const int ord = orders[g];
            const REAL* dzg = dz + ((long)n * G + g) * C * HW;
            REAL* dxg = dx + ((long)n * G + g) * C * HW;
            const REAL* wg = w + (long)g * C * C * kH * kW;
            for (int i = 0; i < C; ++i)
                for (int p = 0; p < H; ++p)
                    for (int q = 0; q < W; ++q) {
                        REAL acc = 0;
                        for (int o = 0; o < C; ++o)
                            for (int a = 0; a < kH; ++a) {
                                const int hh = p - FN(row_off)(ord, a, kH);
                                if (hh < 0 || hh >= H) continue;
                                for (int b = 0; b < kW; ++b) {
                                    const int wc = q - FN(col_off)(ord, b, kW);
                                    if (wc < 0 || wc >= W) continue;
                                    acc += wg[((o * C + i) * kH + a) * kW + b] * dzg[o * HW + hh * W + wc];
                                }
                            }
                        dxg[i * HW + p * W + q] = acc;
                    }
        }
}

/* ---------------------------------------------------------------------------
 * backward wrt weight (cuDNN wgrad for conv.py:102-105) followed, when
 * apply_mask != 0, by PaddedConv2d.reset_gradients (conv.py:81-99):
 *   dw[o,i,a,b] = sum_{n,h,w} dz[n,o,h,w] * x[n,i,h+r(a),w+c(b)]
 *   dw[o,i,a*,b*] = 0 for i >= o        (corner tap (a*,b*) of the order)
 * ------------------------------------------------------------------------- */
void FN(finc_oracle_backward_weight)(const REAL* dz, const REAL* x, REAL* dw, int B, int G, int C,
                                     int H, int W, int kH, int kW, const int* orders,
                                     int apply_mask) {
    const long HW = (long)H * W;
#pragma omp parallel for collapse(2) schedule(static)
    for (int g = 0; g < G; ++g)
        for (int o = 0; o < C; ++o) {
            const int ord = orders[g];
            const int ca = (ord & 2) ? 0 : kH - 1;
            const int cb = (ord & 1) ? 0 : kW - 1;
            for (int i = 0; i < C; ++i)
                for (int a = 0; a < kH; ++a)
                    for (int b = 0; b < kW; ++b) {
                        double acc = 0; /* long reduction: always accumulate wide */
                        const int ro = FN(row_off)(ord, a, kH), co = FN(col_off)(ord, b, kW);
                        for (int n = 0; n < B; ++n) {
                            const REAL* dzo = dz + (((long)n * G + g) * C + o) * HW;
                            const REAL* xi = x + (((long)n * G + g) * C + i) * HW;
                            for (int h = 0; h < H; ++h) {
                                const int hh = h + ro;
                                if (hh < 0 || hh >= H) continue;
                                for (int ww = 0; ww < W; ++ww) {
                                    const int wc = ww + co;
                                    if (wc < 0 || wc >= W) continue;
                                    acc += (double)dzo[h * W + ww] * (double)xi[hh * W + wc];
                                }
                            }
                        }
                        if (apply_mask && a == ca && b == cb && i >= o) acc = 0;
                        dw[(((long)g * C + o) * C + i) * kH * kW + a * kW + b] = (REAL)acc;
                    }
        }
}

/* mask only: PaddedConv2d.get_mask / reset_gradients, conv.py:81-99 */
void FN(finc_oracle_apply_grad_mask)(REAL* dw, int G, int C, int kH, int kW, const int* orders) {
    for (int g = 0; g < G; ++g) {
        const int ca = (orders[g] & 2) ? 0 : kH - 1;
        const int cb = (orders[g] & 1) ? 0 : kW - 1;
        for (int o = 0; o < C; ++o)
            for (int i = o; i < C; ++i) dw[(((long)g * C + o) * C + i) * kH * kW + ca * kW + cb] = 0;
    }
}

/* ---------------------------------------------------------------------------
 * inverse (sampling direction).  Restates, without the activation/weight flips,
 *   fastflow/utils/fastflow_inverse/solve_parallel_mc.pyx:100-124 (Cython, f64),
 *   fastflow/utils/solve_mc.py:88-114 (raster-order python `solve`),
 *   fastflow/utils/fastflow_cuda_inverse/cinc_cuda_kernel_level2.cu:57-70 (CUDA):
 *
 *   y = z; for every pixel in sweep order, channel c = 0..C-1:
 *     for k_h, for k_w, for k_c   (in this order, sequential in-place subtraction)
 *        skip (k_h,k_w,k_c) == (0,0,c);  at (0,0) stop at k_c > c
 *        y[c,h,w] -= y[k_c, h -/+ k_h, w -/+ k_w] * Wtl[c,k_c,kH-1-k_h,kW-1-k_w]
 *
 * The reference brings TR/BL/BR to TL form by flipping activations and weights
 * (fastflow/fastflow.py:79-99, layers/conv.py:118-157); here the flips are
 * folded into the index map: sweep coordinate h' = h (top padded) or H-1-h,
 * and Wtl[c,kc,kH-1-k_h,kW-1-k_w] == Ws[c,kc,a,b] with a = kH-1-k_h (top padded)
 * or k_h, b likewise.  Raster order over (h',w') satisfies the same dependencies
 * as the anti-diagonal order; per element the subtraction order is identical,
 * so the result is bit-identical to the wavefront order in the same precision.
 * No division: the unit diagonal is assumed exactly as in the reference.
 * ------------------------------------------------------------------------- */
void FN(finc_oracle_inverse)(const REAL* z, const REAL* w, REAL* y, int B, int G, int C, int H,
                             int W, int kH, int kW, const int* orders) {
    const long HW = (long)H * W;
#pragma omp parallel for collapse(2) schedule(static)
    for (int n = 0; n < B; ++n)
        for (int g = 0; g < G; ++g) {
            const int ord = orders[g];
            const int bot = (ord & 2) != 0, right = (ord & 1) != 0;
            const REAL* zg = z + ((long)n * G + g) * C * HW;
            REAL* yg = y + ((long)n * G + g) * C * HW;
            const REAL* wg = w + (long)g * C * C * kH * kW;
            for (long e = 0; e < C * HW; ++e) yg[e] = zg[e];
            for (int hs = 0; hs < H; ++hs)
                for (int ws = 0; ws < W; ++ws) {
                    const int h = bot ? H - 1 - hs : hs;
                    const int ww = right ? W - 1 - ws : ws;
                    for (int c = 0; c < C; ++c) {
                        REAL acc = yg[c * HW + h * W + ww];
                        for (int k_h = 0; k_h < kH; ++k_h) {
                            if (hs - k_h < 0) break;
                            const int hh = bot ? h + k_h : h - k_h;
                            const int a = bot ? k_h : kH - 1 - k_h;
                            for (int k_w = 0; k_w < kW; ++k_w) {
                                if (ws - k_w < 0) break;
                                const int wc = right ? ww + k_w : ww - k_w;
                                const int b = right ? k_w : kW - 1 - k_w;
                                for (int k_c = 0; k_c < C; ++k_c) {
                                    if (k_h == 0 && k_w == 0) {
                                        if (k_c == c) continue;
                                        if (c - k_c < 0) break;
                                    }
                                    acc -= yg[k_c * HW + hh * W + wc] *
                                           wg[((c * C + k_c) * kH + a) * kW + b];
                                }
                            }
                        }
                        yg[c * HW + h * W + ww] = acc;
                    }
                }
        }
}

/* logdet[n] = H*W * sum_g sum_o log|Ws_g[o,o,a*,b*]|.  The reference returns the
 * python float 0.0 (conv.py:106, :220-221) because init + gradient mask keep the
 * corner diagonal at exactly 1; this is the general formula (SURVEY.md App. A). */
double FN(finc_oracle_logdet)(const REAL* w, int G, int C, int H, int W, int kH, int kW,
                              const int* orders) {
    double s = 0;
    for (int g = 0; g < G; ++g) {
        const int ca = (orders[g] & 2) ? 0 : kH - 1;
        const int cb = (orders[g] & 1) ? 0 : kW - 1;
        for (int o = 0; o < C; ++o)
            s += log(fabs((double)w[(((long)g * C + o) * C + o) * kH * kW + ca * kW + cb]));
    }
    return s * (double)H * (double)W;
}

#undef FN
#undef CAT
#undef CAT_

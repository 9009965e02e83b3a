/*
 * fincflow_b200.h -- C ABI of the B200-native FInC invertible k x k convolution hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types.  Every entry
 * point names the reference interface it replaces (paths relative to the reference repo
 * aditya-v-kallappa/FInCFlow).  The reference's native interface for this path is a
 * JIT-built pybind11 module with one function
 *     inverse(input[B,4Cq,H,W], kernel[4Cq,Cq,kH,kW], output zero-filled) -> [output]
 * (fastflow/utils/fastflow_cuda_inverse/cinc_cuda_level2.cpp:19-32, call site
 * fastflow/fastflow.py:91-92); forward / backward go through F.pad + nn.Conv2d (cuDNN)
 * (fastflow/layers/conv.py:102-107).  All of those are covered here.
 *
 * Conventions
 *   - fp32, contiguous NCHW device memory.  A tensor is [B, G*C, H, W]: G independent
 *     groups of C channels.  A reference PaddedConv2d is G = 1; a FastFlowUnit is G = 4
 *     with orders (TL, TR, BL, BR) on its four channel quarters (fastflow/fastflow.py:24-48).
 *   - weights are [G*C, C, kH, kW] = the G PaddedConv2d `conv.weight` tensors concatenated
 *     on dim 0, each in its STORED orientation (already flipped for TR/BL/BR by
 *     layers/conv.py:72-79).  No host-side flips are ever needed.
 *   - `orders` packs 2 bits per group, group g at bits [2g, 2g+2):
 *     bit0 = padded on the right, bit1 = padded at the bottom
 *     (TL = 0, TR = 1, BL = 2, BR = 3; layers/conv.py:41-55).  G <= 16.
 *     FINC_ORDERS_UNIT is the FastFlowUnit packing.
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = the
 *     legacy default stream) of the calling thread's current CUDA device, allocates
 *     nothing, keeps no state between calls, and returns 0 or a negative FINC_E_* code /
 *     positive cudaError_t.  It never throws.
 *   - outputs must not alias inputs, except finc_inverse_f32 where x == z is allowed and
 *     finc_inverse_adjoint_f32 where dz == dx is allowed.
 */
#ifndef FINCFLOW_B200_H_
#define FINCFLOW_B200_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FINC_ABI_VERSION 1

#define FINC_ORDER_TL 0u
#define FINC_ORDER_TR 1u
#define FINC_ORDER_BL 2u
#define FINC_ORDER_BR 3u
#define FINC_ORDERS_UNIT 0xE4u /* TL | TR<<2 | BL<<4 | BR<<6 */

/* flags */
#define FINC_FLAG_NAIVE 1u        /* force the generic one-thread-per-output kernels (testing) */
#define FINC_FLAG_NO_MASK 2u      /* backward_weight: do NOT apply the FInC gradient mask */
#define FINC_FLAG_ACCUMULATE 4u   /* backward_weight: dw += result instead of dw = result */
#define FINC_FLAG_GENERIC_TILED 16u /* inverse: skip the shape-specialised kernel, use the generic tiled one (testing) */
#define FINC_FLAG_WORKSPACE_CLEAN 32u /* backward_weight: the first 4 KiB of `workspace` are zero (as every call leaves them) */
#define FINC_FLAG_PREPARED 64u /* forward / backward_input / inverse: `w` is a table made by finc_prepare_weights_f32 */
#define FINC_FLAG_QUARTER_GPU 128u /* backward_weight: plan for a quarter of the SMs (several independent launches run side by side on different streams) */
#define FINC_FLAG_HALF_GPU 256u /* forward / backward_input: use at most half of the SMs (leaves room for concurrent launches on other streams) */
#define FINC_FLAG_WAVE_SMEM 512u /* inverse: skip the register-window kernel, use the shared-memory wavefront kernel (testing) */
#define FINC_FLAG_LOGDET_ACCUMULATE 8u /* forward: logdet[n] += ... (FlowSequential's `logdet += layer_logdet`) */
#define FINC_FLAG_TF32_1PASS 1024u /* tensor-core entry points: single-pass TF32 products (PyTorch's default conv precision, ~5e-4) instead of the fp32-accurate 3xTF32 split */
#define FINC_FLAG_CHAIN_TRANSPOSE 2048u /* finc_chain_f32: backward-data chain (transposed weights, opposite corner) */
#define FINC_FLAG_NEGATE 4096u /* backward_weight (and _batched): dw = -result (dw += -result with FINC_FLAG_ACCUMULATE); masked entries stay +0 */
#define FINC_FLAG_COUPLING_REVERSE 8192u /* finc_coupling_backward_f32: the backward of the reverse direction (finc_coupling_apply_f32 with reverse = 1) */

/* error codes (negative); positive return values are cudaError_t */
#define FINC_OK 0
#define FINC_E_BADARG (-1)     /* null pointer, non-positive dimension, G > 16, ... */
#define FINC_E_WORKSPACE (-2)  /* workspace too small */
#define FINC_E_UNSUPPORTED (-3)

int finc_abi_version(void);
const char* finc_error_string(int code);

/* Bind the library's CUDA runtime to `device` for the calling thread (call once after
 * selecting the device in the host framework, e.g. after torch.cuda.set_device). */
int finc_set_device(int device);
/* Number of SMs of the current device (148 on B200); <0 on error. */
int finc_sm_count(void);

/* z[n, gC+o, h, w] = sum_{i,a,b} w[gC+o, i, a, b] * x[n, gC+i, h+r_g(a), w+c_g(b)]
 * and, when logdet != NULL, logdet[n] = H*W * sum_g sum_o log|w[gC+o, o, a*_g, b*_g]|
 * for n < B (the reference returns the python float 0.0 because that diagonal is 1).
 * Replaces PaddedConv2d.forward (layers/conv.py:102-107: F.pad + cuDNN conv) and
 * FastFlowUnit.forward (fastflow/fastflow.py:31-50: chunk, 4 pads, 4 convs, cat). */
int finc_forward_f32(const float* x, const float* w, float* z, float* logdet,
                     int B, int G, int C, int H, int W, int kH, int kW,
                     unsigned orders, unsigned flags, void* stream);

/* dx[n, gC+i, p, q] = sum_{o,a,b} w[gC+o, i, a, b] * dz[n, gC+o, p-r_g(a), q-c_g(b)]
 * Replaces the cuDNN dgrad autograd runs for layers/conv.py:102-105 (plus the
 * pad/chunk/cat backward slices of fastflow/fastflow.py:31-50). */
int finc_backward_input_f32(const float* dz, const float* w, float* dx,
                            int B, int G, int C, int H, int W, int kH, int kW,
                            unsigned orders, unsigned flags, void* stream);

/* dw[gC+o, i, a, b] = sum_{n,h,w} dz[n, gC+o, h, w] * x[n, gC+i, h+r_g(a), w+c_g(b)]
 * then (unless FINC_FLAG_NO_MASK) dw[gC+o, i, a*_g, b*_g] = 0 for i >= o.
 * Replaces cuDNN wgrad + PaddedConv2d.reset_gradients / clear_grad
 * (layers/conv.py:81-99, train/experiment.py:16-18,250).  `dw` may point into a flat
 * gradient bucket.  `workspace` must hold finc_backward_weight_workspace_bytes(...)
 * bytes of device memory.  Its first 4 KiB are ticket counters: they are cleared by the call
 * (one memset node) unless FINC_FLAG_WORKSPACE_CLEAN promises they are already zero; every
 * successful call leaves them zero, so a workspace zeroed once can be reused with the flag.
 * Calls sharing a workspace must be stream-ordered. */
size_t finc_backward_weight_workspace_bytes(int B, int G, int C, int H, int W, int kH, int kW);  /* valid for any flags */
int finc_backward_weight_f32(const float* dz, const float* x, float* dw,
                             void* workspace, size_t workspace_bytes,
                             int B, int G, int C, int H, int W, int kH, int kW,
                             unsigned orders, unsigned flags, void* stream);

/* Solve forward(x) = z for x by anti-diagonal wavefront substitution, all groups in one
 * launch, unit diagonal assumed (no division), `x` need not be zero-filled:
 *   x[n,o,h,w] = z[n,o,h,w] - sum_{(a,b)!=(a*,b*), i} w[o,i,a,b] x[n,i,h+r(a),w+c(b)]
 *                           - sum_{i<o} w[o,i,a*,b*] x[n,i,h,w]
 * Replaces cinc_cuda_level2.inverse / FastFlowUnit.reverse_level2 including its six
 * flips, three cats and zeros_like (fastflow/fastflow.py:78-100,
 * utils/fastflow_cuda_inverse/cinc_cuda_kernel_level2.cu:14-136: (H+W-1)*Cq launches each
 * followed by cudaDeviceSynchronize), cinc_cuda_level1.inverse / PaddedConv2d.reverse_cuda
 * (cinc_cuda_kernel_level1.cu:14-131, layers/conv.py:191-218) and the Cython CPU solver
 * behind PaddedConv2d.reverse (layers/conv.py:109-163, solve_parallel_mc.pyx:77-126). */
int finc_inverse_f32(const float* z, const float* w, float* x,
                     int B, int G, int C, int H, int W, int kH, int kW,
                     unsigned orders, unsigned flags, void* stream);

/* The exact adjoint (transpose) of finc_inverse_f32 -- the input gradient of the sampling direction: with
 * A the map finc_inverse_f32 inverts (x = A^-1 z), dz = A^-T dx, i.e. <dx, inverse(z)> = <adjoint(dx), z> for all z.
 * Equivalently finc_backward_input_f32(dz) == dx.  With autograd this gives, for x = inverse(z; w) and an upstream
 * gradient dx:  dL/dz = dz  and  dL/dw = -(finc_backward_weight_f32(dz, x), masked), i.e. one call of
 * finc_backward_weight_f32 with FINC_FLAG_NEGATE (the inverse never reads w[o, i>=o, a*, b*], so their derivative
 * is 0 whatever the mask setting of the forward layer).
 * It is a FInC inverse in its own right, swept from the opposite corner of every group; one launch, same kernels and
 * cost as finc_inverse_f32 of the same shape (register-window kernel where that covers the shape, the generic
 * kernel otherwise).  Arguments as finc_inverse_f32; dz == dx is allowed; B = 0 is a no-op.  flags: FINC_FLAG_NAIVE
 * forces the generic kernel (testing); FINC_FLAG_PREPARED is not supported (FINC_E_UNSUPPORTED). */
int finc_inverse_adjoint_f32(const float* dx, const float* w, float* dz,
                             int B, int G, int C, int H, int W, int kH, int kW,
                             unsigned orders, unsigned flags, void* stream);

/* dw[gC+o, i, a*_g, b*_g] = 0 for i >= o.  Replaces PaddedConv2d.reset_gradients
 * (layers/conv.py:98-99: H2D copy of the CPU mask + multiply). */
int finc_apply_grad_mask_f32(float* dw, int G, int C, int kH, int kW,
                             unsigned orders, void* stream);

/* logdet[n] = H*W * sum_g sum_o log|w[gC+o, o, a*_g, b*_g]|, n < B.
 * Replaces PaddedConv2d.logdet (layers/conv.py:220-221, constant 0.0). */
int finc_logdet_f32(const float* w, float* logdet, int B, int G, int C, int H, int W,
                    int kH, int kW, unsigned orders, void* stream);

/* Standard-normal base distribution of a flow that ends in FInC layers:
 *   logp[n]  = -0.5*sum_d z[n,d]^2 - 0.5*D*log(2*pi) + (logdet ? logdet[n] : 0)
 *   dz[n,d]  = dz_scale * z[n,d]            (when dz != NULL; d(-mean logp)/dz with dz_scale = 1/B)
 * Replaces NegativeGaussianLoss.log_prob (train/losses.py:17-45: MultivariateNormal with a dense
 * D x D identity on cuda:0) + `logprob + logdet` (layers/flowsequential.py:41-44) and the autograd
 * backward of that sum.  z is [B, D] contiguous. */
int finc_gaussian_logp_f32(const float* z, const float* logdet, float* logp, float* dz, float dz_scale,
                           int B, long D, void* stream);

/* Adam update of a flat fp32 parameter buffer in one launch (the optimiser step that follows the
 * masked FInC gradients; reference scripts: torch.optim.Adam, fastflow_imagenet_multi_gpu.py:463):
 *   m = b1*m + (1-b1)*g;  v = b2*v + (1-b2)*g*g;  p -= lr * (m/(1-b1^t)) / (sqrt(v/(1-b2^t)) + eps)
 * `step` is a device counter (float, incremented by the kernel) so the launch can be replayed
 * inside a CUDA graph. */
int finc_adam_step_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, float* step,
                       float lr, float beta1, float beta2, float eps, long n, void* stream);

/* Fused gradient all-reduce + Adam over NVLink peer memory (multi-GPU training only).
 * peer_grad / peer_signal: DEVICE arrays of `world` pointers to every rank's gradient bucket and
 * signal pad (>= 128 bytes each, zero-initialised once) -- symmetric allocations, e.g.
 * torch.distributed._symmetric_memory (buffer_ptrs_dev / signal_pad_ptrs_dev).  `local` is a
 * zero-initialised 16-byte device scratch of this rank.  Every rank must launch the call once per
 * step; the kernel waits for all peers, sums the buckets in rank order (bit-identical parameters
 * on every rank), scales by grad_scale and applies Adam to this rank's replica.  world <= 16.
 * Replaces DataParallel's reduce-to-GPU0 + broadcast (fastflow_cifar_multi_gpu.py:439-440). */
int finc_allreduce_adam_f32(const void* peer_grad, const void* peer_signal, void* local,
                            float* param, float* exp_avg, float* exp_avg_sq, float* step,
                            float lr, float beta1, float beta2, float eps, float grad_scale,
                            long n, int rank, int world, void* stream);

/* Squeeze (space-to-depth) and its inverse, the glue between the levels of the multi-scale flow:
 *   squeeze:   y[n, 4c + 2dh + dw, h, w] = x[n, c, 2h + dh, 2w + dw]      x: [B,C,H,W] -> y: [B,4C,H/2,W/2]
 *   unsqueeze: the inverse map                                           x: [B,4C,H,W] -> y: [B,C,2H,2W]
 * Replaces space_to_depth / depth_to_space (layers/squeeze.py:5-24: view + permute + contiguous).
 * H and W of the un-squeezed tensor must be even.  One HBM round trip, coalesced both ways. */
int finc_squeeze_f32(const float* x, float* y, int B, int C, int H, int W, void* stream);
int finc_unsqueeze_f32(const float* x, float* y, int B, int C4, int H, int W, void* stream);

/* log|det W_i| and W_i^-1 for a batch of n small matrices [n, C, C] (C <= 128) in one launch (Gauss-Jordan with
 * partial pivoting, one CTA per matrix).  Replaces `torch.slogdet(self.W)` in Conv1x1.forward and
 * `torch.inverse(self.W)` in Conv1x1.reverse (layers/conv1x1.py:22,36: a cuSOLVER call with a host round trip per
 * layer per call); W^-1 is also the gradient of the log-determinant: d log|det W| / dW = W^-T. */
int finc_slogdet_inverse_f32(const float* W, float* logabsdet, float* Winv, int n, int C, void* stream);

/* Input preprocessing of the image flows, forward and reverse, in one pass (x, y: [B, D] contiguous):
 *   forward: p = ((x + noise) / 256 + alpha) * (1 - 2 alpha);  y = log p - log(1 - p)
 *            logdet[n] = D * (log(1 - 2 alpha) - log 256) + sum_d (-log p - log(1 - p))   (logdet may be NULL)
 *   reverse: y = floor((sigmoid(x) / (1 - 2 alpha) - alpha) * 256)
 * `noise` = the dequantisation noise u ~ U[0,1) drawn by the caller (NULL = 0).  Replaces the four
 * layers of Preprocess (fastflow_cifar_multi_gpu.py:162-186: layers/dequantize.py:13-19,
 * layers/normalize.py:18-31 twice, layers/transforms.py:11-18) and their logdet adds. */
int finc_preprocess_f32(const float* x, const float* noise, float* y, float* logdet, int B, long D, float alpha,
                        int reverse, void* stream);

/* Per-pixel affine map over the channel axis, x and y [B, C, HW] contiguous (NCHW with HW = H*W):
 *   y[n, o, p] = sum_i A[o, i] * x[n, i, p] + (bias ? bias[o] : 0)           A: [C, C] row-major
 * One pass for the glue that follows every FastFlowUnit in the reference's flow step
 * (fastflow_cifar_multi_gpu.py:188-236): ActNorm (layers/actnorm.py:14-52) then Conv1x1
 * (layers/conv1x1.py:18-43) compose to A = W diag(exp(-log_scale)), bias = -A translation; their
 * reverse is A^-1 with bias = translation (instead of torch.inverse + conv2d per call), and the
 * backward-data pass is A^T without bias.  x != y. */
int finc_affine1x1_f32(const float* x, const float* A, const float* bias, float* y,
                       int B, int C, long HW, void* stream);

/* Weight gradient of finc_affine1x1_f32 (deterministic, no floating-point atomics):
 *   dA[o, i] = sum_{n,p} dy[n, o, p] * x[n, i, p]        dbias[o] = sum_{n,p} dy[n, o, p]   (dbias may be NULL)
 * From these the host gets dW = dA diag(exp(-log_s)), dlog_s and dtranslation by the chain rule
 * (autograd of ActNorm + Conv1x1, layers/actnorm.py:14-52, layers/conv1x1.py:18-43).  `workspace` must
 * hold finc_affine1x1_backward_weight_workspace_bytes(B, C, HW) bytes of device memory. */
size_t finc_affine1x1_backward_weight_workspace_bytes(int B, int C, long HW);
int finc_affine1x1_backward_weight_f32(const float* dy, const float* x, float* dA, float* dbias,
                                       void* workspace, size_t workspace_bytes,
                                       int B, int C, long HW, void* stream);

/* Prepared weight tables (optional fast path for fixed shapes, e.g. CUDA-graph replays).
 * The tiled kernels need the weights transposed / sweep-ordered in shared memory; by default
 * every launch re-stages them from the raw [G*C, C, kH, kW] tensor (~1-2 us).  A table prepared
 * once per weight update is instead fetched with a single TMA bulk copy.
 *   kind: FINC_PREP_FORWARD | FINC_PREP_BACKWARD_INPUT | FINC_PREP_INVERSE
 *   finc_prepared_weights_bytes: size of ONE unit's table for this kind and shape, 0 if the shape
 *     is not covered by the tiled kernels (then FINC_FLAG_PREPARED must not be used).
 *   finc_prepare_weights_f32: builds `n_units` tables in one launch; unit u reads
 *     w + u*w_stride_floats and writes prepared + u*prepared_stride_bytes.
 * A table is valid for exactly the (kind, B, G, C, H, W, kH, kW, orders) it was prepared for -- the SAME batch size
 * B included: the forward / backward-input layout depends on the launch plan chosen for B -- and until the weights
 * change.  The kernels check the table header (magic, kind, layout parameters) and trap on a mismatch.  Pass it as `w` together with FINC_FLAG_PREPARED (the forward table
 * carries the unit's logdet, so `logdet` output keeps working). */
#define FINC_PREP_FORWARD 0
#define FINC_PREP_BACKWARD_INPUT 1
#define FINC_PREP_INVERSE 2
size_t finc_prepared_weights_bytes(int kind, int B, int G, int C, int H, int W, int kH, int kW);
int finc_prepare_weights_f32(const float* w, void* prepared, int kind, int n_units,
                             size_t w_stride_floats, size_t prepared_stride_bytes,
                             int B, int G, int C, int H, int W, int kH, int kW,
                             unsigned orders, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Tensor-core path (tcgen05.mma kind::tf32, accumulators in TMEM, TMA tensor maps).
 *
 * Channels-last convolution  y[b,h,w,n] = act(sum_{tap,c} x[b, h+dy, w+dx, c] * Wt[tap][n][c] + bias[n])
 * for taps = 1 (1x1) or 9 (3x3, zero padding 1).  x is [B,H,W,Cin_pad] and y [B,H,W,Npad] fp32 with
 * Cin_pad % 32 == 0 and Npad % 32 == 0 (pad channels are zero).  Products are 3xTF32
 * (a_hi*b_hi + a_lo*b_hi + a_hi*b_lo, fp32-accurate) unless FINC_FLAG_TF32_1PASS.  `relu_mask`
 * (channels-last [B,H,W,Npad], may be NULL) zeroes outputs where mask <= 0 (ReLU backward).
 * Weights are prepared once per update by finc_tc_conv_prepare_weights_f32:
 *   mode 0: w = OIHW [N, Cin, kh, kw]                      -> rows n (padded to 32), K = Cin (padded to 32)
 *   mode 1: im2col form of a 3x3 conv: one tap, K = 9*Cin  (pairs with a [B,H,W,9*Cin] patch tensor)
 *   mode 2: transposed + flipped (the backward-data convolution): rows = Cin, K = N
 * Replaces the nn.Conv2d (cuDNN) calls of the Coupling network, fastflow/layers/coupling.py:56-66. */
size_t finc_tc_conv_weights_bytes(int N, int Cin, int taps, int mode);
int finc_tc_conv_prepare_weights_f32(const float* w, void* prepared, int N, int Cin, int taps, int mode, void* stream);
int finc_tc_conv_nhwc_f32(const float* x, const void* prepared, const float* bias, const float* relu_mask, float* y,
                          int B, int H, int W, int Cin_pad, int Npad, int taps, int relu, unsigned flags, void* stream);

/* Weight-gradient GEMM on the tensor cores (reduction over pixels, deterministic split-K):
 *   dW[m, n] (+)= sum_p P[p, m] * Q[p, n]     P: [np, ldP], Q: [np, ldQ] channels-last fp32, dW: [M, ld_dW]
 * P = gradient at a convolution's output, Q = its (im2col-form) input.  N must be a multiple of 64
 * (128 / 160 preferred), ldP and ldQ multiples of 4; FINC_FLAG_ACCUMULATE adds into dW,
 * FINC_FLAG_TF32_1PASS selects single-pass TF32.  Replaces the cuDNN wgrad autograd runs for the
 * Coupling network's nn.Conv2d layers (fastflow/layers/coupling.py:56-66). */
size_t finc_tc_wgrad_workspace_bytes(long np, int M, int N);
int finc_tc_wgrad_f32(const float* P, const float* Q, float* dW, void* workspace, size_t workspace_bytes,
                      long np, int M, int N, int ldP, int ldQ, int ld_dW, unsigned flags, void* stream);

/* Affine coupling layer (fastflow/layers/coupling.py:44-105) in four launches:
 *   h = Conv2dZero(relu(conv1x1(relu(conv3x3(x[:, :C/2])))));  log_s = 2 tanh(h[:, ::2] / 2);  t = h[:, 1::2]
 *   forward:  y = cat(x1, x2 * exp(log_s) + t),   logdet[n] (+)= sum log_s        (Coupling.forward)
 *   reverse:  y = cat(x1, (x2 - t) * exp(-log_s)), logdet[n] (+)= -sum log_s      (Coupling.reverse)
 * `logdet` (nullable, [B]) is log|det dy/dx| of the direction that runs: with reverse = 1 it is minus the forward's
 * log-det at the reconstructed input (the log-density term of a sample); one more launch when given.
 * FINC_FLAG_LOGDET_ACCUMULATE adds into it in both directions.
 * x, y: NCHW [B, C, H, W] (y == x allowed); the hidden activations stay channels-last in `workspace`.
 * `prepared` = finc_coupling_prepare_f32(net.0.weight [width,C/2,3,3], net.0.bias, net.2.weight
 * [width,width,1,1], net.2.bias, net.4.weight [C,width,3,3], net.4.bias, net.4.logs, logscale_factor).
 * finc_coupling_prepared_bytes returns 0 for shapes the path does not cover
 * (C even, round_up(C,16) in {16,32,48,64,96}, width % 32 == 0). */
size_t finc_coupling_prepared_bytes(int C, int width, int with_backward);
size_t finc_coupling_workspace_bytes(int B, int C, int H, int W, int width);
int finc_coupling_prepare_f32(const float* w1, const float* b1, const float* w2, const float* b2, const float* w3,
                              const float* b3, const float* logs3, float logscale_factor, void* prepared,
                              int C, int width, int with_backward, void* stream);
int finc_coupling_apply_f32(const float* x, float* y, float* logdet, const void* prepared, void* workspace,
                            size_t workspace_bytes, int B, int C, int H, int W, int width, int reverse,
                            unsigned flags, void* stream);

/* Backward of finc_coupling_apply_f32: given dy = dL/dy and dlogdet = dL/dlogdet [B] (may be NULL) it produces dx and
 * the gradients of the seven parameters (same shapes as the parameters).
 * `forward_workspace` is the workspace the apply call filled (it holds the hidden activations), `x` that call's input
 * and `prepared` a blob made with with_backward = 1 (it carries the transposed weights).  Without flags this is the
 * backward of the forward direction (reverse = 0); with FINC_FLAG_COUPLING_REVERSE it is the backward of the reverse
 * direction (reverse = 1), `dlogdet` then being the gradient of the reverse log-det -sum log_s.  The network
 * h = net(x1) is the same in both directions, so only the pointwise step differs.  Eleven GEMM-class launches on the
 * tensor cores (three weight-gradient GEMMs over the pixels, three backward-data GEMMs) plus small
 * deterministic reductions; no floating-point atomics.  width % 128 == 0.  Replaces the autograd graph of
 * Coupling.forward / Coupling.reverse (fastflow/layers/coupling.py:85-99; cuDNN dgrad / wgrad). */
size_t finc_coupling_backward_workspace_bytes(int B, int C, int H, int W, int width);
int finc_coupling_backward_f32(const float* x, const float* dy, const float* dlogdet, const void* prepared,
                               const void* forward_workspace, void* scratch, size_t scratch_bytes, float* dx,
                               float* dw1, float* db1, float* dw2, float* db2, float* dw3, float* db3, float* dlogs3,
                               int B, int C, int H, int W, int width, unsigned flags, void* stream);

/* Dense form of the inverse for the deep, small levels (n = C*H*W unknowns per (image, group), 64 <= n <= 1024,
 * n % 64 == 0: the 4x4 and 8x8 tiles of the flows).  x = L^-1 z is the same linear map for every image, so a batch
 * is one tensor-core GEMM per group (3xTF32, fp32 parity) instead of an anti-diagonal recurrence 4 .. 8 pixels wide.
 * finc_inverse_dense_prepare_f32 builds L^-1 for every group by running finc_inverse_f32 on the identity -- once per
 * weight update; `scratch` >= finc_inverse_dense_scratch_bytes.  Same result as finc_inverse_f32 up to fp32
 * rounding; for sampling with fixed weights (fastflow/fastflow.py:78-100 called per layer per sample batch). */
size_t finc_inverse_dense_bytes(int G, int C, int H, int W);           /* 0 = shape not covered */
size_t finc_inverse_dense_scratch_bytes(int G, int C, int H, int W);
int finc_inverse_dense_prepare_f32(const float* w, void* prepared, void* scratch, size_t scratch_bytes,
                                   int G, int C, int H, int W, int kH, int kW, unsigned orders, void* stream);
int finc_inverse_dense_f32(const float* z, const void* prepared, float* x, int B, int G, int C, int H, int W,
                           unsigned flags, void* stream);

/* A chain of FInC units -- each optionally followed by its ActNorm o Conv1x1 affine map -- in ONE launch; the
 * image tiles stay in shared memory between units.
 *   cur = x;  for j in 0 .. n_units-1:  u = u_first + j*u_step;
 *       cur = FInC(cur; w + u*w_stride)            (fastflow/fastflow.py:31-50, layers/conv.py:102-107; with
 *                                                   FINC_FLAG_CHAIN_TRANSPOSE its backward-data map)
 *       if A:  cur = (A + u*GC*GC) cur + (bias + u*GC)      (layers/actnorm.py:14-52 + layers/conv1x1.py:18-43,
 *                                                   composed as for finc_affine1x1_f32; GC = G*C)
 *       y + u*y_stride = cur                       (y_stride == 0: only the last unit's result is written to y)
 *   logdet (nullable, [B]) = sum over the chain's units of H*W*sum log|diag| (affine terms are the caller's;
 *   FINC_FLAG_LOGDET_ACCUMULATE adds into it).
 * One launch replaces the FastFlowUnit + ActNorm + Conv1x1 sequence of a FastFlowStep (n_units = 1), or the
 * n_units forward / backward-data launches of a stack of consecutive units.  Results are bit-identical to the
 * per-unit calls.  kH = kW = 3, C in {1,2,3,6,12,24}; other shapes: FINC_E_UNSUPPORTED (finc_chain_supported = 0). */
/* finc_backward_weight_f32 for n_units units in ONE launch (each unit gets 1/n_units of the SMs): unit u reads
 * dz + u*dz_unit_stride and x + u*x_unit_stride (floats) and writes dw + u*dw_unit_stride -- e.g. every unit of a
 * level once its backward-data chain has produced all dz (the reference: one cuDNN wgrad + `grad * mask` per
 * layer, layers/conv.py:98-99).  Same masked, deterministic result as the per-unit call.  FINC_E_UNSUPPORTED when
 * the tiled kernel does not cover the shape (call finc_backward_weight_f32 per unit then). */
size_t finc_backward_weight_batched_workspace_bytes(int B, int G, int C, int H, int W, int kH, int kW, int n_units);
int finc_backward_weight_batched_f32(const float* dz, const float* x, float* dw, void* workspace, size_t workspace_bytes,
                                     int B, int G, int C, int H, int W, int kH, int kW, unsigned orders, unsigned flags,
                                     int n_units, long dz_unit_stride, long x_unit_stride, long dw_unit_stride,
                                     void* stream);

/* The sampling direction of a chain: x = FInC_u^-1(... ) for the units u_first, u_first + u_step, ... (n_units of
 * them) solved IN PLACE by the register-window wavefront kernel while the tiles stay in shared memory: one launch,
 * no intermediate result written (reference: one reverse_level2 call and (H+W-1)*Cq launches per unit,
 * fastflow/fastflow.py:78-100).  `prepared` = FINC_PREP_INVERSE tables (finc_prepare_weights_f32), unit u's table at
 * prepared + u * prepared_stride_bytes.  Bit-identical to n_units finc_inverse_f32 calls.  FINC_E_UNSUPPORTED when
 * the shape is not covered by the register-window kernel or the tables of the chain do not fit shared memory. */
int finc_inverse_chain_f32(const float* z, const void* prepared, size_t prepared_stride_bytes, float* x, int B, int G,
                           int C, int H, int W, int kH, int kW, unsigned orders, int n_units, int u_first, int u_step,
                           void* stream);

/* The sampling chains of several levels (independent inputs, e.g. the levels of a multi-scale flow) in ONE launch:
 * level i is what finc_inverse_chain_f32 with levels[i]'s arguments computes, bit for bit.  The warp items of all
 * levels run side by side, so small batches -- where one level's chain leaves most SMs idle -- take about as long as
 * the slowest level instead of the sum.  Levels with B = 0 are skipped.  FINC_E_UNSUPPORTED when a level is not one
 * of the instantiated kinds (kH = kW = 3 and (C, P) = (3, 1), (6, 2), (12, 4), P being what the single-level launch
 * picks), when n_levels > 4, or when the levels do not fit on the GPU at once (shared memory per CTA,
 * every CTA resident); call finc_inverse_chain_f32 per level then. */
typedef struct FincInverseLevel {
    const float* z;
    const void* prepared;
    size_t prepared_stride_bytes;
    float* x;
    int B, G, C, H, W, kH, kW;
    unsigned orders;
    int n_units, u_first, u_step;
} FincInverseLevel;
int finc_inverse_chain_multi_f32(const FincInverseLevel* levels, int n_levels, void* stream);

int finc_chain_supported(int G, int C, int H, int W, int kH, int kW, int with_affine);
int finc_chain_f32(const float* x, const float* w, long w_stride, float* y, long y_stride, const float* A,
                   const float* bias, float* logdet, int B, int G, int C, int H, int W, int kH, int kW,
                   unsigned orders, int n_units, int u_first, int u_step, unsigned flags, void* stream);

/* Debug aid, inactive unless the environment has FINC_DEBUG_TS=1: the tiled kernels then record
 * per-CTA %globaltimer marks (8 slots per CTA); this call synchronises the device and copies them. */
int finc_debug_timestamps(unsigned long long* host_out, int n);

#ifdef __cplusplus
}
#endif
#endif /* FINCFLOW_B200_H_ */

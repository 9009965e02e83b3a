// finc_wgrad.cu -- masked weight gradient of the FInC convolution, sm_100a.
//
//   dw[g][o][i][a][b] = sum_{n,h,w} dz[n,gC+o,h,w] * x[n,gC+i,h+r(a),w+c(b)]
//   dw[g][o][i][a*][b*] = 0 for i >= o                    (PaddedConv2d.reset_gradients)
//
// Replaces cuDNN wgrad + the post-hoc `grad * mask.to(device)` of the reference
// (layers/conv.py:98-99, train/experiment.py:16-18,250).  The result can be written
// straight into a flat gradient bucket (the NCCL all-reduce buffer).
//
// A long reduction (B*H*W terms) into few outputs (C*C*kH*kW per group):
//   * grid = (X, G, Z): CTA (x, g, z) streams every X-th chunk of CH images of group g -- the
//     x and dz tiles, 2*CH TMA bulk copies per chunk on a full/empty mbarrier ring fed by a
//     producer warp -- and owns the (input channel, output block) combos of slice z.
//   * output-stationary lanes: a lane owns one combo (i, OB output channels) and one slot
//     (tile of the chunk, WT-wide column strip, row range); it keeps OB*kH*kW accumulators
//     in registers for the whole kernel.  Sweeping its rows it holds a sliding window of kH
//     input row strips in registers (one new row = two vector loads per step, rotated at
//     compile time) and loads OB dz strips: (2 + OB) shared loads feed OB*kH*kW*WT FMAs.
//     Rows / halos outside the image are redirected to a zero strip (no branches).
//   * deterministic reduction: segmented xor-shuffle over the slots of a combo, fixed-order
//     sums over warps (shared) and over the X CTAs (global partials; the last CTA to finish,
//     found with one atomic ticket per (g,z), applies the mask and writes dw).  No
//     floating-point atomics anywhere.
#include "finc_common.cuh"

#include <cstdio>
#include <cstdlib>

namespace finc {

namespace {

constexpr int kMaxConsumerWarps = 16;
// accumulators + window + dz strips of an OB=6 lane need ~150 registers: 12 consumer warps
constexpr int max_consumer_warps(int ob, int kh) { return (ob >= 6 || (kh >= 5 && ob >= 2)) ? 12 : kMaxConsumerWarps; }
constexpr int kCounterBytes = 4096;
constexpr int kFrontPad = 32;

struct WgArgs {
    const float* dz;
    const float* x;
    float* dw;
    float* partial;
    unsigned* counters;
    Shape s;
    unsigned flags;
    int CH, S, bulk, tile_floats;
    int tile_stride;           // floats between tiles in shared memory: tile_floats + 4, so that lanes that differ
                               // in the tile index (fastest in the slot order) hit different 16-byte bank groups
    int nob, nstrip, RR, rpr;  // output blocks, strips per row, row ranges per tile, rows per range
    int slots, SP;             // slots per combo and its padded size (power of two <= 32, or multiple of 32)
    int ncombo, cpc;           // combos in total / per CTA
    int X, Z, nchunks;
    unsigned long long* dbg;
    unsigned m_nstrip, m_ch;
    // batched over units (one launch for every unit of a level): blockIdx.z = unit * Z + slice; unit u reads
    // dz + u * dz_ustride and x + u * x_ustride, writes dw + u * dw_ustride, reduces in workspace + u * ws_ustride
    int n_units;
    long dz_ustride, x_ustride, dw_ustride, ws_ustride;
};

__device__ __forceinline__ unsigned fastdiv(unsigned n, unsigned m) { return m ? __umulhi(n, m) : n; }

template <int N>
__device__ __forceinline__ void ldn(const float* p, float* out) {
    if constexpr (N == 4) {
        const float4 v = *reinterpret_cast<const float4*>(p);
        out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
    } else if constexpr (N == 2) {
        const float2 v = *reinterpret_cast<const float2*>(p);
        out[0] = v.x; out[1] = v.y;
    } else {
        out[0] = p[0];
    }
}

template <int WT, int HALO>
__device__ __forceinline__ void ld_halo(const float* p, float* out) {
    if constexpr (WT == 4 && HALO == 4) { ldn<4>(p, out); }
    else {
#pragma unroll
        for (int q = 0; q < HALO; q += 2) ldn<2>(p + q, out + q);
    }
}

// strip of x row hh (WT + HALO floats starting at column w0 - HALO (left padded) or w0)
template <int WT, int HALO, bool RIGHT>
__device__ __forceinline__ void load_row(const float* __restrict__ xc, const float* __restrict__ zrow, int hh, int H,
                                         int W, int w0, float* out) {
    const bool ok = hh >= 0 && hh < H;
    const float* row = xc + hh * W + w0;
    const bool hok = ok && (RIGHT ? (w0 + WT < W) : (w0 > 0));
    const float* mp = ok ? row : zrow;
    const float* hp = hok ? (RIGHT ? row + WT : row - HALO) : zrow;
    if constexpr (RIGHT) {
        ldn<WT>(mp, out);
        ld_halo<WT, HALO>(hp, out + WT);
    } else {
        ld_halo<WT, HALO>(hp, out);
        ldn<WT>(mp, out + HALO);
    }
}

template <int OB, int WT, int KH, int KW, bool RIGHT>
__device__ __forceinline__ void sweep(float (&acc)[OB][KH][KW], const float* __restrict__ xc,
                                      const float* __restrict__ dzc, const float* __restrict__ zrow, int nvalid_o,
                                      int H, int W, int HW, int w0, int r0, int h0, int h1) {
    constexpr int HALO = KW - 1;
    float win[KH][WT + HALO];
    // rows h0+r0 .. h0+r0+KH-2 of the window; the last row is loaded inside the step
#pragma unroll
    for (int a = 0; a < KH - 1; ++a) load_row<WT, HALO, RIGHT>(xc, zrow, h0 + r0 + a, H, W, w0, win[a]);
    for (int hb = h0; hb < h1; hb += KH) {
#pragma unroll
        for (int rot = 0; rot < KH; ++rot) {
            const int h = hb + rot;
            if (h < h1) {
                // window row for tap a lives in win[(a + rot) % KH]
                load_row<WT, HALO, RIGHT>(xc, zrow, h + r0 + KH - 1, H, W, w0, win[(KH - 1 + rot) % KH]);
                float dzv[OB][WT];
#pragma unroll
                for (int o = 0; o < OB; ++o) {
                    const float* dp = (o < nvalid_o) ? dzc + o * HW + h * W + w0 : zrow;
                    ldn<WT>(dp, dzv[o]);
                }
#pragma unroll
                for (int a = 0; a < KH; ++a)
#pragma unroll
                    for (int b = 0; b < KW; ++b)
#pragma unroll
                        for (int o = 0; o < OB; ++o)
#pragma unroll
                            for (int q = 0; q < WT; ++q)
                                acc[o][a][b] = fmaf(dzv[o][q], win[(a + rot) % KH][q + b], acc[o][a][b]);
            }
        }
    }
}

template <int OB, int WT, int KH, int KW>
__global__ void __launch_bounds__((max_consumer_warps(OB, KH) + 1) * 32, 1) wgrad_kernel(const WgArgs a) {
    constexpr int NACC = OB * KH * KW;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const Shape& s = a.s;
    const int C = s.C, H = s.H, W = s.W, HW = H * W;
    float* front = reinterpret_cast<float*>(smem_raw);  // kFrontPad zero floats
    float* zrow = front + 8;
    float* bufs = front + kFrontPad;
    const int half = a.CH * a.tile_stride;  // floats of x (or dz) tiles per stage
    float* red = bufs + (size_t)a.S * 2 * half + 8;
    const int nthreads_c = blockDim.x - 32;
    const int nseg_max = nthreads_c / (a.SP < 32 ? a.SP : 32);
    uint64_t* full = reinterpret_cast<uint64_t*>(red + ((nseg_max * NACC + 1) & ~1));
    uint64_t* empty = full + a.S;
    __shared__ int s_last;

    const int g = blockIdx.y, uu = (int)blockIdx.z / a.Z, zz = (int)blockIdx.z - uu * a.Z;
    const float* const dz_u = a.dz + (long)uu * a.dz_ustride;
    const float* const x_u = a.x + (long)uu * a.x_ustride;
    float* const dw_u = a.dw + (long)uu * a.dw_ustride;
    float* const partial_u = a.partial + (long)uu * a.ws_ustride;
    unsigned* const counters_u = a.counters + (long)uu * a.ws_ustride;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool is_producer = warp == (nthreads_c >> 5);
    const int ord = order_of(s.orders, g);
    const bool right = (ord & 1) != 0;
    const int r0 = (ord & 2) ? 0 : -(KH - 1);

    auto issue = [&](int chunk, int st) {  // the whole producer warp: copies are issued by 32 lanes
        const int n0 = chunk * a.CH;
        const int nt = min(a.CH, s.B - n0);
        if (lane == 0) mbar_arrive_expect_tx(&full[st], (uint32_t)(2 * nt * a.tile_floats * 4));
        __syncwarp();
        float* xs = bufs + (size_t)st * 2 * half;
        float* ds = xs + half;
        for (int t = lane; t < nt; t += 32) {
            const long off = ((long)(n0 + t) * s.G + g) * a.tile_floats;
            bulk_g2s(xs + t * a.tile_stride, x_u + off, (uint32_t)(a.tile_floats * 4), &full[st]);
            bulk_g2s(ds + t * a.tile_stride, dz_u + off, (uint32_t)(a.tile_floats * 4), &full[st]);
        }
    };

    if (threadIdx.x == 0) dbg_mark(a.dbg, 0);
    if (a.bulk && is_producer && lane == 0) {
        for (int st = 0; st < a.S; ++st) {
            mbar_init(&full[st], 1);
            mbar_init(&empty[st], nthreads_c >> 5);
        }
        fence_mbar_init();
    }
    pdl_wait();
    pdl_trigger();
    if (a.bulk && is_producer) {
        for (int st = 0; st < a.S; ++st) {
            const int chunk = blockIdx.x + st * a.X;
            if (chunk < a.nchunks) issue(chunk, st);
        }
    }
    if (threadIdx.x < kFrontPad) front[threadIdx.x] = 0.f;
    __syncthreads();

    if (is_producer) {
        if (a.bulk) {
            int k = a.S;
            for (int chunk = blockIdx.x + a.S * a.X; chunk < a.nchunks; chunk += a.X, ++k) {
                const int st = k % a.S;
                mbar_wait(&empty[st], (uint32_t)(((k / a.S) - 1) & 1));
                issue(chunk, st);
            }
        }
    } else {
        // ---- consumers: lane <-> (combo, slot) -------------------------------------------------------
        const int cl = threadIdx.x / a.SP;            // combo slot inside the CTA
        const int slot = threadIdx.x - cl * a.SP;
        const int combo = zz * a.cpc + cl;
        const bool lane_on = cl < a.cpc && combo < a.ncombo && slot < a.slots;
        const int ci = lane_on ? combo / a.nob : 0;
        const int ob = lane_on ? combo - ci * a.nob : 0;
        // slot = (rr * nstrip + strip) * CH + t: the tile index varies fastest across lanes
        const unsigned q1 = fastdiv((unsigned)slot, a.m_ch);
        const int t = slot - (int)q1 * a.CH;
        const unsigned q2 = fastdiv(q1, a.m_nstrip);
        const int strip = (int)q1 - (int)q2 * a.nstrip;
        const int rr = (int)q2;
        const int w0 = strip * WT;
        const int h0 = rr * a.rpr, h1 = min(H, h0 + a.rpr);
        const int nvalid_o = min(OB, C - ob * OB);

        float acc[OB][KH][KW];
#pragma unroll
        for (int o = 0; o < OB; ++o)
#pragma unroll
            for (int aa = 0; aa < KH; ++aa)
#pragma unroll
                for (int b = 0; b < KW; ++b) acc[o][aa][b] = 0.f;

        int k = 0;
        for (int chunk = blockIdx.x; chunk < a.nchunks; chunk += a.X, ++k) {
            const int st = k % a.S;
            const int n0 = chunk * a.CH;
            const int nt = min(a.CH, s.B - n0);
            float* xs = bufs + (size_t)st * 2 * half;
            float* ds = xs + half;
            if (a.bulk) {
                mbar_wait(&full[st], (uint32_t)((k / a.S) & 1));
                if (threadIdx.x == 0 && k == 0) dbg_mark(a.dbg, 1);
            } else {
                asm volatile("bar.sync 1, %0;" ::"r"(nthreads_c) : "memory");
                for (int tt = 0; tt < nt; ++tt) {
                    const long off = ((long)(n0 + tt) * s.G + g) * a.tile_floats;
                    for (int e = threadIdx.x; e < a.tile_floats; e += nthreads_c) {
                        xs[tt * a.tile_stride + e] = x_u[off + e];
                        ds[tt * a.tile_stride + e] = dz_u[off + e];
                    }
                }
                asm volatile("bar.sync 1, %0;" ::"r"(nthreads_c) : "memory");
            }
            if (lane_on && rr < a.RR && t < nt && h0 < h1) {
                const float* xc = xs + t * a.tile_stride + ci * HW;
                const float* dzc = ds + t * a.tile_stride + (ob * OB) * HW;
                if (right) sweep<OB, WT, KH, KW, true>(acc, xc, dzc, zrow, nvalid_o, H, W, HW, w0, r0, h0, h1);
                else sweep<OB, WT, KH, KW, false>(acc, xc, dzc, zrow, nvalid_o, H, W, HW, w0, r0, h0, h1);
            }
            if (a.bulk) {
                __syncwarp();
                if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&empty[st])) : "memory");
            }
        }

        if (threadIdx.x == 0) dbg_mark(a.dbg, 2);
        // ---- lanes of a combo -> one value per segment (segment = min(SP,32) consecutive lanes) ------
        // level-major: the NACC shuffles of one level are independent and pipeline
        const int SPw = a.SP < 32 ? a.SP : 32;
        const int seg = threadIdx.x / SPw;
        for (int off = 1; off < SPw; off <<= 1) {
#pragma unroll
            for (int o = 0; o < OB; ++o)
#pragma unroll
                for (int aa = 0; aa < KH; ++aa)
#pragma unroll
                    for (int b = 0; b < KW; ++b) acc[o][aa][b] += __shfl_xor_sync(0xffffffffu, acc[o][aa][b], off);
        }
        if ((threadIdx.x & (SPw - 1)) == 0) {
#pragma unroll
            for (int o = 0; o < OB; ++o)
#pragma unroll
                for (int aa = 0; aa < KH; ++aa)
#pragma unroll
                    for (int b = 0; b < KW; ++b) red[seg * NACC + (o * KH + aa) * KW + b] = acc[o][aa][b];
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) dbg_mark(a.dbg, 3);

    // ---- segments -> CTA value per output (fixed order), then CTAs -> dw ----------------------------
    // partial slices are stored in CTA-local order [x][g][z][cl*NACC + idx]: coalesced both ways
    const int ca = corner_a(ord, KH), cbn = corner_b(ord, KW);
    const int segs_per_combo = a.SP <= 32 ? 1 : a.SP / 32;
    const bool direct = a.X == 1;
    const int nloc = a.cpc * NACC;
    const long slice = ((long)g * a.Z + zz) * nloc;
    const long xstride = (long)s.G * a.Z * nloc;
    auto finish = [&](int l, float v) {
        const int cl = l / NACC, idx = l - cl * NACC;
        const int combo = zz * a.cpc + cl;
        if (combo >= a.ncombo) return;
        const int i = combo / a.nob, ob = combo - i * a.nob;
        const int o = ob * OB + idx / (KH * KW);
        if (o >= C) return;
        const int ab = idx % (KH * KW);
        const long out = (((long)g * C + o) * C + i) * KH * KW + ab;
        if (!(a.flags & FINC_FLAG_NO_MASK) && ab == ca * KW + cbn && i >= o) v = 0.f;
        else if (a.flags & FINC_FLAG_NEGATE) v = -v;
        if (a.flags & FINC_FLAG_ACCUMULATE) v += dw_u[out];
        dw_u[out] = v;
    };
    for (int l = threadIdx.x; l < nloc; l += blockDim.x) {
        const int cl = l / NACC;
        float v = 0.f;
        for (int r = 0; r < segs_per_combo; ++r) v += red[(cl * segs_per_combo + r) * NACC + (l - cl * NACC)];
        if (direct) finish(l, v);
        else partial_u[(long)blockIdx.x * xstride + slice + l] = v;
    }
    if (direct) return;

    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned ticket = atomicAdd(&counters_u[g * a.Z + zz], 1u);
        s_last = (ticket == (unsigned)(a.X - 1));
    }
    __syncthreads();
    if (threadIdx.x == 0) dbg_mark(a.dbg, 4);
    if (!s_last) return;
    __threadfence();
    // the last CTA of (g, z) sums the X slices per output.  `parts` threads share one output:
    // thread (l, q) sums slices q, q+parts, ... (independent coalesced loads, one L2 round trip
    // for the usual X <= 64), the parts are combined in fixed order through shared memory.
    {
        int parts = (int)blockDim.x / nloc;
        if (parts > 8) parts = 8;
        if (parts < 1) parts = 1;
        float* comb = bufs;  // pipeline buffers are free now; needs nloc*parts floats
        if ((long)nloc * parts > (long)a.S * 2 * half) parts = 1;
        for (int l0 = 0; l0 < nloc; l0 += (int)blockDim.x / parts) {
            const int tl = threadIdx.x / parts, q = threadIdx.x - tl * parts;
            const int l = l0 + tl;
            float v = 0.f;
            if (l < nloc && tl < (int)blockDim.x / parts) {
                const float* pp = partial_u + slice + l;
                for (int xx0 = q; xx0 < a.X; xx0 += 8 * parts) {  // 8 independent loads in flight
                    float t8[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int xx = xx0 + u * parts;
                        t8[u] = xx < a.X ? __ldcg(pp + (long)xx * xstride) : 0.f;
                    }
#pragma unroll
                    for (int u = 0; u < 8; ++u) v += t8[u];
                }
            }
            if (parts == 1) {
                if (l < nloc) finish(l, v);
            } else {
                comb[threadIdx.x] = v;
                __syncthreads();
                if (q == 0 && l < nloc && tl < (int)blockDim.x / parts) {
                    float t = 0.f;
                    for (int qq = 0; qq < parts; ++qq) t += comb[threadIdx.x + qq];
                    finish(l, t);
                }
                __syncthreads();
            }
        }
    }
    if (threadIdx.x == 0) counters_u[g * a.Z + zz] = 0u;  // leave the ticket clean
    __syncthreads();
    if (threadIdx.x == 0) dbg_mark(a.dbg, 5);
}

template <int OB, int WT, int KH, int KW>
int launch_inst(const WgArgs& a, dim3 grid, int threads, size_t smem, cudaStream_t st) {
    auto kern = wgrad_kernel<OB, WT, KH, KW>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    return launch_kernel(kern, grid, threads, smem, st, a);
}

template <int OB, int WT>
int dispatch_k(int kH, const WgArgs& a, dim3 grid, int threads, size_t smem, cudaStream_t st) {
    if (kH == 3) return launch_inst<OB, WT, 3, 3>(a, grid, threads, smem, st);
    if constexpr (OB <= 2) {
        if (kH == 5) return launch_inst<OB, WT, 5, 5>(a, grid, threads, smem, st);
    }
    return FINC_E_UNSUPPORTED;
}

template <int OB>
int dispatch_wt(int WT, int kH, const WgArgs& a, dim3 grid, int threads, size_t smem, cudaStream_t st) {
    if (WT == 4) return dispatch_k<OB, 4>(kH, a, grid, threads, smem, st);
    return dispatch_k<OB, 2>(kH, a, grid, threads, smem, st);
}

unsigned magic(unsigned d) { return d <= 1 ? 0u : (unsigned)(((1ull << 32) + d - 1) / d); }

struct Plan {
    int OB, WT, nob, nstrip, RR, rpr, slots, SP, ncombo, cpc, Z, X, CH, S, nchunks, threads;
    size_t smem;
};

// Plan = (output block OB, combos per CTA / output slices Z, batch slices X, chunk size CH, row
// ranges RR).  More X = more CTAs sweeping but more partial vectors for the last CTA to sum;
// more Z = shorter partial vectors but every slice re-reads the tiles.  A small cost model
// (microseconds, calibrated with tools/kernel_timeline.py) picks the cheapest combination.
bool make_plan(const Shape& s, Plan* p, int sm_div = 1) {
    if (s.B < 1) return false;  // no chunks to spread: the per-CTA chunk count would divide by zero
    if (!(s.kH == s.kW && (s.kH == 3 || s.kH == 5))) return false;
    int WT;
    if (s.W % 4 == 0) WT = 4;
    else if (s.W % 2 == 0 && s.kW - 1 <= 2) WT = 2;  // vector halo needs HALO <= WT
    else return false;
    const long tile_bytes = (long)s.C * s.H * s.W * 4;
    if (tile_bytes > 24 * 1024) return false;
    int sms = sm_count_cached() / sm_div;  // sm_div > 1: leave room for sibling launches on other streams
    if (sms < s.G) sms = s.G;
    const int nstrip = s.W / WT;
    const int max_ob = s.kH == 3 ? 6 : 2;
    const size_t budget = max_optin_smem_cached() > 8192 ? max_optin_smem_cached() - 4096 : 0;
    const int kk = s.kH * s.kW;
    bool have = false;
    double best_cost = 1e30;
    Plan best{};
    // FINC_WG_FORCE="ob,z,ch" pins parts of the plan (0 = free): used by tools/sweep_wgrad.py
    int f_ob = 0, f_z = 0, f_ch = 0;
    if (const char* e = getenv("FINC_WG_FORCE")) sscanf(e, "%d,%d,%d", &f_ob, &f_z, &f_ch);
    for (int ob : {6, 4, 3, 2, 1}) {
        if (f_ob && ob != f_ob) continue;
        if (ob > max_ob || ob > s.C) continue;
        if (s.C % ob != 0 && !(ob == 4 && s.C > 6) && ob != 1) continue;
        const int nob = (s.C + ob - 1) / ob;
        const int ncombo = s.C * nob;
        const int nacc = ob * kk;
        const int maxthr = max_consumer_warps(ob, s.kH) * 32;
        for (int zt = 1; zt <= ncombo; zt = zt < 4 ? zt + 1 : zt + zt / 2) {
            Plan q{};
            q.OB = ob; q.WT = WT; q.nob = nob; q.nstrip = nstrip; q.ncombo = ncombo;
            q.cpc = (ncombo + zt - 1) / zt;
            q.Z = (ncombo + q.cpc - 1) / q.cpc;
            if (f_z && q.Z != f_z) continue;
            if ((long)s.G * q.Z * 4 > kCounterBytes) continue;
            if (s.G * q.Z > sms) continue;  // one wave of CTAs
            int x = sms / (s.G * q.Z);
            if (x < 1) x = 1;
            int CH = (s.B + x - 1) / x;  // one chunk per CTA when it fits
            const long ch_mem = (long)((budget - 16384) / (2 * (tile_bytes + 16)));
            if (CH > ch_mem) CH = (int)ch_mem;
            if (CH > 32) CH = 32;
            if (f_ch && CH > f_ch) CH = f_ch;
            if (CH < 1) CH = 1;
            // row ranges and slot padding so that the CTA's combos fit its threads
            int RR = 1, SP = 0;
            for (;;) {
                bool ok = false;
                for (int r : {4, 2, 1}) {
                    if (r > 1 && (s.H + r - 1) / r < 2) continue;
                    const int slots = CH * nstrip * r;
                    const int sp = slots <= 32 ? (slots <= 1 ? 1 : 1 << (32 - __builtin_clz(slots - 1))) : ((slots + 31) / 32) * 32;
                    if ((long)sp * q.cpc <= maxthr) { RR = r; SP = sp; ok = true; break; }
                }
                if (ok || CH == 1) break;
                CH = CH > 2 ? CH - CH / 4 - (CH < 4 ? 1 : 0) : 1;
            }
            if (SP == 0 || (long)SP * q.cpc > maxthr) continue;
            q.CH = CH; q.RR = RR; q.SP = SP;
            q.slots = CH * nstrip * RR;
            q.rpr = (s.H + RR - 1) / RR;
            q.nchunks = (s.B + CH - 1) / CH;
            q.X = x < q.nchunks ? x : q.nchunks;
            const int cpcta = (q.nchunks + q.X - 1) / q.X;
            q.S = cpcta < 3 ? cpcta : 3;
            q.threads = ((q.cpc * q.SP + 31) / 32 + 1) * 32;
            const int nseg = (q.threads - 32) / (q.SP < 32 ? q.SP : 32);
            for (;;) {
                q.smem = (size_t)kFrontPad * 4 + (size_t)q.S * 2 * CH * (tile_bytes + 16) + 32 + (size_t)(nseg * nacc + 2) * 4 +
                         2 * q.S * 8 + 64;
                if (q.smem <= budget || q.S == 1) break;
                --q.S;
            }
            if (q.smem > budget) continue;
            // ---- cost model (microseconds; constants fitted to tools/sweep_wgrad.py on B200) ----
            const double warps = (q.threads - 32) / 32.0;
            const double per_smsp = warps > 4 ? warps / 4 : 1.0;
            const double row_instr = ob * kk * WT + 4 * ob + 20;  // FMAs + strip loads + per-row bookkeeping
            const double t_sweep = cpcta * (q.rpr + s.kH - 1) * row_instr * per_smsp / 1200.0;
            int lg = 0;
            for (int v = 1; v < (SP < 32 ? SP : 32); v <<= 1) ++lg;
            const double t_reduce = 0.4 + nacc * lg * 2.0 * per_smsp / 1200.0;
            const double nloc = (double)q.cpc * nacc;
            const double batches = (nloc * q.X) / ((q.threads) * 8.0);
            const double t_tail = q.X > 1 ? 1.3 + 0.6 * (batches < 1 ? 1 : batches) : 0.0;
            const double occupancy_penalty = (double)(s.G * q.Z * q.X) < 0.5 * sms ? 0.5 : 0.0;
            // a chunk: copy issue (2*CH bulk copies over 32 lanes) + bytes at ~40 KB/us per SM; the first
            // one is exposed, the others overlap the sweep but bound it from below
            const double t_chunk = 0.07 * ((2 * CH + 31) / 32) + (2.0 * CH * tile_bytes) / 40000.0;
            const double t_ingest = (cpcta - 1) * t_chunk;
            // every output slice re-reads the tiles of its group: Z-fold L2 traffic
            const double t_traffic = (double)q.Z * 2.0 * s.B * s.G * tile_bytes / 4.0e6;
            double cost = 1.3 + t_chunk + (t_sweep > t_ingest ? t_sweep : t_ingest) + t_reduce + t_tail + occupancy_penalty +
                          1.5 * (cpcta - 1);
            if (t_traffic > cost) cost = t_traffic;
            if (cost < best_cost) { best_cost = cost; best = q; have = true; }
        }
    }
    if (!have) return false;
    *p = best;
    return true;
}

}  // namespace

static size_t partial_floats(const Shape& s, const Plan& p) {
    return (size_t)p.X * s.G * p.Z * p.cpc * p.OB * s.kH * s.kW;
}

size_t wgrad_workspace_floats(const Shape& s) {
    Plan p{}, q{};
    size_t f = 0;
    if (make_plan(s, &p)) f = partial_floats(s, p);
    for (int div : {2, 4, 8})
        if (make_plan(s, &q, div)) f = f > partial_floats(s, q) ? f : partial_floats(s, q);
    return kCounterBytes / 4 + f;
}

// workspace floats of ONE unit in a batched launch over n_units units (the units' regions are laid out back to back)
size_t wgrad_batched_workspace_floats(const Shape& s, int n_units) {
    Plan p{};
    if (!make_plan(s, &p, n_units)) return 0;
    return kCounterBytes / 4 + partial_floats(s, p);
}

int launch_wgrad_fast(const float* dz, const float* x, float* dw, float* workspace, size_t ws_floats, const Shape& s,
                      unsigned flags, cudaStream_t st, bool* handled) {
    return launch_wgrad_batched(dz, x, dw, workspace, ws_floats, s, flags, 1, 0, 0, 0, st, handled);
}

// n_units > 1: every unit of a level in ONE launch (each gets 1/n_units of the SMs); unit u reads dz + u*dz_ustride,
// x + u*x_ustride and writes dw + u*dw_ustride; the workspace holds n_units regions of
// wgrad_batched_workspace_floats(s, n_units) floats
int launch_wgrad_batched(const float* dz, const float* x, float* dw, float* workspace, size_t ws_floats, const Shape& s,
                         unsigned flags, int n_units, long dz_ustride, long x_ustride, long dw_ustride,
                         cudaStream_t st, bool* handled) {
    *handled = false;
    Plan p{};
    static const int quarter_div = getenv("FINC_WG_DIV") ? atoi(getenv("FINC_WG_DIV")) : 4;  // experiment knob
    if (!make_plan(s, &p, n_units > 1 ? n_units : ((flags & FINC_FLAG_QUARTER_GPU) ? quarter_div : 1))) return 0;
    const size_t ws_unit = kCounterBytes / 4 + partial_floats(s, p);
    if (ws_floats < ws_unit * (size_t)n_units) return FINC_E_WORKSPACE;
    if ((long)p.Z * n_units > 65535) return 0;
    {
        static const bool dbg_plan = getenv("FINC_WG_DEBUG") != nullptr;
        if (dbg_plan)
            fprintf(stderr, "wgrad plan B%d G%d C%d %dx%d k%d: OB=%d WT=%d nob=%d nstrip=%d RR=%d rpr=%d slots=%d SP=%d ncombo=%d cpc=%d Z=%d X=%d CH=%d S=%d nchunks=%d threads=%d smem=%zu\n",
                    s.B, s.G, s.C, s.H, s.W, s.kH, p.OB, p.WT, p.nob, p.nstrip, p.RR, p.rpr, p.slots, p.SP, p.ncombo, p.cpc,
                    p.Z, p.X, p.CH, p.S, p.nchunks, p.threads, p.smem);
    }
    WgArgs a{};
    a.dz = dz; a.x = x; a.dw = dw; a.s = s; a.flags = flags; a.dbg = debug_ts_buffer();
    a.counters = reinterpret_cast<unsigned*>(workspace);
    a.partial = workspace + kCounterBytes / 4;
    a.n_units = n_units; a.dz_ustride = dz_ustride; a.x_ustride = x_ustride; a.dw_ustride = dw_ustride;
    a.ws_ustride = (long)ws_unit;
    a.CH = p.CH; a.S = p.S; a.nob = p.nob; a.nstrip = p.nstrip; a.RR = p.RR; a.rpr = p.rpr;
    a.slots = p.slots; a.SP = p.SP; a.ncombo = p.ncombo; a.cpc = p.cpc; a.X = p.X; a.Z = p.Z; a.nchunks = p.nchunks;
    a.m_nstrip = magic(p.nstrip); a.m_ch = magic(p.CH);
    a.tile_floats = s.C * s.H * s.W;
    a.tile_stride = a.tile_floats + 4;
    a.bulk = (a.tile_floats % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) &&
             ((reinterpret_cast<uintptr_t>(dz) & 15) == 0);
    if (a.X > 1 && !(flags & FINC_FLAG_WORKSPACE_CLEAN)) {
        // the tickets of every unit (n_units = 1: just the first G*Z counters)
        const size_t bytes = n_units > 1 ? ((size_t)(n_units - 1) * ws_unit + kCounterBytes / 4) * 4 : (size_t)s.G * a.Z * 4;
        cudaError_t e = cudaMemsetAsync(a.counters, 0, bytes, st);
        if (e != cudaSuccess) return (int)e;
    }
    dim3 grid(a.X, s.G, a.Z * n_units);
    int rc;
    switch (p.OB) {
        case 1: rc = dispatch_wt<1>(p.WT, s.kH, a, grid, p.threads, p.smem, st); break;
        case 2: rc = dispatch_wt<2>(p.WT, s.kH, a, grid, p.threads, p.smem, st); break;
        case 3: rc = dispatch_wt<3>(p.WT, s.kH, a, grid, p.threads, p.smem, st); break;
        case 4: rc = dispatch_wt<4>(p.WT, s.kH, a, grid, p.threads, p.smem, st); break;
        default: rc = dispatch_wt<6>(p.WT, s.kH, a, grid, p.threads, p.smem, st); break;
    }
    if (rc == FINC_E_UNSUPPORTED) return 0;
    *handled = true;
    return rc;
}

}  // namespace finc

// finc_inverse_rw.cuh -- register-window wavefront inverse (sampling direction), sm_100a.
//
// Third generation of the FInC inverse (reference: fastflow/fastflow.py:78-100 +
// utils/fastflow_cuda_inverse/cinc_cuda_kernel_level2.cu:49-132, (H+W-1)*Cq launches per unit;
// recurrence: utils/solve_mc.py:88-114).  Same contract and data movement as
// finc_inverse_wave.cuh (warp-persistent workers, TMA bulk load -> in-place solve -> TMA bulk
// store, one launch per unit) but the solve itself never touches shared memory for its
// dependencies:
//
//   * lane = (part p, stack q, sweep column j), column fastest.  The sweep is skewed -- at step s lane j solves
//     stacked row s-j -- so the pixel to the LEFT (row r, column j-1) was finished by lane j-1 one
//     step ago and the pixel ABOVE (row r-1, column j) by this very lane.  Every input of the
//     recurrence therefore arrives either from the lane's own registers or by ONE shuffle from
//     the left neighbour: each lane keeps a KH x KW window of solved pixels in registers
//     (win[kw][row][channel]); column kw of the window is refilled each step with what lane j-1
//     held in column kw-1 one step earlier.  The row index of the window is rotated at compile
//     time (the step loop is unrolled KH times), so the window costs no moves.
//   * no __syncwarp and no shared-memory round trip between diagonals: the critical path of a
//     step is shuffle -> C FMAs -> triangular solve.  Shared memory only supplies z (one load per
//     channel) and receives x (one store per channel) for the TMA engine.
//   * P > 1 splits the INPUT channels of every tap over P adjacent lanes (window and weights
//     shrink by P; partial sums meet in log2(P) xor-shuffles); the channel-triangular corner
//     solve then runs redundantly in registers.  Narrow images put 32/(WP*P) independent tile
//     stacks side by side in one warp instead of splitting taps, so a 16x16x3 tile pair or
//     eight 4x4x12 tiles fill a warp with no reduction at all.
//   * weights: registers when C*C/P*(KH*KW-1) is small (sign folded in), else 128-bit broadcast
//     loads from the sweep-ordered table (same table as finc_inverse_wave.cuh).
//   * ADJ = true solves the adjoint system A^T g = dx of the same map instead (the input gradient of the
//     inverse, finc_inverse_adjoint_f32).  A^T is itself a FInC inverse, swept from the opposite corner
//     (the host flips every group's order) with the weights w''[o, i, a, b] = w[C-1-i, C-1-o, kH-1-a, kW-1-b]
//     and the channels reversed on the way in and out.  The staging builds the sweep-ordered table of w''
//     straight from the raw weights and the channel reversal lives in compile-time register indices, so the
//     recurrence, the data movement and the register budget are those of the inverse.
#pragma once
#include "finc_inverse_wave.cuh"

namespace finc {
namespace rw {

using wave::Pad4;

struct RwArgs {
    const float* z;
    const float* w;
    float* x;
    Shape s;
    int T;         // tiles per stack
    int S;         // pipeline stages per warp (1 or 2)
    int WP;        // column slots per stack (power of two >= W)
    int NSTK;      // stacks per warp in use (<= 32 / (WP * P); lanes beyond them idle)
    int gsplit;
    int bulk;
    int tile_floats;
    int tile_stride;
    int stack_stride;  // floats between the stacks of an item (T*tile_stride + bank skew)
    int wk_floats;
    int prepared;
    unsigned long long* dbg;
    long n_items;
    // chain: n_units > 1 solves the units u_first, u_first + u_step, ... one after the other IN PLACE while the
    // tiles stay in shared memory (prepared tables only; unit u's table at w + u * unit_stride floats); no
    // intermediate result is ever written -- a sampling pass through consecutive units is one launch
    int n_units, u_first, u_step;
    long unit_stride;
};

template <int C, int KH, int KW, int P>
struct Cfg {
    static constexpr int CL = C / P;                      // input channels per lane
    static constexpr int NT = KH * KW - 1;                // non-corner taps
    static constexpr int WIN = KH * KW * CL;              // window registers
    static constexpr int WREGS = C * CL * NT;             // weights per lane
    static constexpr bool WREG = WREGS <= 150;
    static constexpr int CORNER = C * (C - 1) / 2;
    static constexpr bool CREG = CORNER + WIN + (WREG ? WREGS : 0) + C <= 200;
    static constexpr int EST = WIN + C + (WREG ? WREGS : 16) + (CREG ? CORNER : 8) + 30;
    static constexpr int MAXW = EST <= 100 ? 16 : 8;   // (12 warps with shallower stacks measured slower)
};

// The whole solve of one launch's share of a level.  (vblock, vgrid) take the place of (blockIdx.x, gridDim.x) and
// grp that of blockIdx.y (the group of a gsplit launch), so that one launch can host several levels.
// MT: stacks hold more than one tile (large batches).  With one tile per stack the window never
// has to be cleared at a tile top and the row pointer never wraps, which shortens the step.
// WREG / CREG: tap / corner weights held in registers (sign folded in) instead of read from the shared-memory table;
// x * (-w) and (-x) * w round identically, so both give the same bits.
template <int C, int KH, int KW, int P, bool MT, bool WREG, bool CREG, bool ADJ>
__device__ __forceinline__ void inverse_rw_body(const RwArgs& a, int vblock, int vgrid, int grp) {
    using K = Cfg<C, KH, KW, P>;
    constexpr int CL = K::CL;
    constexpr int CPP = Pad4<C>::value;
    constexpr int TS = Pad4<C>::tap_stride;

    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* wk = reinterpret_cast<float*>(smem_raw);
    const int nwarps = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const Shape& s = a.s;
    const int H = s.H, W = s.W;
    const int HW = H * W;
    // channel c of the solved system is channel rv(c) of z and x.  The adjoint reverses the channels in the register
    // indices only (all compile-time), so its shared-memory addressing and register allocation are the inverse's:
    // lane p's window entry il holds system channel rv(il*P + p), and row r of the weight table belongs to system
    // input channel rv(r).  (Reversing them in the addresses instead cost the C = 12, 5x5 kernel spills.)
    auto rv = [](int c) -> int { return ADJ ? C - 1 - c : c; };
    const int NSTK = a.NSTK;
    const int item_tiles = NSTK * a.T;
    const int stage_floats = NSTK * a.stack_stride;
    const int wk_pad = (a.wk_floats + 31) & ~31;
    const int wk_all = wk_pad * a.n_units;
    float* bufs = wk + wk_all + (size_t)warp * a.S * stage_floats;
    uint64_t* bar0 = reinterpret_cast<uint64_t*>(wk + wk_all + (size_t)nwarps * a.S * stage_floats);
    uint64_t* bars = bar0 + warp * a.S;
    uint64_t* wbar = bar0 + nwarps * a.S;

    const int g_fixed = a.gsplit ? grp : -1;
    const long gw = (long)warp * vgrid + vblock;
    const long gstride = (long)vgrid * nwarps;

    auto item_g = [&](long item) -> int { return a.gsplit ? g_fixed : (int)(item % s.G); };
    auto item_n0 = [&](long item) -> int { return (int)(a.gsplit ? item : item / s.G) * item_tiles; };
    auto tile_smem = [&](float* buf, int tt) -> float* { return buf + (tt / a.T) * a.stack_stride + (tt % a.T) * a.tile_stride; };
    auto issue_load = [&](long item, int st) {  // whole warp
        const int g = item_g(item), n0 = item_n0(item);
        const int nt = min(item_tiles, s.B - n0);
        if (lane == 0) mbar_arrive_expect_tx(&bars[st], (uint32_t)(nt * a.tile_floats * 4));
        __syncwarp();
        for (int tt = lane; tt < nt; tt += 32)
            bulk_g2s(tile_smem(bufs + st * stage_floats, tt), a.z + ((long)(n0 + tt) * s.G + g) * a.tile_floats,
                     (uint32_t)(a.tile_floats * 4), &bars[st]);
    };

    if (threadIdx.x == 0) dbg_mark(a.dbg, 0);
    if (a.bulk && lane == 0) {
        for (int st = 0; st < a.S; ++st) mbar_init(&bars[st], 1);
        if (warp == 0) mbar_init(wbar, 1);
        fence_mbar_init();
    }
    if (a.prepared) __syncthreads();  // wbar initialised before anyone waits on it
    else __syncwarp();
    pdl_wait();
    pdl_trigger();
    if (a.prepared && threadIdx.x == 0) {  // the whole weight table of every unit of the chain: one bulk copy each
        if (vblock == 0 && grp == 0) {   // refuse a table of another kind / layout
            const float* h = a.w + (long)a.u_first * a.unit_stride;
            if (__ldg(h) != 1179208259.f || (int)__ldg(h + 1) != 2 || (int)__ldg(h + 2) != CPP || (int)__ldg(h + 3) != TS) __trap();
        }
        const uint32_t wbytes = (uint32_t)a.wk_floats * 4;
        mbar_arrive_expect_tx(wbar, wbytes * (uint32_t)a.n_units);
        for (int uu = 0; uu < a.n_units; ++uu)
            bulk_g2s(wk + (size_t)uu * wk_pad,
                     a.w + (long)(a.u_first + uu * a.u_step) * a.unit_stride + kPrepHeaderFloats +
                         (a.gsplit ? (size_t)g_fixed * a.wk_floats : 0),
                     wbytes, wbar);
    }
    if (a.bulk) {
        for (int st = 0; st < a.S; ++st) {
            const long item = gw + st * gstride;
            if (item < a.n_items) issue_load(item, st);
        }
    }
    if (a.prepared) {
        mbar_wait(wbar, 0);
    } else {
        // sweep-ordered weights: wk[gl][kh][kw][i][CPP] = Ws[g][o][i][a(kh)][b(kw)]
        constexpr int per_g = C * C * KH * KW;
        const int ng = a.gsplit ? 1 : s.G;
        const float* wsrc = a.w + (a.gsplit ? (long)g_fixed * per_g : 0);
        stage_weights(wsrc, ng * per_g, [&](int e, float v) {
            const int gl = e / per_g;
            const int g = a.gsplit ? g_fixed : gl;
            int r = e - gl * per_g;
            const int b = r % KW;
            r /= KW;
            const int aa = r % KH;
            r /= KH;
            int i = r % C, o = r / C;
            int ta = aa, tb = b;
            if constexpr (ADJ) {   // raw w[o][i][aa][b] is w''[C-1-i][C-1-o][KH-1-aa][KW-1-b], in table row rv(C-1-o) = o
                const int o2 = C - 1 - i;
                i = o;
                o = o2;
                ta = KH - 1 - aa;
                tb = KW - 1 - b;
            }
            const int ord = order_of(s.orders, g);
            const int kh = (ord & 2) ? ta : KH - 1 - ta;
            const int kw = (ord & 1) ? tb : KW - 1 - tb;
            wk[((gl * KH + kh) * KW + kw) * TS + i * CPP + o] = v;
        });
        __syncthreads();
    }
    if (threadIdx.x == 0) dbg_mark(a.dbg, 1);

    // lane = (p * QMAX + q) * WP + j: the part index is the SLOW one, so the 8 lanes of a 128-bit
    // shared-memory phase read the same weight vector (with p fastest every LDS.128 of the weight
    // table cost 4 wavefronts and the C = 12 kernel was bound by shared-memory bandwidth)
    constexpr int LP = 32 / P;         // lanes per part
    const int p = lane / LP;
    const int j = lane % a.WP;         // sweep column
    const int q = (lane % LP) / a.WP;  // stack inside the item
    const bool col_on = j < W && q < NSTK;

    long k = 0;
    for (long item = gw; item < a.n_items; item += gstride, ++k) {
        const int st = (int)(k % a.S);
        const int g = item_g(item), n0 = item_n0(item);
        const int nt = min(item_tiles, s.B - n0);
        float* buf = bufs + st * stage_floats;
        if (a.bulk) {
            mbar_wait(&bars[st], (uint32_t)((k / a.S) & 1));
            if (threadIdx.x == 0 && k == 0) dbg_mark(a.dbg, 2);
        } else {
            for (int tt = 0; tt < nt; ++tt) {
                const float* src = a.z + ((long)(n0 + tt) * s.G + g) * a.tile_floats;
                float* dst = tile_smem(buf, tt);
                for (int e = lane; e < a.tile_floats; e += 32) dst[e] = src[e];
            }
            __syncwarp();
        }
        const int ord = order_of(s.orders, g);
        const bool bot = ord & 2, right = ord & 1;
        for (int uu = 0; uu < a.n_units; ++uu) {   // the chain: every unit solves in place what the one before left
        const float* wg = wk + (size_t)uu * wk_pad + (size_t)(a.gsplit ? 0 : g) * KH * KW * TS;
        const float* wgp = wg + p * CPP;  // rows of this lane's input channels: i = il*P + p

        // per-item register weights (negated: acc += x * (-w))
        float wr[WREG ? KH * KW : 1][WREG ? CL : 1][WREG ? C : 1];
        float wc[CREG ? C : 1][CREG ? C : 1];
        if constexpr (WREG) {
#pragma unroll
            for (int t = 1; t < KH * KW; ++t)
#pragma unroll
                for (int il = 0; il < CL; ++il)
#pragma unroll
                    for (int o = 0; o < C; ++o) wr[t][il][o] = -wgp[t * TS + il * P * CPP + o];
        }
        if constexpr (CREG) {
#pragma unroll
            for (int i = 0; i < C; ++i)
#pragma unroll
                for (int o = 0; o < C; ++o) wc[i][o] = wg[rv(i) * CPP + o];
        }

        // this lane's stack
        const int ntq = max(0, min(a.T, nt - q * a.T));
        const int nsteps = min(a.T, nt) * H + W - 1;   // stack 0 is the tallest
        const int s_begin = j;                         // lane j solves stacked row (step - j)
        const int s_end = col_on ? j + ntq * H : j;
        const int wst = right ? W - 1 - j : j;
        const int rowstep = bot ? -W : W;
        const int wrap_adj = a.tile_stride - rowstep * H;
        float* ptr = buf + q * a.stack_stride + (bot ? (H - 1) * W : 0) + (col_on ? wst : 0);
        if constexpr (!MT) ptr -= j * rowstep;         // advanced every step, dereferenced only when active
        int hn = 0;

        float win[KW][KH][CL];
#pragma unroll
        for (int kw = 0; kw < KW; ++kw)
#pragma unroll
            for (int kh = 0; kh < KH; ++kh)
#pragma unroll
                for (int il = 0; il < CL; ++il) win[kw][kh][il] = 0.f;
        float zc[C];   // z of the pixel solved in the current step (loaded one step ahead)
#pragma unroll
        for (int o = 0; o < C; ++o) zc[rv(o)] = (s_begin == 0 && s_end > 0 && p == 0) ? ptr[o * HW] : 0.f;

        for (int step0 = 0; step0 < nsteps; step0 += KH) {
#pragma unroll
            for (int ph = 0; ph < KH; ++ph) {
                const int step = step0 + ph;
                if (step >= nsteps) break;
                const int sp = (ph + KH - 1) % KH;  // slot written one step ago
                const bool active = step >= s_begin && step < s_end;
                // (1) row r of the columns to the left: what lane j-1 held one column closer, one step ago
                float sh[KW - 1][CL];
#pragma unroll
                for (int kw = KW - 1; kw >= 1; --kw)
#pragma unroll
                    for (int il = 0; il < CL; ++il) sh[kw - 1][il] = __shfl_up_sync(0xffffffffu, win[kw - 1][sp][il], 1);
                // (2) z of the next step's pixel travels while this one is solved
                float* nptr = ptr;
                int nhn = hn;
                if constexpr (MT) {
                    if (active) {
                        nptr += rowstep;
                        if (++nhn == H) { nhn = 0; nptr += wrap_adj; }
                    }
                } else {
                    nptr += rowstep;
                }
                const bool act_n = step + 1 >= s_begin && step + 1 < s_end;
                float zn[C];
#pragma unroll
                for (int o = 0; o < C; ++o) zn[rv(o)] = (act_n && p == 0) ? nptr[o * HW] : 0.f;
                // (3) first row of a tile: nothing above it (the zero padding of the reference)
                if constexpr (MT) {
                    if (hn == 0) {
#pragma unroll
                        for (int kw = 0; kw < KW; ++kw)
#pragma unroll
                            for (int kh = 1; kh < KH; ++kh)
#pragma unroll
                                for (int il = 0; il < CL; ++il) win[kw][(ph + KH - kh) % KH][il] = 0.f;
                    }
                }
                // (4) taps of the rows above (all in registers since the previous step) ...
                float acc[C], accb[C];
#pragma unroll
                for (int o = 0; o < C; ++o) { acc[o] = zc[o]; accb[o] = 0.f; }
                auto tap = [&](float (&ac)[C], int kh, int kw, const float (&xs)[CL]) {
                    const int t = kh * KW + kw;
#pragma unroll
                    for (int il = 0; il < CL; ++il) {
                        const float xv = xs[il];
                        if constexpr (WREG) {
#pragma unroll
                            for (int o = 0; o < C; ++o) ac[o] = fmaf(xv, wr[t][il][o], ac[o]);
                        } else if constexpr (CPP % 4 == 0) {
                            const float* wrow = wgp + t * TS + il * P * CPP;
#pragma unroll
                            for (int v = 0; v < CPP / 4; ++v) {
                                const float4 f = *reinterpret_cast<const float4*>(wrow + 4 * v);
                                if (4 * v + 0 < C) ac[4 * v + 0] = fmaf(-xv, f.x, ac[4 * v + 0]);
                                if (4 * v + 1 < C) ac[4 * v + 1] = fmaf(-xv, f.y, ac[4 * v + 1]);
                                if (4 * v + 2 < C) ac[4 * v + 2] = fmaf(-xv, f.z, ac[4 * v + 2]);
                                if (4 * v + 3 < C) ac[4 * v + 3] = fmaf(-xv, f.w, ac[4 * v + 3]);
                            }
                        } else {
                            const float* wrow = wgp + t * TS + il * P * CPP;
#pragma unroll
                            for (int o = 0; o < C; ++o) ac[o] = fmaf(-xv, wrow[o], ac[o]);
                        }
                    }
                };
#pragma unroll
                for (int kh = KH - 1; kh >= 1; --kh)
#pragma unroll
                    for (int kw = KW - 1; kw >= 0; --kw) tap(acc, kh, kw, win[kw][(ph + KH - kh) % KH]);
                // (5) ... then the taps of this row, fed by the shuffles
#pragma unroll
                for (int kw = KW - 1; kw >= 1; --kw) {
#pragma unroll
                    for (int il = 0; il < CL; ++il) win[kw][ph][il] = (j >= kw) ? sh[kw - 1][il] : 0.f;
                    tap(accb, 0, kw, win[kw][ph]);
                }
#pragma unroll
                for (int o = 0; o < C; ++o) acc[o] += accb[o];
                // (6) the P partial sums of the pixel meet
                if constexpr (P > 1) {
#pragma unroll
                    for (int off = LP; off < 32; off <<= 1)
#pragma unroll
                        for (int o = 0; o < C; ++o) acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], off);
                }
                // (7) corner tap: x[o] = acc[o] - sum_{i<o} W[o,i,corner] x[i]
#pragma unroll
                for (int i = 0; i < C - 1; ++i) {
                    if constexpr (CREG) {
#pragma unroll
                        for (int o = i + 1; o < C; ++o) acc[o] = fmaf(-acc[i], wc[i][o], acc[o]);
                    } else if constexpr (CPP % 4 == 0) {
#pragma unroll
                        for (int v = (i + 1) / 4; v < CPP / 4; ++v) {
                            const float4 f = *reinterpret_cast<const float4*>(wg + rv(i) * CPP + 4 * v);
                            if (4 * v + 0 > i && 4 * v + 0 < C) acc[4 * v + 0] = fmaf(-acc[i], f.x, acc[4 * v + 0]);
                            if (4 * v + 1 > i && 4 * v + 1 < C) acc[4 * v + 1] = fmaf(-acc[i], f.y, acc[4 * v + 1]);
                            if (4 * v + 2 > i && 4 * v + 2 < C) acc[4 * v + 2] = fmaf(-acc[i], f.z, acc[4 * v + 2]);
                            if (4 * v + 3 > i && 4 * v + 3 < C) acc[4 * v + 3] = fmaf(-acc[i], f.w, acc[4 * v + 3]);
                        }
                    } else {
#pragma unroll
                        for (int o = i + 1; o < C; ++o) acc[o] = fmaf(-acc[i], wg[rv(i) * CPP + o], acc[o]);
                    }
                }
                // (8) keep this lane's channels in the window; one lane per channel stores
#pragma unroll
                for (int il = 0; il < CL; ++il) {
                    float v = acc[rv(il * P)];
#pragma unroll
                    for (int pp = 1; pp < P; ++pp) v = (p == pp) ? acc[rv(il * P + pp)] : v;
                    win[0][ph][il] = v;
                    if (active) ptr[(il * P + p) * HW] = v;
                }
                ptr = nptr;
                hn = nhn;
#pragma unroll
                for (int o = 0; o < C; ++o) zc[o] = zn[o];
            }
        }
        if (a.n_units > 1) __syncwarp();   // the next unit reads what other lanes stored
        }   // units of the chain

        if (threadIdx.x == 0 && k == 0) dbg_mark(a.dbg, 3);
        if (a.bulk) {
            fence_proxy_async_smem();
            __syncwarp();
            for (int tt = lane; tt < nt; tt += 32)
                bulk_s2g(a.x + ((long)(n0 + tt) * s.G + g) * a.tile_floats, tile_smem(buf, tt),
                         (uint32_t)(a.tile_floats * 4));
            bulk_commit();
            const long nxt = item + (long)a.S * gstride;
            if (nxt < a.n_items) {
                bulk_wait_read_all();   // the stage is reused: its stores must have read it
                __syncwarp();
                issue_load(nxt, st);
            }
        } else {
            __syncwarp();
            for (int tt = 0; tt < nt; ++tt) {
                float* dst = a.x + ((long)(n0 + tt) * s.G + g) * a.tile_floats;
                const float* src = tile_smem(buf, tt);
                for (int e = lane; e < a.tile_floats; e += 32) dst[e] = src[e];
            }
            __syncwarp();
        }
    }
    if (a.bulk) bulk_wait_all();
    if (threadIdx.x == 0) dbg_mark(a.dbg, 4);
}

// the corner weights of the C = 12, P = 1 single-tile adjoint come from the shared-memory table: held in registers
// they spill (24 B; the inverse of that family spills 20 B and keeps them, as before)
template <int C, int P, bool MT, bool ADJ>
constexpr bool creg_of(bool creg) { return creg && !(ADJ && C == 12 && P == 1 && !MT); }

template <int C, int KH, int KW, int P, bool MT, bool ADJ>
__global__ void __launch_bounds__(Cfg<C, KH, KW, P>::MAXW * 32, 1) inverse_rw_kernel(const RwArgs a) {
    using K = Cfg<C, KH, KW, P>;
    inverse_rw_body<C, KH, KW, P, MT, K::WREG, creg_of<C, P, MT, ADJ>(K::CREG), ADJ>(
        a, (int)blockIdx.x, (int)gridDim.x, (int)blockIdx.y);
}

// ---- several levels in one launch (finc_inverse_chain_multi_f32) ------------------------------------------------
// Every level of a stack has independent inputs, and one level's chain leaves most of the GPU idle at small batches
// (a dependent 16-unit x (H+W-1)-step chain per warp, few warps per SM).  One launch hosts the warp items of all
// levels at once: CTA b belongs to the level l with first[l] <= b < first[l+1] and runs the body of its kind.  The
// cap of 2 CTAs x 6 warps per SM (<= 168 registers) is why the C = 6 taps and the C = 12 corner come from the
// shared-memory table here.
constexpr int kRwMultiLevels = kInverseMultiMaxLevels;
constexpr int kRwMultiWarps = 6;    // warps per CTA

struct RwMultiArgs {
    RwArgs lv[kRwMultiLevels];
    int first[kRwMultiLevels + 1];  // CTAs of level l: [first[l], first[l+1]); first[n] = grid size
    int vgrid[kRwMultiLevels];      // CTAs per group slice of level l
    int kind[kRwMultiLevels];       // which body (template argument) solves level l
};

// one (C, K, P) body of the multi-level kernel
template <int C_, int K_, int P_, bool WREG_, bool CREG_>
struct RwKind {
    static constexpr int C = C_, KS = K_, P = P_;
    static constexpr bool WREG = WREG_, CREG = CREG_;
};

template <class K>
__device__ __forceinline__ void run_kind(const RwArgs& a, int vblock, int vgrid, int grp) {
    inverse_rw_body<K::C, K::KS, K::KS, K::P, false, K::WREG, K::CREG, false>(a, vblock, vgrid, grp);
}

template <class K0, class K1, class K2>
__global__ void __launch_bounds__(kRwMultiWarps * 32, 2) inverse_rw_multi_kernel(const RwMultiArgs m) {
    const int b = (int)blockIdx.x;
    int l = 0;
#pragma unroll
    for (int i = 1; i < kRwMultiLevels; ++i) l += b >= m.first[i];
    const int r = b - m.first[l], vg = m.vgrid[l];
    switch (m.kind[l]) {
        case 0: run_kind<K0>(m.lv[l], r % vg, vg, r / vg); break;
        case 1: run_kind<K1>(m.lv[l], r % vg, vg, r / vg); break;
        default: run_kind<K2>(m.lv[l], r % vg, vg, r / vg); break;
    }
}

// the kinds instantiated: the levels of cifar10_levels / imagenet32_levels at k = 3 ([12,16,16], [24,8,8], [48,4,4];
// C = 3, 6, 12 per group) with the P the per-level planner picks for them
using RwKind0 = RwKind<3, 3, 1, true, true>;
using RwKind1 = RwKind<6, 3, 2, false, true>;
using RwKind2 = RwKind<12, 3, 4, false, false>;
int launch_multi(const RwMultiArgs& m, int n_ctas, size_t smem, cudaStream_t st);   // finc_inverse_rw_multi.cu
int multi_ctas_per_sm(size_t smem);   // CTAs of the multi-level kernel one SM holds with `smem` bytes each (0 on error)

template <int C, int KH, int KW, int P, bool ADJ>
int launch_inst(const RwArgs& a, dim3 grid, int nwarps, size_t smem, cudaStream_t st) {
    if (a.T > 1) {
        auto kern = inverse_rw_kernel<C, KH, KW, P, true, ADJ>;
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        return launch_kernel(kern, grid, nwarps * 32, smem, st, a);
    }
    auto kern = inverse_rw_kernel<C, KH, KW, P, false, ADJ>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    return launch_kernel(kern, grid, nwarps * 32, smem, st, a);
}

// (C, K, P) combinations that are instantiated: the window must fit the register file
constexpr bool rw_supported(int C, int KH, int KW, int P) {
    if (C % P != 0) return false;
    if (KH * KW * (C / P) > (KH == 3 ? 110 : 80)) return false;
    if (C <= 3 && P > 1) return false;
    if (C == 4 && P > 2) return false;
    if (C >= 12 && P == 2) return false;   // 1 and 4 cover the small- and large-batch regimes
    if (C > 12) return false;
    return true;
}
constexpr int rw_max_warps(int C, int KH, int KW, int P) {
    const int CL = C / P, NT = KH * KW - 1, WIN = KH * KW * CL, WREGS = C * CL * NT, CORNER = C * (C - 1) / 2;
    const bool WREG = WREGS <= 150;
    const bool CREG = CORNER + WIN + (WREG ? WREGS : 0) + C <= 200;
    const int EST = WIN + C + (WREG ? WREGS : 16) + (CREG ? CORNER : 8) + 30;
    return EST <= 100 ? 16 : 8;
}

template <int C, int KH, int KW, bool ADJ>
int dispatch_p(int P, const RwArgs& a, dim3 grid, int nwarps, size_t smem, cudaStream_t st) {
    if constexpr (rw_supported(C, KH, KW, 1)) { if (P == 1) return launch_inst<C, KH, KW, 1, ADJ>(a, grid, nwarps, smem, st); }
    if constexpr (rw_supported(C, KH, KW, 2)) { if (P == 2) return launch_inst<C, KH, KW, 2, ADJ>(a, grid, nwarps, smem, st); }
    if constexpr (rw_supported(C, KH, KW, 4)) { if (P == 4) return launch_inst<C, KH, KW, 4, ADJ>(a, grid, nwarps, smem, st); }
    if constexpr (rw_supported(C, KH, KW, 8)) { if (P == 8) return launch_inst<C, KH, KW, 8, ADJ>(a, grid, nwarps, smem, st); }
    return FINC_E_UNSUPPORTED;
}

// explicitly instantiated in finc_inverse_rw_c<N>k<K>.cu (inverse) and finc_inverse_rw_adj_c<N>k<K>.cu (adjoint)
// so the instantiations compile in parallel
template <int C, int KS, bool ADJ = false>
int dispatch_ck(int P, const RwArgs& a, dim3 grid, int nwarps, size_t smem, cudaStream_t st) {
    return dispatch_p<C, KS, KS, ADJ>(P, a, grid, nwarps, smem, st);
}

}  // namespace rw
}  // namespace finc

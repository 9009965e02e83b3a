// finc_inverse_rw.cu -- host-side planning for the register-window wavefront inverse
// (kernel: finc_inverse_rw.cuh; instantiations: finc_inverse_rw_c<N>k<K>.cu, adjoint: finc_inverse_rw_adj_c<N>k<K>.cu).
#include "finc_inverse_rw.cuh"

#include <cstdlib>

namespace finc {

namespace rw {
#define FINC_RW_EXTERN(C)                                                                                   \
    extern template int dispatch_ck<C, 3>(int, const RwArgs&, dim3, int, size_t, cudaStream_t);             \
    extern template int dispatch_ck<C, 5>(int, const RwArgs&, dim3, int, size_t, cudaStream_t);             \
    extern template int dispatch_ck<C, 3, true>(int, const RwArgs&, dim3, int, size_t, cudaStream_t);       \
    extern template int dispatch_ck<C, 5, true>(int, const RwArgs&, dim3, int, size_t, cudaStream_t);
FINC_RW_EXTERN(1)
FINC_RW_EXTERN(2)
FINC_RW_EXTERN(3)
FINC_RW_EXTERN(4)
FINC_RW_EXTERN(6)
FINC_RW_EXTERN(12)
#undef FINC_RW_EXTERN
}  // namespace rw

using rw::RwArgs;

namespace {
int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return (e && *e) ? atoi(e) : dflt;
}
}  // namespace

bool rw_shape_supported(const Shape& s) {
    if (!((s.kH == 3 && s.kW == 3) || (s.kH == 5 && s.kW == 5))) return false;
    const int C = s.C;
    // (C = 24 stays on the shared-memory wavefront kernel: its 276-term corner solve, run redundantly
    //  by the 8 lanes of a pixel, makes the register-window variant slower -- tools/ab_inverse.py)
    if (!(C == 1 || C == 2 || C == 3 || C == 4 || C == 6 || C == 12)) return false;
    if (s.W > 32 || (long)C * s.H * s.W * 4 > 32 * 1024) return false;
    int WP = 4;
    while (WP < s.W) WP *= 2;
    // some instantiated P must fit the warp
    if (s.kH == 5 && C == 4 && WP > 16) return false;   // 5x5, C = 4: P = 2 only
    if (s.kH == 5 && C == 12 && WP > 8) return false;   // 5x5, C = 12: P = 4 only
    if (s.kH == 5 && C == 6 && WP > 16) return false;   // 5x5, C = 6: P >= 2
    return true;
}

// FINC_RW=0 disables the kernel (A/B runs against the shared-memory wavefront kernel)
int launch_inverse_rw(const float* z, const float* w, float* x, const Shape& s, bool prepared, cudaStream_t st,
                      bool* handled) {
    return launch_inverse_rw_chain(z, w, x, s, prepared, 1, 0, 1, 0, st, handled);
}

namespace {
// what the per-level planner picks for one launch of the kernel
struct RwPlan {
    RwArgs a;
    int P, nwarps;
    dim3 grid;
    size_t smem, wk_bytes, stage_bytes;
};

// plans one level's launch; *planned = false (rc 0) when the register-window kernel does not cover it
int plan_inverse_rw(const float* z, const float* w, float* x, const Shape& s, bool prepared, int n_units, int u_first,
                    int u_step, long unit_stride, RwPlan& plan, bool* planned) {
    *planned = false;
    if (n_units > 1 && !prepared) return FINC_E_UNSUPPORTED;
    static const int enabled = env_int("FINC_RW", 1);
    if (!enabled) return 0;
    if (!((s.kH == 3 && s.kW == 3) || (s.kH == 5 && s.kW == 5))) return 0;
    const int C = s.C, KS = s.kH;
    if (!rw_shape_supported(s)) return 0;
    const long tile_floats_l = (long)C * s.H * s.W;
    RwArgs a{};
    a.z = z; a.w = w; a.x = x; a.s = s; a.dbg = debug_ts_buffer(); a.prepared = prepared ? 1 : 0;
    a.n_units = n_units; a.u_first = u_first; a.u_step = u_step; a.unit_stride = unit_stride;
    a.tile_floats = (int)tile_floats_l;
    a.tile_stride = (a.tile_floats + 3) & ~3;
    const int CPP = C <= 2 ? C : ((C + 3) / 4) * 4;
    const int tap_stride = (C <= 2) ? C * CPP : (((C * CPP / 4) % 2 == 1) ? C * CPP : C * CPP + 4);
    const size_t wk_per_g = (size_t)s.kH * s.kW * tap_stride;
    const size_t smem_max = max_optin_smem_cached();
    const size_t budget = smem_max > 8192 ? smem_max - 4096 : 0;
    if (wk_per_g * s.G * 4 * n_units <= budget / 2) { a.gsplit = 0; a.wk_floats = (int)(wk_per_g * s.G); }
    else if (wk_per_g * 4 * n_units <= budget / 2) { a.gsplit = 1; a.wk_floats = (int)wk_per_g; }
    else return n_units > 1 ? FINC_E_UNSUPPORTED : 0;
    a.bulk = (a.tile_floats % 4 == 0) && ((reinterpret_cast<uintptr_t>(z) & 15) == 0) &&
             ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
    if (prepared && (!a.bulk || (reinterpret_cast<uintptr_t>(w) & 15) != 0 || wave_prepared_floats(s) == 0))
        return FINC_E_UNSUPPORTED;

    int WP = 4;
    while (WP < s.W) WP *= 2;
    a.WP = WP;
    const int sms = sm_count_cached();
    const long ctas_max = a.gsplit ? (sms / s.G > 0 ? sms / s.G : 1) : sms;
    const long tiles = a.gsplit ? s.B : (long)s.B * s.G;   // per blockIdx.y slice

    // parts per pixel: the smallest instantiated P that still gives every SM sub-partition a warp
    // (small batches split the input channels of a pixel over more lanes; large batches do not)
    int cand[4], nc = 0;
    for (int P = 1; P <= 8; P *= 2) {
        if (P * WP > 32) break;
        bool ok = false;
        switch (C) {
            case 1: ok = rw::rw_supported(1, KS, KS, P); break;
            case 2: ok = rw::rw_supported(2, KS, KS, P); break;
            case 3: ok = rw::rw_supported(3, KS, KS, P); break;
            case 4: ok = rw::rw_supported(4, KS, KS, P); break;
            case 6: ok = rw::rw_supported(6, KS, KS, P); break;
            default: ok = rw::rw_supported(12, KS, KS, P); break;
        }
        if (ok) cand[nc++] = P;
    }
    if (nc == 0) return prepared ? FINC_E_UNSUPPORTED : 0;
    int P = cand[nc - 1];
    for (int i = 0; i < nc; ++i) {
        const long warps = tiles * WP * cand[i] / 32;
        if (warps >= ctas_max * 4) { P = cand[i]; break; }
    }
    if (C == 6 && KS == 3 && nc > 1 && P == 1) P = 2;  // P = 2 keeps the C = 6 weights in registers
    // FINC_RW_P / _NSTK / _T / _S / _WARPS (experiment and test knobs, read per call) pin parts of the plan; a value
    // outside what the planner itself could choose is ignored, so a knob never addresses lanes or shared memory the
    // kernel does not own
    {
        const int fp = env_int("FINC_RW_P", 0);
        for (int i = 0; i < nc; ++i)
            if (cand[i] == fp) P = fp;
    }
    // stacks per warp: all 32/(WP*P) lanes groups when the batch can fill the SMs, fewer (idle lanes,
    // more warps) when it cannot
    int NSTK = 32 / (WP * P);
    while (NSTK > 1 && tiles / NSTK < ctas_max * 2) NSTK /= 2;   // (x4 was measured slower at batch 256)
    {
        const int fn = env_int("FINC_RW_NSTK", 0);   // a power of two whose stacks fit the warp
        if (fn >= 1 && (fn & (fn - 1)) == 0 && fn * WP * P <= 32) NSTK = fn;
    }
    a.NSTK = NSTK;
    const int maxw_k = rw::rw_max_warps(C, KS, KS, P);
    const int fw = env_int("FINC_RW_WARPS", 0);
    const int maxw = (fw >= 1 && fw < maxw_k) ? fw : maxw_k;

    const size_t wk_bytes = (size_t)((a.wk_floats + 31) & ~31) * 4 * n_units;
    const size_t avail = budget - wk_bytes;
    const int skew = NSTK > 1 ? 32 / NSTK : 0;   // stacks of a warp land on disjoint banks
    auto stage_bytes_of = [&](int T) { return (size_t)NSTK * ((size_t)T * a.tile_stride + skew) * 4; };
    // stack depth: 1 while the batch cannot even fill the warps; deeper stacks keep the skewed
    // wavefront busy (a lone HxW tile uses H/(H+W-1) of the lane-steps)
    int T = 1;
    while (T < 8) {
        const int T2 = T * 2;
        const long items2 = (tiles + (long)NSTK * T2 - 1) / ((long)NSTK * T2);
        if (items2 < ctas_max * maxw * 2) break;
        if (stage_bytes_of(T2) * maxw + 64 > avail && stage_bytes_of(T2) * 8 + 64 > avail) break;
        T = T2;
    }
    {
        const int ft = env_int("FINC_RW_T", 0);
        if (ft == 1 || ft == 2 || ft == 4 || ft == 8) T = ft;
    }
    a.T = T;
    a.stack_stride = T * a.tile_stride + skew;
    const size_t stage_bytes = stage_bytes_of(T);
    const long n_blocks = (s.B + (long)NSTK * T - 1) / ((long)NSTK * T);
    a.n_items = a.gsplit ? n_blocks : n_blocks * s.G;
    long ctas = ctas_max;
    if (ctas > a.n_items) ctas = a.n_items;
    const long items_per_cta = (a.n_items + ctas - 1) / ctas;
    int nwarps = (int)(items_per_cta < maxw ? items_per_cta : maxw);
    a.S = 1;
    if ((size_t)nwarps * (stage_bytes + 8) + 64 > avail) nwarps = (int)((avail - 64) / (stage_bytes + 8));
    if (nwarps < 1) return prepared ? FINC_E_UNSUPPORTED : 0;
    // a second stage only pays when warps loop over several items and memory is left
    if (items_per_cta > nwarps && (size_t)nwarps * 2 * (stage_bytes + 8) + 64 <= avail) a.S = 2;
    {
        const int fs = env_int("FINC_RW_S", 0);
        if (fs == 1 || fs == 2) a.S = fs;
    }
    const size_t smem = wk_bytes + (size_t)nwarps * a.S * (stage_bytes + 8) + 8 + 16;
    if (smem > budget + 2048) return prepared ? FINC_E_UNSUPPORTED : 0;
    plan.a = a;
    plan.P = P;
    plan.nwarps = nwarps;
    plan.grid = dim3((unsigned)ctas, a.gsplit ? s.G : 1, 1);
    plan.smem = smem;
    plan.wk_bytes = wk_bytes;
    plan.stage_bytes = stage_bytes;
    *planned = true;
    return 0;
}

// the instantiation of the planned (C, K) family
template <bool ADJ>
int dispatch_plan(const RwPlan& plan, const Shape& s, cudaStream_t st) {
    const RwArgs& a = plan.a;
    const int P = plan.P, nwarps = plan.nwarps;
    const dim3 grid = plan.grid;
    const size_t smem = plan.smem;
    if (s.kH == 3) {
        switch (s.C) {
            case 1: return rw::dispatch_ck<1, 3, ADJ>(P, a, grid, nwarps, smem, st);
            case 2: return rw::dispatch_ck<2, 3, ADJ>(P, a, grid, nwarps, smem, st);
            case 3: return rw::dispatch_ck<3, 3, ADJ>(P, a, grid, nwarps, smem, st);
            case 4: return rw::dispatch_ck<4, 3, ADJ>(P, a, grid, nwarps, smem, st);
            case 6: return rw::dispatch_ck<6, 3, ADJ>(P, a, grid, nwarps, smem, st);
            default: return rw::dispatch_ck<12, 3, ADJ>(P, a, grid, nwarps, smem, st);
        }
    }
    switch (s.C) {
        case 1: return rw::dispatch_ck<1, 5, ADJ>(P, a, grid, nwarps, smem, st);
        case 2: return rw::dispatch_ck<2, 5, ADJ>(P, a, grid, nwarps, smem, st);
        case 3: return rw::dispatch_ck<3, 5, ADJ>(P, a, grid, nwarps, smem, st);
        case 4: return rw::dispatch_ck<4, 5, ADJ>(P, a, grid, nwarps, smem, st);
        case 6: return rw::dispatch_ck<6, 5, ADJ>(P, a, grid, nwarps, smem, st);
        default: return rw::dispatch_ck<12, 5, ADJ>(P, a, grid, nwarps, smem, st);
    }
}
}  // namespace

// n_units > 1: a chain of units solved in place in one launch (prepared tables, unit u at w + u * unit_stride)
int launch_inverse_rw_chain(const float* z, const float* w, float* x, const Shape& s, bool prepared, int n_units,
                            int u_first, int u_step, long unit_stride, cudaStream_t st, bool* handled) {
    *handled = false;
    RwPlan plan;
    bool planned = false;
    int rc = plan_inverse_rw(z, w, x, s, prepared, n_units, u_first, u_step, unit_stride, plan, &planned);
    if (rc || !planned) return rc;
    rc = dispatch_plan<false>(plan, s, st);
    if (rc == FINC_E_UNSUPPORTED) return prepared ? FINC_E_UNSUPPORTED : 0;
    *handled = true;
    return rc;
}

// The adjoint solve dz = A^-T dx (`s.orders` already flipped by the caller): the launch the inverse of the same shape
// would make -- same plan, same P, NSTK, T -- of the ADJ instantiation.  *handled = false when the shape is not covered.
int launch_inverse_rw_adjoint(const float* dx, const float* w, float* dz, const Shape& s, cudaStream_t st,
                              bool* handled) {
    *handled = false;
    RwPlan plan;
    bool planned = false;
    int rc = plan_inverse_rw(dx, w, dz, s, false, 1, 0, 1, 0, plan, &planned);
    if (rc || !planned) return rc;
    rc = dispatch_plan<true>(plan, s, st);
    if (rc == FINC_E_UNSUPPORTED) return 0;
    *handled = true;
    return rc;
}

// The sampling chains of several levels in ONE launch of inverse_rw_multi_kernel.  Every level keeps the P, NSTK and T
// its own launch would use (so every tile sees the same arithmetic, bit for bit); its CTAs of 6 warps are sized so
// that each warp solves at most one item, and the launch is refused unless all CTAs are resident at once.
int launch_inverse_rw_multi(const RwChainLevel* lv, int n, cudaStream_t st) {
    if (n < 1 || n > rw::kRwMultiLevels) return FINC_E_UNSUPPORTED;
    rw::RwMultiArgs m{};
    constexpr int NW = rw::kRwMultiWarps;
    size_t smem = 0;
    int ctas = 0, nl = 0;
    for (int i = 0; i < n; ++i) {
        const RwChainLevel& c = lv[i];
        if (c.s.B == 0) continue;
        RwPlan plan;
        bool planned = false;
        const int rc = plan_inverse_rw(c.z, c.w, c.x, c.s, true, c.n_units, c.u_first, c.u_step, c.unit_stride, plan,
                                       &planned);
        if (rc || !planned) return FINC_E_UNSUPPORTED;
        const int C = c.s.C, KS = c.s.kH, P = plan.P;
        int kind = -1;
        if (C == rw::RwKind0::C && KS == rw::RwKind0::KS && P == rw::RwKind0::P) kind = 0;
        if (C == rw::RwKind1::C && KS == rw::RwKind1::KS && P == rw::RwKind1::P) kind = 1;
        if (C == rw::RwKind2::C && KS == rw::RwKind2::KS && P == rw::RwKind2::P) kind = 2;
        if (kind < 0 || plan.a.T != 1) return FINC_E_UNSUPPORTED;   // (multi-tile stacks: not instantiated)
        RwArgs a = plan.a;
        a.S = 1;
        const long vgrid = (a.n_items + NW - 1) / NW;
        const long lctas = vgrid * plan.grid.y;
        m.lv[nl] = a;
        m.kind[nl] = kind;
        m.vgrid[nl] = (int)vgrid;
        m.first[nl] = ctas;
        ctas += (int)lctas;
        const size_t need = plan.wk_bytes + (size_t)NW * (plan.stage_bytes + 8) + 8 + 16;
        if (need > smem) smem = need;
        ++nl;
    }
    if (nl == 0) return 0;
    for (int i = nl; i <= rw::kRwMultiLevels; ++i) m.first[i] = ctas;
    if (smem > max_optin_smem_cached()) return FINC_E_UNSUPPORTED;
    if (ctas > (long)rw::multi_ctas_per_sm(smem) * sm_count_cached()) return FINC_E_UNSUPPORTED;
    return rw::launch_multi(m, ctas, smem, st);
}

}  // namespace finc

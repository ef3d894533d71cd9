// Generation-2 per-thread code of the two Chambolle-Pock passes: instruction-lean "strip" form.
//
// Why: generation 1 (tv_core.cuh, one quad per thread) moved exactly the algorithmic bytes but spent ~1300
// instructions per quad (IEEE divisions, 64-bit block decode, a 64-bit address computation and a boundary
// predicate per neighbour load) and ran at 62 % (pass A) / 82 % (pass B) of the measured HBM peak with the
// issue slots 50-60 % busy (profiles/r01a_gen1_cp_ncu_full.txt).  Here:
//   * everything that depends only on (z, t) - plane base pointers of the centre and of the z / t
//     neighbours, weights, boundary factors - is computed once per CTA and is warp-uniform;
//   * a thread walks R consecutive rows of one quad column and addresses every array as
//     `uniform plane pointer + 32-bit element offset`;
//   * neighbours that do not exist are CLAMPED to the centre, which makes the difference exactly zero
//     (x[k] - x[k] = 0: the reference's "out-of-range difference is zero" rule, tv_operators_CPU.py:118)
//     without a predicate; only the centred scheme needs 0/1 factors;
//   * the projection uses one rsqrt: scale = min(1, lam * rsqrt(|y|^2)); no division.
// The functions are __host__ __device__ (plain loads only) so tests/emul runs them on the CPU too.
#pragma once
#include <cuda_fp16.h>

#include "core.cuh"

namespace pytvb {

PYTVB_HD float fast_rsqrt(float a) {
#if defined(__CUDA_ARCH__)
    return rsqrtf(a);            // MUFU.RSQ + one fix-up, ~2 ulp
#else
    return 1.0f / sqrtf(a);
#endif
}
PYTVB_HD double fast_rsqrt(double a) { return 1.0 / sqrt(a); }
PYTVB_HD float fast_sqrt(float a) {
#if defined(__CUDA_ARCH__)
    float r;
    asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(a));   // MUFU.SQRT, no IEEE slow path (feeds a sum of 1e8+ terms)
    return r;
#else
    return sqrtf(a);
#endif
}
PYTVB_HD double fast_sqrt(double a) { return sqrt(a); }

// Loads / stores of the dual field y, which may be STORED in a narrower type than the arithmetic type T
// (YT = __half: SURVEY 8f-4, halves the dominant Nd*V traffic; values are kept normalised to the unit ball so
// that half precision's 11 significant bits cover them uniformly).
template <typename T, typename YT, int VEC>
PYTVB_HD void ld_y(T* dst, const YT* src) {
    const Pack<YT, VEC> p = ld_pack<YT, VEC>(src);
#pragma unroll
    for (int e = 0; e < VEC; ++e) dst[e] = (T)p.v[e];
}
template <typename T, typename YT, int VEC>
PYTVB_HD void st_y(YT* dst, const T* v) {
    Pack<YT, VEC> p;
#pragma unroll
    for (int e = 0; e < VEC; ++e) p.v[e] = (YT)v[e];
    st_pack<YT, VEC>(dst, p);
}

// Streaming store (st.global.cs) for outputs that the kernel never reads back: +3 % on the write-dominated D kernel
// (3.26 -> 3.16 ms on the C4 slab).
template <typename T, int VEC>
PYTVB_HD void st_pack_stream(T* p, const Pack<T, VEC>& v) {
#if defined(__CUDA_ARCH__)
    if constexpr (sizeof(T) == 4 && VEC == 4) { __stcs(reinterpret_cast<float4*>(p), *reinterpret_cast<const float4*>(&v)); return; }
    if constexpr (sizeof(T) == 8 && VEC == 2) { __stcs(reinterpret_cast<double2*>(p), *reinterpret_cast<const double2*>(&v)); return; }
#endif
    st_pack<T, VEC>(p, v);
}

// Warp-uniform context of one (z, t) image plane for the dual pass.
template <typename T, typename YT = T>
struct DualPlane {
    const T* c;                       // plane (z, t) of xbar
    const T* zm; const T* zp;         // planes (z-1, t), (z+1, t): clamped to c at the volume boundary, halo planes at slab edges
    const T* tm; const T* tp;         // planes (z, t-1), (z, t+1), clamped
    YT* y;                            // component 0 of y at plane (z, t); component k at + k*sC
    T fz, ft;                         // centred scheme only: 1 where the centred z / t difference exists, else 0
    const T* ts;                      // plane (z, t) of the per-voxel time scale, or null
};

template <typename T, int SCHEME, typename YT = T>
PYTVB_HD DualPlane<T, YT> make_dual_plane(const ImgView<T>& X, YT* y, const Params<T>& P, int z, int t) {
    DualPlane<T, YT> d;
    const long long zg = P.zg0 + z;
    const bool v_zm = zg > 0, v_zp = zg < P.NzG - 1, v_tm = t > 0, v_tp = t < P.M - 1;
    d.c = X.row(P, z, t, 0);
    d.zm = v_zm ? X.row(P, z - 1, t, 0) : d.c;
    d.zp = v_zp ? X.row(P, z + 1, t, 0) : d.c;
    d.tm = v_tm ? X.row(P, z, t - 1, 0) : d.c;
    d.tp = v_tp ? X.row(P, z, t + 1, 0) : d.c;
    d.y = y + (long long)z * P.sZf + (long long)t * P.sT;
    d.fz = d.ft = T(1);
    d.ts = (P.tscale && z >= 0 && z < P.Nz) ? P.tscale + (long long)z * P.sZ + (long long)t * P.sT : nullptr;
    if (SCHEME == CENTRAL) {
        // centred difference exists iff both neighbours do; on a length-2 axis it degrades to the forward
        // difference (minus pointer := centre, the clamped plus pointer already gives 0 on the last plane)
        if (P.z_fwd_fallback) d.zm = d.c; else d.fz = (v_zm && v_zp) ? T(1) : T(0);
        if (P.t_fwd_fallback) d.tm = d.c; else d.ft = (v_tm && v_tp) ? T(1) : T(0);
    }
    return d;
}

// Factor of the time component(s) at a quad: sqrt(factor_reg_static) on static pixels (tv_operators_CPU.py:148-150)
// times the per-voxel time scale, if any (extension: the reference's TODO README.md:258).
template <typename T, int VEC>
PYTVB_HD void time_factor(T* f, const Params<T>& P, const T* ts_plane, int i, int j0, int o) {
    static_factor<T, VEC>(f, P, i, j0);
    if (ts_plane) {
        const Pack<T, VEC> sc = ld_pack<T, VEC>(ts_plane + o);
#pragma unroll
        for (int e = 0; e < VEC; ++e) f[e] *= sc.v[e];
    }
}
template <typename T, int VEC>
PYTVB_HD void scale_by(T* v, const T* ts_plane, int o) {
    if (ts_plane) {
        const Pack<T, VEC> sc = ld_pack<T, VEC>(ts_plane + o);
#pragma unroll
        for (int e = 0; e < VEC; ++e) v[e] *= sc.v[e];
    }
}

// Raw differences of one quad: d[k][e] = weight * (x[k+1] - x[k]) etc. WITHOUT the scheme's global divisor.
// o = i*Nj + j0; o_up / o_dn = offsets of rows i-1 / i+1 clamped to [0, Ni).
// (TS = a per-voxel time scale is present.  It is a template parameter all the way up to the kernels: folding the null
// checks into the common body cost pass B 12 %, and even two variants behind one uniform branch inside one kernel cost
// 7 % (register pressure), so the no-weight-map kernels are kept bit-identical to what they were before the extension.)
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, typename YT, bool TS>
PYTVB_HD void strip_raw_diffs_impl(T (*d)[VEC], const DualPlane<T, YT>& pl, const Params<T>& P, int i, int j0, int o, int o_up, int o_dn) {
    typedef Comp<SCHEME, Z_ON, T_ON> C;
    T c[VEC + 2], up[VEC], dn[VEC], zm[VEC], zp[VEC], tm[VEC], tp[VEC];
    ld_into<T, VEC>(c + 1, pl.c + o);
    c[0] = (C::NEED_BWD && j0 > 0) ? pl.c[o - 1] : c[1];
    c[VEC + 1] = (C::NEED_FWD && j0 + VEC < P.Nj) ? pl.c[o + VEC] : c[VEC];
    if (C::NEED_BWD) ld_into<T, VEC>(up, pl.c + o_up);
    if (C::NEED_FWD) ld_into<T, VEC>(dn, pl.c + o_dn);
    if (Z_ON && C::NEED_BWD) ld_into<T, VEC>(zm, pl.zm + o);
    if (Z_ON && C::NEED_FWD) ld_into<T, VEC>(zp, pl.zp + o);
    if (T_ON && C::NEED_BWD) ld_into<T, VEC>(tm, pl.tm + o);
    if (T_ON && C::NEED_FWD) ld_into<T, VEC>(tp, pl.tp + o);
    T fac[VEC];
    if (T_ON) { if constexpr (TS) time_factor<T, VEC>(fac, P, pl.ts, i, j0, o); else static_factor<T, VEC>(fac, P, i, j0); }
    // centred scheme: in-plane factors (rows: uniform per row; columns: only the volume's first / last column)
    const T fi = (SCHEME == CENTRAL) ? ((i > 0 && i < P.Ni - 1) ? T(1) : T(0)) : T(1);
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
        const T x = c[e + 1];
        if (SCHEME == HYBRID) {
            d[C::I_F][e] = dn[e] - x;
            d[C::J_F][e] = c[e + 2] - x;
            d[C::I_B][e] = x - up[e];
            d[C::J_B][e] = x - c[e];
            if (Z_ON) { d[C::Z_F][e] = P.srz * (zp[e] - x); d[C::Z_B][e] = P.srz * (x - zm[e]); }
            if (T_ON) { const T w = P.srt * fac[e]; d[C::T_F][e] = w * (tp[e] - x); d[C::T_B][e] = w * (x - tm[e]); }
        } else if (SCHEME == UPWIND) {
            d[0][e] = dn[e] - x;
            d[1][e] = c[e + 2] - x;
            if (Z_ON) d[C::Z_F][e] = P.srz * (zp[e] - x);
            if (T_ON) d[C::T_F][e] = P.srt * fac[e] * (tp[e] - x);
        } else if (SCHEME == DOWNWIND) {
            d[0][e] = x - up[e];
            d[1][e] = x - c[e];
            if (Z_ON) d[C::Z_F][e] = P.srz * (x - zm[e]);
            if (T_ON) d[C::T_F][e] = P.srt * fac[e] * (x - tm[e]);
        } else {
            const int j = j0 + e;
            const T fj = (j > 0 && j < P.Nj - 1) ? T(1) : T(0);
            d[0][e] = fi * (dn[e] - up[e]);
            d[1][e] = fj * (c[e + 2] - c[e]);
            if (Z_ON) d[C::Z_F][e] = (P.srz * pl.fz) * (zp[e] - zm[e]);
            if (T_ON) d[C::T_F][e] = (P.srt * pl.ft * fac[e]) * (tp[e] - tm[e]);
        }
    }
}

template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, typename YT = T, bool TS = false>
PYTVB_HD void strip_raw_diffs(T (*d)[VEC], const DualPlane<T, YT>& pl, const Params<T>& P, int i, int j0, int o, int o_up, int o_dn) {
    strip_raw_diffs_impl<T, VEC, SCHEME, Z_ON, T_ON, YT, TS && T_ON>(d, pl, P, i, j0, o, o_up, o_dn);
}

// One quad of the dual pass.  sig = sigma * inv_div (so that y + sigma*D = y + sig*raw_difference).
// Returns sum_e sqrt(sum_k raw_k^2) (the caller multiplies the total by inv_div to get L21(D xbar)).
// Peer-memory halo push (multi-GPU, opt-in): the boundary planes a neighbouring rank will read as its halos are
// stored a second time, straight into that rank's halo buffer (a peer-mapped pointer over NVLink), by the kernel that
// produces them - no separate exchange step.  `prev` / `next`: plane (t) of the buffer in the previous / next rank,
// or null.  MIR is a kernel-level template parameter so that the single-GPU kernels stay untouched.
template <typename YT>
struct MirrorPlanes {
    YT* prev;
    YT* next;
};

// Peer halo buffers of the two z-neighbours (one (M, Ni, Nj) plane each), or null: see MirrorPlanes.
template <typename YT>
struct MirrorBufs {
    YT* prev;
    YT* next;
};
template <typename YT, typename PT>
PYTVB_HD MirrorPlanes<YT> mirror_planes(const MirrorBufs<YT>& m, const PT& P, int z, int t) {
    MirrorPlanes<YT> r;
    r.prev = (m.prev && z == 0) ? m.prev + (long long)t * P.sT : nullptr;
    r.next = (m.next && z == P.Nz - 1) ? m.next + (long long)t * P.sT : nullptr;
    return r;
}
// strip_quad_cp_dual that also leaves the new y of the quad in `y` (the dual pass that finishes part of the adjoint).
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, typename YT, bool TS, bool MIR>
PYTVB_HD T strip_quad_cp_dual_y(T (*y)[VEC], const DualPlane<T, YT>& pl, const Params<T>& P, int i, int j0, int o, int o_up, int o_dn, T sig, T lam,
                                MirrorPlanes<YT> mir) {
    typedef Comp<SCHEME, Z_ON, T_ON> C;
    constexpr int ND = C::ND;
    T d[ND][VEC];
#pragma unroll
    for (int k = 0; k < ND; ++k) ld_y<T, YT, VEC>(y[k], pl.y + (long long)k * P.sC + o);
    strip_raw_diffs<T, VEC, SCHEME, Z_ON, T_ON, YT, TS>(d, pl, P, i, j0, o, o_up, o_dn);
    T l21 = T(0);
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
        T s = T(0), sd = T(0);
#pragma unroll
        for (int k = 0; k < ND; ++k) {
            sd += d[k][e] * d[k][e];
            y[k][e] += sig * d[k][e];
            s += y[k][e] * y[k][e];
        }
        l21 += fast_sqrt(sd);
        // y / max(1, |y|/lam)  ==  y * min(1, lam / |y|);  |y| = 0 gives rsqrt = inf -> min = 1
        const T r = lam * fast_rsqrt(s);
        const T scale = r < T(1) ? r : T(1);   // a NaN (lam = 0 and y = 0) falls through to 1
#pragma unroll
        for (int k = 0; k < ND; ++k) y[k][e] *= scale;
    }
#pragma unroll
    for (int k = 0; k < ND; ++k) st_y<T, YT, VEC>(pl.y + (long long)k * P.sC + o, y[k]);
    if constexpr (MIR && Z_ON) {
        // the previous rank's adjoint reads my backward-type z slot of my first plane, the next rank's my forward-type
        // slot of my last plane (see pytvb_DT)
        if (mir.prev) st_y<T, YT, VEC>(mir.prev + o, y[C::Z_B]);
        if (mir.next) st_y<T, YT, VEC>(mir.next + o, y[C::Z_F]);
    }
    return l21;
}
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, typename YT = T, bool TS = false, bool MIR = false>
PYTVB_HD T strip_quad_cp_dual(const DualPlane<T, YT>& pl, const Params<T>& P, int i, int j0, int o, int o_up, int o_dn, T sig, T lam,
                              MirrorPlanes<YT> mir = MirrorPlanes<YT>{nullptr, nullptr}) {
    T y[Comp<SCHEME, Z_ON, T_ON>::ND][VEC];
    return strip_quad_cp_dual_y<T, VEC, SCHEME, Z_ON, T_ON, YT, TS, MIR>(y, pl, P, i, j0, o, o_up, o_dn, sig, lam, mir);
}

// D_scheme at one quad, stored to the field plane `out` (component 0 of plane (z,t); component k at + k*sC).
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, bool TS = false>
PYTVB_HD void strip_quad_D(T* out, const DualPlane<T>& pl, const Params<T>& P, int i, int j0, int o, int o_up, int o_dn) {
    typedef Comp<SCHEME, Z_ON, T_ON> C;
    T d[C::ND][VEC];
    strip_raw_diffs<T, VEC, SCHEME, Z_ON, T_ON, T, TS>(d, pl, P, i, j0, o, o_up, o_dn);
#pragma unroll
    for (int k = 0; k < C::ND; ++k) {
        Pack<T, VEC> pk;
#pragma unroll
        for (int e = 0; e < VEC; ++e) pk.v[e] = d[k][e] * P.inv_div;
        st_pack_stream<T, VEC>(out + (long long)k * P.sC + o, pk);
    }
}

// TV sweep 1 at one quad: w = 1/|D x| (0 where the norm is 0) into `w_plane`, optional norms (inf where 0)
// into `n_plane`; returns the sum of the norms.  |D x| = inv_div * sqrt(sum raw^2).
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, bool TS = false>
PYTVB_HD T strip_quad_tv_norm(T* w_plane, T* n_plane, const DualPlane<T>& pl, const Params<T>& P, int i, int j0, int o, int o_up, int o_dn) {
    typedef Comp<SCHEME, Z_ON, T_ON> C;
    T d[C::ND][VEC];
    strip_raw_diffs<T, VEC, SCHEME, Z_ON, T_ON, T, TS>(d, pl, P, i, j0, o, o_up, o_dn);
    Pack<T, VEC> w, n;
    T sum = T(0);
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
        T s = T(0);
#pragma unroll
        for (int k = 0; k < C::ND; ++k) s += d[k][e] * d[k][e];
        const T rs = fast_rsqrt(s);                 // inf for s == 0
        const T nr = s > T(0) ? s * rs * P.inv_div : T(0);
        w.v[e] = s > T(0) ? rs * P.div : T(0);
        n.v[e] = s > T(0) ? nr : T(INFINITY);
        sum += nr;
    }
    if (w_plane) st_pack<T, VEC>(w_plane + o, w);
    if (n_plane) st_pack<T, VEC>(n_plane + o, n);
    return sum;
}

// ------------------------------------------------------------------------------------------------
// Warp-uniform context of one (z, t) plane for the primal pass.
template <typename T, typename YT = T>
struct PrimalPlane {
    const YT* y;       // component 0 of y at plane (z, t)
    const YT* zf_m;    // forward-type z component at plane z-1 (halo at a slab edge); any valid pointer when unused
    const YT* zb_p;    // backward-type z component at plane z+1
    const YT* tf_m;    // forward-type t component at plane t-1
    const YT* tb_p;    // backward-type t component at plane t+1
    T az, bz, at, bt;  // weights * existence factors of the minus / plus z and t terms (see adjoint rule below)
    long long img;     // offset of image plane (z, t) in x / xbar / x0
    const T* ts_m; const T* ts_c; const T* ts_p;   // per-voxel time scale at planes t-1, t, t+1 (clamped), or null
};

// Adjoint rule per axis (tv_operators_CPU.py:555-560, :488-493, :623-628), k = index along the axis:
//   forward-type slot F:  + [k>0] F[k-1] - [k<L-1] F[k]          backward-type slot B:  + [k>0] B[k] - [k<L-1] B[k+1]
//   centred slot C:       + [k>=2] C[k-1] - [k<=L-3] C[k+1]      (length-2 z / t axis: the forward rule)
template <typename T, int SCHEME>
PYTVB_HD void adj_factors(T& a, T& b, long long k, long long L, bool fallback) {
    if (SCHEME == CENTRAL && !fallback) {
        a = (k >= 2) ? T(1) : T(0);
        b = (k <= L - 3) ? T(1) : T(0);
    } else {
        a = (k > 0) ? T(1) : T(0);
        b = (k < L - 1) ? T(1) : T(0);
    }
}

template <typename T, int SCHEME, bool Z_ON, bool T_ON, typename YT = T>
PYTVB_HD PrimalPlane<T, YT> make_primal_plane(const FieldView<YT>& Y, const Params<T>& P, int z, int t) {
    typedef Comp<SCHEME, Z_ON, T_ON> C;
    PrimalPlane<T, YT> p;
    p.y = Y.row(P, z, 0, t, 0);
    p.img = (long long)z * P.sZ + (long long)t * P.sT;
    p.zf_m = p.zb_p = p.tf_m = p.tb_p = p.y;
    p.az = p.bz = p.at = p.bt = T(0);
    p.ts_m = p.ts_c = p.ts_p = nullptr;
    if (T_ON && P.tscale) {
        p.ts_c = P.tscale + p.img;
        p.ts_m = t > 0 ? p.ts_c - P.sT : p.ts_c;
        p.ts_p = t < P.M - 1 ? p.ts_c + P.sT : p.ts_c;
    }
    if (Z_ON) {
        const long long zg = P.zg0 + z;
        T a, b;
        adj_factors<T, SCHEME>(a, b, zg, P.NzG, P.z_fwd_fallback != 0);
        p.az = a * P.srz;
        p.bz = b * P.srz;
        if (zg > 0) p.zf_m = Y.row(P, z - 1, C::Z_F, t, 0);
        if (zg < P.NzG - 1) p.zb_p = Y.row(P, z + 1, C::Z_B, t, 0);
    }
    if (T_ON) {
        T a, b;
        adj_factors<T, SCHEME>(a, b, t, P.M, P.t_fwd_fallback != 0);
        p.at = a * P.srt;
        p.bt = b * P.srt;
        if (t > 0) p.tf_m = Y.row(P, z, C::T_F, t - 1, 0);
        if (t < P.M - 1) p.tb_p = Y.row(P, z, C::T_B, t + 1, 0);
    }
    return p;
}

// Arithmetic of the adjoint with its rounding pinned: no contraction into fma.  D^T y is computed in two places - whole in
// the primal pass, or split into an in-plane / time prefix (dual pass, cp_dual_adj_kernel) and the z term (primal pass) -
// and both must round identically.
PYTVB_HD float add_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fadd_rn(a, b);
#else
    return a + b;
#endif
}
PYTVB_HD float sub_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fsub_rn(a, b);
#else
    return a - b;
#endif
}
PYTVB_HD float mul_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fmul_rn(a, b);
#else
    return a * b;
#endif
}
PYTVB_HD double add_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
PYTVB_HD double sub_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
PYTVB_HD double mul_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}

// One axis term of the adjoint, a * m - b * p, from the slot values at k-1 / k / k+1.  m and p:
//   upwind: (F[k-1], F[k])   downwind: (B[k], B[k+1])   hybrid: (F[k-1]+B[k], F[k]+B[k+1])   central: (C[k-1], C[k+1])
template <typename T, int SCHEME>
PYTVB_HD T adj_term(T a, T b, T f_m, T f_c, T b_c, T b_p, bool fallback) {
    T m, p;
    if (SCHEME == UPWIND || (SCHEME == CENTRAL && fallback)) { m = f_m; p = f_c; }
    else if (SCHEME == DOWNWIND) { m = b_c; p = b_p; }
    else if (SCHEME == HYBRID) { m = add_rn(f_m, b_c); p = add_rn(f_c, b_p); }
    else { m = f_m; p = b_p; }
    return sub_rn(mul_rn(a, m), mul_rn(b, p));
}

// Column term of the adjoint at one quad from the J slots of the quad (jf, jb) and the three values next to it that the
// scheme reads: J_F at j0-1 and j0+VEC, J_B at j0+VEC (zero where they are outside the image).
template <typename T, int VEC, int SCHEME>
PYTVB_HD void adj_cols(T* out, const T* jf, const T* jb, T jf_left, T jf_right, T jb_right, int j0, int Nj) {
    T f[VEC + 2], bq[VEC + 2];
    f[0] = jf_left;
#pragma unroll
    for (int e = 0; e < VEC; ++e) f[e + 1] = jf[e];
    f[VEC + 1] = jf_right;
#pragma unroll
    for (int e = 0; e < VEC + 2; ++e) bq[e] = (SCHEME == DOWNWIND) ? f[e] : T(0);
    if (SCHEME == HYBRID) {
#pragma unroll
        for (int e = 0; e < VEC; ++e) bq[e + 1] = jb[e];
    }
    if (SCHEME == HYBRID || SCHEME == DOWNWIND) bq[VEC + 1] = jb_right;
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
        T a, b;
        adj_factors<T, SCHEME>(a, b, j0 + e, Nj, false);
        out[e] = (SCHEME == CENTRAL) ? adj_term<T, SCHEME>(a, b, f[e], T(0), T(0), f[e + 2], false)
                                     : adj_term<T, SCHEME>(a, b, f[e], f[e + 1], bq[e + 1], bq[e + 2], false);
    }
}

// The in-plane / time prefix of the adjoint, ((rows + t) + cols), and D^T y = (prefix + z) * inv_div: the one order of
// summation of every path.  (rows + t) alone is what the dual pass stores where a column neighbour lies outside its tile.
template <typename T, bool T_ON>
PYTVB_HD T adj_rows_t(T rows, T t) {
    return T_ON ? add_rn(rows, t) : rows;
}
template <typename T, bool T_ON>
PYTVB_HD T adj_prefix(T rows, T cols, T t) {
    return add_rn(adj_rows_t<T, T_ON>(rows, t), cols);
}
template <typename T, bool Z_ON>
PYTVB_HD T adj_finish(T prefix, T z, T inv_div) {
    return mul_rn(Z_ON ? add_rn(prefix, z) : prefix, inv_div);
}

// Loads of the dual field in the adjoint.  CG = true (generation 3 only, device only): ld.global.cg, because the
// field was rewritten by other CTAs of the SAME launch and this SM's L1 may hold pre-update lines.
template <typename T, int VEC> struct CgLoad;
#if defined(__CUDACC__)
template <> struct CgLoad<float, 4> { static __device__ __forceinline__ void ld(float* d, const float* p) { const float4 v = __ldcg(reinterpret_cast<const float4*>(p)); d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w; } };
template <> struct CgLoad<float, 1> { static __device__ __forceinline__ void ld(float* d, const float* p) { d[0] = __ldcg(p); } };
template <> struct CgLoad<double, 2> { static __device__ __forceinline__ void ld(double* d, const double* p) { const double2 v = __ldcg(reinterpret_cast<const double2*>(p)); d[0] = v.x; d[1] = v.y; } };
template <> struct CgLoad<double, 1> { static __device__ __forceinline__ void ld(double* d, const double* p) { d[0] = __ldcg(p); } };
#endif
template <typename T, int VEC, bool CG, typename YT>
PYTVB_HD void ld_field(T* dst, const YT* src) {
#if defined(__CUDA_ARCH__)
    if constexpr (CG) { CgLoad<T, VEC>::ld(dst, (const T*)src); return; }   // CG only with YT == T
#endif
    ld_y<T, YT, VEC>(dst, src);
}
template <typename T, bool CG, typename YT>
PYTVB_HD T ld_field1(const YT* src) {
#if defined(__CUDA_ARCH__)
    if constexpr (CG) { T v; CgLoad<T, 1>::ld(&v, (const T*)src); return v; }
#endif
    T v;
    ld_y<T, YT, 1>(&v, src);
    return v;
}

// Pinned form of scale_by (the time-scale products of the adjoint must round alike wherever they are formed).
template <typename T, int VEC>
PYTVB_HD void scale_by_rn(T* v, const T* ts_plane, int o) {
    if (ts_plane) {
        const Pack<T, VEC> sc = ld_pack<T, VEC>(ts_plane + o);
#pragma unroll
        for (int e = 0; e < VEC; ++e) v[e] = mul_rn(v[e], sc.v[e]);
    }
}

// Time term of the adjoint at one quad (before the static factor) from the (time-scaled) slot values; see adj_term.
template <typename T, int VEC, int SCHEME>
PYTVB_HD void adj_time(T* out, const T* f_m, const T* f_c, const T* b_c, const T* b_p, const T* fac, T at, T bt, bool fb) {
#pragma unroll
    for (int e = 0; e < VEC; ++e) out[e] = mul_rn(adj_term<T, SCHEME>(at, bt, f_m[e], f_c[e], b_c[e], b_p[e], fb), fac[e]);
}

// In-plane and time prefix of D^T y at one quad (adj_prefix; not yet times inv_div), strip addressing.
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, bool CG, typename YT, bool TS>
PYTVB_HD void strip_quad_DT_prefix(T* pre, const PrimalPlane<T, YT>& pl, const Params<T>& P, int i, int j0, int o, int o_up, int o_dn) {
    typedef Comp<SCHEME, Z_ON, T_ON> C;
    constexpr bool NF = (SCHEME != DOWNWIND);   // reads the forward-type slot at k-1 (centred: C[k-1])
    constexpr bool NB = (SCHEME != UPWIND);     // reads the backward-type slot at k+1 (centred: C[k+1])
    constexpr bool CTR = (SCHEME == CENTRAL);
    const YT* yI_F = pl.y + (long long)C::I_F * P.sC;
    const YT* yI_B = pl.y + (long long)C::I_B * P.sC;
    const YT* yJ_F = pl.y + (long long)C::J_F * P.sC;
    const YT* yJ_B = pl.y + (long long)C::J_B * P.sC;
    T rows[VEC], cols[VEC], tt[VEC];
    // ---- rows
    {
        T a, b, f_m[VEC], f_c[VEC], b_c[VEC], b_p[VEC];
        adj_factors<T, SCHEME>(a, b, i, P.Ni, false);
        if (NF) ld_field<T, VEC, CG>(f_m, yI_F + o_up); else zero_into<T, VEC>(f_m);
        if (!CTR && NF) ld_field<T, VEC, CG>(f_c, yI_F + o); else zero_into<T, VEC>(f_c);
        if (!CTR && NB) ld_field<T, VEC, CG>(b_c, yI_B + o); else zero_into<T, VEC>(b_c);
        if (NB) ld_field<T, VEC, CG>(b_p, yI_B + o_dn); else zero_into<T, VEC>(b_p);
#pragma unroll
        for (int e = 0; e < VEC; ++e) rows[e] = adj_term<T, SCHEME>(a, b, f_m[e], f_c[e], b_c[e], b_p[e], false);
    }
    // ---- columns
    {
        T jf[VEC], jb[VEC];
        ld_field<T, VEC, CG>(jf, yJ_F + o);
        if (SCHEME == HYBRID) ld_field<T, VEC, CG>(jb, yJ_B + o); else zero_into<T, VEC>(jb);
        const T jf_l = (NF && j0 > 0) ? ld_field1<T, CG>(yJ_F + o - 1) : T(0);
        const T jf_r = (CTR && j0 + VEC < P.Nj) ? ld_field1<T, CG>(yJ_F + o + VEC) : T(0);
        const T jb_r = ((SCHEME == HYBRID || SCHEME == DOWNWIND) && j0 + VEC < P.Nj) ? ld_field1<T, CG>(yJ_B + o + VEC) : T(0);
        adj_cols<T, VEC, SCHEME>(cols, jf, jb, jf_l, jf_r, jb_r, j0, P.Nj);
    }
    if (T_ON) {
        const bool fb = P.t_fwd_fallback != 0;
        const bool up_form = !CTR || fb;
        T f_m[VEC], f_c[VEC], b_c[VEC], b_p[VEC], fac[VEC];
        if (NF) ld_field<T, VEC, CG>(f_m, pl.tf_m + o); else zero_into<T, VEC>(f_m);
        if (up_form && NF) ld_field<T, VEC, CG>(f_c, pl.y + (long long)C::T_F * P.sC + o); else zero_into<T, VEC>(f_c);
        if (!CTR && NB) ld_field<T, VEC, CG>(b_c, pl.y + (long long)C::T_B * P.sC + o); else zero_into<T, VEC>(b_c);
        if (NB && !(CTR && fb)) ld_field<T, VEC, CG>(b_p, pl.tb_p + o); else zero_into<T, VEC>(b_p);
        if constexpr (TS) {   // exact adjoint of the per-voxel time scale: every entry is scaled where it lives
            scale_by_rn<T, VEC>(f_m, pl.ts_m, o); scale_by_rn<T, VEC>(f_c, pl.ts_c, o);
            scale_by_rn<T, VEC>(b_c, pl.ts_c, o); scale_by_rn<T, VEC>(b_p, pl.ts_p, o);
        }
        static_factor<T, VEC>(fac, P, i, j0);
        adj_time<T, VEC, SCHEME>(tt, f_m, f_c, b_c, b_p, fac, pl.at, pl.bt, fb);
    }
#pragma unroll
    for (int e = 0; e < VEC; ++e) pre[e] = adj_prefix<T, T_ON>(rows[e], cols[e], T_ON ? tt[e] : T(0));
}

// z term of D^T y at one quad (not yet times inv_div).
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, bool CG, typename YT>
PYTVB_HD void strip_quad_DT_z(T* zt, const PrimalPlane<T, YT>& pl, const Params<T>& P, int o) {
    typedef Comp<SCHEME, Z_ON, T_ON> C;
    constexpr bool NF = (SCHEME != DOWNWIND), NB = (SCHEME != UPWIND), CTR = (SCHEME == CENTRAL);
    const bool fb = P.z_fwd_fallback != 0;
    const bool up_form = !CTR || fb;   // needs the slot at k itself
    T f_m[VEC], f_c[VEC], b_c[VEC], b_p[VEC];
    if (NF) ld_field<T, VEC, CG>(f_m, pl.zf_m + o); else zero_into<T, VEC>(f_m);
    if (up_form && NF) ld_field<T, VEC, CG>(f_c, pl.y + (long long)C::Z_F * P.sC + o); else zero_into<T, VEC>(f_c);
    if (!CTR && NB) ld_field<T, VEC, CG>(b_c, pl.y + (long long)C::Z_B * P.sC + o); else zero_into<T, VEC>(b_c);
    if (NB && !(CTR && fb)) ld_field<T, VEC, CG>(b_p, pl.zb_p + o); else zero_into<T, VEC>(b_p);
#pragma unroll
    for (int e = 0; e < VEC; ++e) zt[e] = adj_term<T, SCHEME>(pl.az, pl.bz, f_m[e], f_c[e], b_c[e], b_p[e], fb);
}

// D^T y at one quad (times inv_div), strip addressing.
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, bool CG, typename YT, bool TS>
PYTVB_HD void strip_quad_DT_impl(T* out, const PrimalPlane<T, YT>& pl, const Params<T>& P, int i, int j0, int o, int o_up, int o_dn) {
    T pre[VEC], zt[VEC];
    strip_quad_DT_prefix<T, VEC, SCHEME, Z_ON, T_ON, CG, YT, TS>(pre, pl, P, i, j0, o, o_up, o_dn);
    if (Z_ON) strip_quad_DT_z<T, VEC, SCHEME, Z_ON, T_ON, CG, YT>(zt, pl, P, o); else zero_into<T, VEC>(zt);
#pragma unroll
    for (int e = 0; e < VEC; ++e) out[e] = adj_finish<T, Z_ON>(pre[e], zt[e], P.inv_div);
}

template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, bool CG = false, typename YT = T, bool TS = false>
PYTVB_HD void strip_quad_DT(T* out, const PrimalPlane<T, YT>& pl, const Params<T>& P, int i, int j0, int o, int o_up, int o_dn) {
    strip_quad_DT_impl<T, VEC, SCHEME, Z_ON, T_ON, CG, YT, TS && T_ON>(out, pl, P, i, j0, o, o_up, o_dn);
}

// Primal update at one quad given D^T y there (dty); off = offset of the quad in the images.  VARIANT 0: ROF prox + over-relaxation
// (aux = xbar); 1: README form (aux = y_f).
template <typename T, int VEC, bool Z_ON, int VARIANT, bool MIR, bool WM>
PYTVB_HD T cp_primal_update(const T* dty, T* x, T* aux, const T* x0, long long off, int o, T tau, T c1, T c2, T tau_x0, MirrorPlanes<T> mir,
                            const T* wgt) {
    if (tau_x0 < T(0)) tau_x0 = tau;
    const Pack<T, VEC> xo = ld_pack<T, VEC>(x + off), x0q = ld_pack<T, VEC>(x0 + off);
    Pack<T, VEC> xn, ax;
    T fid = T(0);
    if constexpr (VARIANT == 0) {
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            xn.v[e] = (xo.v[e] - tau * dty[e] + tau_x0 * x0q.v[e]) * c1;
            ax.v[e] = xn.v[e] + c2 * (xn.v[e] - xo.v[e]);
            const T r = xn.v[e] - x0q.v[e];
            fid += r * r;
        }
    } else if constexpr (VARIANT == 1) {
        const Pack<T, VEC> yf = ld_pack<T, VEC>(aux + off);
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            ax.v[e] = (yf.v[e] + c2 * (xo.v[e] - x0q.v[e])) * c1;
            xn.v[e] = xo.v[e] - tau * ax.v[e] - tau * dty[e];
            const T r = xn.v[e] - x0q.v[e];
            fid += r * r;
        }
    } else {
        static_assert(VARIANT == 2 || VARIANT == 3, "unknown primal variant");
        Pack<T, VEC> wq;
        if constexpr (WM) wq = ld_pack<T, VEC>(wgt + off);
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            T w = T(1), tw = tau_x0;
            if constexpr (WM) { w = wq.v[e]; tw = tau_x0 * w; }
            const T v = xo.v[e] - tau * dty[e];
            T r;
            if constexpr (VARIANT == 2) {
                xn.v[e] = (v + tw * x0q.v[e]) / (T(1) + tw);
                r = xn.v[e] - x0q.v[e];
                fid += w * (r * r);
            } else {
                const T d = v - x0q.v[e];
                const T a = (d < T(0) ? -d : d) - tw;
                const T s = a > T(0) ? a : T(0);
                xn.v[e] = x0q.v[e] + (d < T(0) ? -s : s);
                r = xn.v[e] - x0q.v[e];
                fid += w * (r < T(0) ? -r : r);
            }
            ax.v[e] = xn.v[e] + c2 * (xn.v[e] - xo.v[e]);
        }
    }
    st_pack<T, VEC>(x + off, xn);
    st_pack<T, VEC>(aux + off, ax);
    if constexpr (MIR && Z_ON) {
        // the image the neighbours' next dual pass differentiates: x (readme) or xbar (every other variant)
        const Pack<T, VEC>& u = (VARIANT == 1) ? xn : ax;
        if (mir.prev) st_pack<T, VEC>(mir.prev + o, u);
        if (mir.next) st_pack<T, VEC>(mir.next + o, u);
    }
    return fid;
}

// The primal update with D^T y read from the dual field, see cp_primal_update.
// c1 = 1/(1+tau) (rof) or 1/(1+sigma_A) (readme); c2 = theta or sigma_A.  Returns sum (x_new - x0)^2.
// `tau` multiplies D^T y: for a normalised half-precision dual the caller passes tau * lam.
// Other data terms, with v = x - tau D^T y, w = data weight at the voxel (wgt[...] if WM, else 1) and tau_x0 the step of
// the data term (aux = xbar, c2 = theta, c1 unused):
//   VARIANT 2: weighted L2, x_new = (v + tau w x0) / (1 + tau w);                  returns sum w (x_new - x0)^2
//   VARIANT 3: L1,          x_new = x0 + sign(v - x0) max(|v - x0| - tau w, 0);    returns sum w |x_new - x0|
// (WM is a template parameter for the reason given at strip_raw_diffs_impl.)
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, int VARIANT, bool CG = false, typename YT = T, bool TS = false, bool MIR = false,
          bool WM = false>
PYTVB_HD T strip_quad_cp_primal(T* x, T* aux, const T* x0, const PrimalPlane<T, YT>& pl, const Params<T>& P, int i, int j0, int o, int o_up, int o_dn,
                                T tau, T c1, T c2, T tau_x0 = T(-1), MirrorPlanes<T> mir = MirrorPlanes<T>{nullptr, nullptr}, const T* wgt = nullptr) {
    T dty[VEC];
    strip_quad_DT<T, VEC, SCHEME, Z_ON, T_ON, CG, YT, TS>(dty, pl, P, i, j0, o, o_up, o_dn);
    return cp_primal_update<T, VEC, Z_ON, VARIANT, MIR, WM>(dty, x, aux, x0, pl.img + o, o, tau, c1, c2, tau_x0, mir, wgt);
}

// ------------------------------------------------------------------------------------------------
// TV sweep 2 (sub-gradient from x and w = 1/|D x|), strip addressing.  See g_axis in tv_core.cuh for the rule.
template <typename T>
struct GradPlane {
    const T* x;  const T* xzm;  const T* xzp;  const T* xtm;  const T* xtp;    // image planes, clamped
    const T* xzm2; const T* xzp2; const T* xtm2; const T* xtp2;                  // centred scheme: distance 2
    const T* w;  const T* wzm;  const T* wzp;  const T* wtm;  const T* wtp;    // inverse-norm planes, clamped
    T az, bz, at, bt;      // centred scheme: weight * existence of the minus / plus term; other schemes: weight
    bool z_fb, t_fb;       // centred scheme on a length-2 axis -> forward rule
    const T* ts_m; const T* ts_c; const T* ts_p;   // per-voxel time scale at planes t-1, t, t+1 (clamped), or null
};

template <typename T, int SCHEME>
PYTVB_HD GradPlane<T> make_grad_plane(const ImgView<T>& X, const ImgView<T>& W, const Params<T>& P, int z, int t) {
    GradPlane<T> g;
    const long long zg = P.zg0 + z;
    const bool v_zm = zg > 0, v_zp = zg < P.NzG - 1, v_tm = t > 0, v_tp = t < P.M - 1;
    g.x = X.row(P, z, t, 0);
    g.w = W.row(P, z, t, 0);
    g.xzm = v_zm ? X.row(P, z - 1, t, 0) : g.x;  g.wzm = v_zm ? W.row(P, z - 1, t, 0) : g.w;
    g.xzp = v_zp ? X.row(P, z + 1, t, 0) : g.x;  g.wzp = v_zp ? W.row(P, z + 1, t, 0) : g.w;
    g.xtm = v_tm ? X.row(P, z, t - 1, 0) : g.x;  g.wtm = v_tm ? W.row(P, z, t - 1, 0) : g.w;
    g.xtp = v_tp ? X.row(P, z, t + 1, 0) : g.x;  g.wtp = v_tp ? W.row(P, z, t + 1, 0) : g.w;
    g.xzm2 = g.xzp2 = g.xtm2 = g.xtp2 = g.x;
    g.az = g.bz = P.srz;
    g.at = g.bt = P.srt;
    g.z_fb = P.z_fwd_fallback != 0;
    g.t_fb = P.t_fwd_fallback != 0;
    g.ts_m = g.ts_c = g.ts_p = nullptr;
    if (P.tscale) {
        g.ts_c = P.tscale + (long long)z * P.sZ + (long long)t * P.sT;
        g.ts_m = v_tm ? g.ts_c - P.sT : g.ts_c;
        g.ts_p = v_tp ? g.ts_c + P.sT : g.ts_c;
    }
    if (SCHEME == CENTRAL) {
        if (!g.z_fb) {
            if (zg >= 2) g.xzm2 = X.row(P, z - 2, t, 0); else g.az = T(0);
            if (zg <= P.NzG - 3) g.xzp2 = X.row(P, z + 2, t, 0); else g.bz = T(0);
        }
        if (!g.t_fb) {
            if (t >= 2) g.xtm2 = X.row(P, z, t - 2, 0); else g.at = T(0);
            if (t <= P.M - 3) g.xtp2 = X.row(P, z, t + 2, 0); else g.bt = T(0);
        }
    }
    return g;
}

// One axis of the sub-gradient with clamped neighbours: the one-sided and hybrid rules vanish by themselves
// at the boundary ((x_k - x_k) = 0); the centred rule takes explicit 0/1 factors a, b.
template <typename T, int SCHEME>
PYTVB_HD T strip_g_axis(bool fallback, T a, T b, T xm2, T xm, T xc, T xp, T xp2, T wm, T wc, T wp) {
    if (SCHEME == UPWIND || (SCHEME == CENTRAL && fallback)) return (xc - xm) * wm - (xp - xc) * wc;
    if (SCHEME == DOWNWIND) return (xc - xm) * wc - (xp - xc) * wp;
    if (SCHEME == HYBRID) return (xc - xm) * (wm + wc) - (xp - xc) * (wc + wp);
    return a * ((xc - xm2) * wm) - b * ((xp2 - xc) * wp);
}

// ROWS = false: the row part of the sub-gradient is supplied by the caller in `g_rows` (row-marching form, below).
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, bool TS, bool ROWS = true>
PYTVB_HD void strip_quad_G_impl(T* g_plane, const GradPlane<T>& pl, const Params<T>& P, int i, int j0, int o, const T* g_rows = nullptr) {
    constexpr bool CEN = (SCHEME == CENTRAL);
    const int Nj = P.Nj;
    const int o_up = i > 0 ? o - Nj : o, o_dn = i < P.Ni - 1 ? o + Nj : o;
    // ---- columns: x with 2 and w with 1 element on each side (clamped)
    T xr[VEC + 4], wr[VEC + 2];
    ld_into<T, VEC>(xr + 2, pl.x + o);
    ld_into<T, VEC>(wr + 1, pl.w + o);
    xr[1] = j0 > 0 ? pl.x[o - 1] : xr[2];
    wr[0] = j0 > 0 ? pl.w[o - 1] : wr[1];
    xr[VEC + 2] = j0 + VEC < Nj ? pl.x[o + VEC] : xr[VEC + 1];
    wr[VEC + 1] = j0 + VEC < Nj ? pl.w[o + VEC] : wr[VEC];
    xr[0] = (CEN && j0 > 1) ? pl.x[o - 2] : xr[1];
    xr[VEC + 3] = (CEN && j0 + VEC + 1 < Nj) ? pl.x[o + VEC + 1] : xr[VEC + 2];
    T g[VEC];
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
        const int j = j0 + e;
        const T a = (CEN && j < 2) ? T(0) : T(1), b = (CEN && j > Nj - 3) ? T(0) : T(1);
        g[e] = strip_g_axis<T, SCHEME>(false, a, b, xr[e], xr[e + 1], xr[e + 2], xr[e + 3], xr[e + 4], wr[e], wr[e + 1], wr[e + 2]);
    }
    // ---- rows
    if constexpr (ROWS) {
        T xm[VEC], xp[VEC], wm[VEC], wp[VEC], xm2[VEC], xp2[VEC];
        ld_into<T, VEC>(xm, pl.x + o_up);  ld_into<T, VEC>(xp, pl.x + o_dn);
        ld_into<T, VEC>(wm, pl.w + o_up);  ld_into<T, VEC>(wp, pl.w + o_dn);
        T a = T(1), b = T(1);
        if (CEN) {
            ld_into<T, VEC>(xm2, pl.x + (i > 1 ? o - 2 * Nj : o));
            ld_into<T, VEC>(xp2, pl.x + (i < P.Ni - 2 ? o + 2 * Nj : o));
            a = i >= 2 ? T(1) : T(0);
            b = i <= P.Ni - 3 ? T(1) : T(0);
        }
#pragma unroll
        for (int e = 0; e < VEC; ++e)
            g[e] += strip_g_axis<T, SCHEME>(false, a, b, CEN ? xm2[e] : T(0), xm[e], xr[e + 2], xp[e], CEN ? xp2[e] : T(0), wm[e], wr[e + 1], wp[e]);
    } else {
#pragma unroll
        for (int e = 0; e < VEC; ++e) g[e] += g_rows[e];
    }
    if (Z_ON) {
        T xm[VEC], xp[VEC], wm[VEC], wp[VEC], xm2[VEC], xp2[VEC];
        ld_into<T, VEC>(xm, pl.xzm + o);  ld_into<T, VEC>(xp, pl.xzp + o);
        ld_into<T, VEC>(wm, pl.wzm + o);  ld_into<T, VEC>(wp, pl.wzp + o);
        if (CEN) { ld_into<T, VEC>(xm2, pl.xzm2 + o); ld_into<T, VEC>(xp2, pl.xzp2 + o); }
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            const T v = strip_g_axis<T, SCHEME>(pl.z_fb, pl.az, pl.bz, CEN ? xm2[e] : T(0), xm[e], xr[e + 2], xp[e], CEN ? xp2[e] : T(0), wm[e], wr[e + 1], wp[e]);
            g[e] += (CEN && !pl.z_fb) ? v : P.srz * v;
        }
    }
    if (T_ON) {
        T xm[VEC], xp[VEC], wm[VEC], wp[VEC], xm2[VEC], xp2[VEC], fac[VEC];
        ld_into<T, VEC>(xm, pl.xtm + o);  ld_into<T, VEC>(xp, pl.xtp + o);
        ld_into<T, VEC>(wm, pl.wtm + o);  ld_into<T, VEC>(wp, pl.wtp + o);
        if (CEN) { ld_into<T, VEC>(xm2, pl.xtm2 + o); ld_into<T, VEC>(xp2, pl.xtp2 + o); }
        static_factor<T, VEC>(fac, P, i, j0);
        T wc[VEC];
#pragma unroll
        for (int e = 0; e < VEC; ++e) wc[e] = wr[e + 1];
        if constexpr (TS) {   // q = D w with D scaled where it lives: along t the inverse norms travel with their voxel's scale
            scale_by<T, VEC>(wm, pl.ts_m, o); scale_by<T, VEC>(wc, pl.ts_c, o); scale_by<T, VEC>(wp, pl.ts_p, o);
        }
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            const T v = strip_g_axis<T, SCHEME>(pl.t_fb, pl.at, pl.bt, CEN ? xm2[e] : T(0), xm[e], xr[e + 2], xp[e], CEN ? xp2[e] : T(0), wm[e], wc[e], wp[e]);
            g[e] += ((CEN && !pl.t_fb) ? v : P.srt * v) * fac[e];
        }
    }
    Pack<T, VEC> pk;
#pragma unroll
    for (int e = 0; e < VEC; ++e) pk.v[e] = g[e] * (P.inv_div * P.inv_div);
    st_pack<T, VEC>(g_plane + o, pk);
}

template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, bool TS = false>
PYTVB_HD void strip_quad_G(T* g_plane, const GradPlane<T>& pl, const Params<T>& P, int i, int j0, int o) {
    strip_quad_G_impl<T, VEC, SCHEME, Z_ON, T_ON, TS && T_ON>(g_plane, pl, P, i, j0, o);
}

// ------------------------------------------------------------------------------------------------
// TV sweeps, row-marching form (one-sided and hybrid schemes here; the centred scheme marches its rows further below).
// A thread walks down the R rows of its strip and keeps the current row, and the row difference (sweep 1) or row term
// (sweep 2) it shares with the next row, in registers: one new row load per array and row instead of three, every
// difference / product that two neighbouring voxels share is computed once, and the axis weights are applied to sums of
// squares instead of to each difference.  Both sweeps were instruction-issue bound (260 instructions per quad each,
// profiles/r01f_*), so the instruction count is what this form cuts.

// S(w_k, w_{k+1}) of the sub-gradient term between voxels k and k+1 along one axis:
//   G_axis(k) = term(k-1) - term(k),  term(k) = (x_{k+1} - x_k) * S(w_k, w_{k+1})
// (upwind: w_k, downwind: w_{k+1}, hybrid: the sum; clamped neighbours make the terms across the boundary vanish).
template <typename T, int SCHEME>
PYTVB_HD T pair_w(T wk, T wk1) {
    return SCHEME == UPWIND ? wk : (SCHEME == DOWNWIND ? wk1 : wk + wk1);
}

// Elements just left / right of this thread's quad in its row (clamped at the image edge).  On the device, when the warp
// covers 32 consecutive quads of one row (`wrow`), they come from the neighbouring lanes' registers: the scalar loads they
// replace cost the L1 as many wavefronts as a 128-bit load, and the TV sweeps are L1-bound.  The lanes at the warp's
// ends - and every lane when the warp spans several rows - load them.  `m`: the lanes that execute the sweep together.
template <typename T>
PYTVB_HD void row_neighbours(T& l, T& r, const T* row_o, T first, T last, bool has_l, bool has_r, int vec, bool wrow, unsigned m,
                             bool need_l, bool need_r) {
#if defined(__CUDA_ARCH__)
    const int lane = threadIdx.x & 31;
    const T sl = need_l ? __shfl_up_sync(m, last, 1) : first, sr = need_r ? __shfl_down_sync(m, first, 1) : last;
    const bool use_l = wrow && lane > 0, use_r = wrow && lane < 31 && has_r;
    l = !need_l ? first : (use_l ? sl : (has_l ? row_o[-1] : first));
    r = !need_r ? last : (use_r ? sr : (has_r ? row_o[vec] : last));
#else
    (void)wrow; (void)m;
    l = (need_l && has_l) ? row_o[-1] : first;
    r = (need_r && has_r) ? row_o[vec] : last;
#endif
}
PYTVB_HD unsigned sweep_lanes() {
#if defined(__CUDA_ARCH__)
    return __activemask();
#else
    return 1u;
#endif
}

// 1/sqrt(s), the norm and its inverse for sweep 1.  float on the device: one MUFU.RSQ without the denormal fix-up of
// rsqrtf (5 instructions per voxel less); a sum of squares below FLT_MIN (all differences < 1.1e-19) counts as zero.
template <typename T>
PYTVB_HD void norm_finish(T s, const Params<T>& P, T& nr, T& w, bool& pos) {
    const T rs = fast_rsqrt(s);                 // inf for s == 0
    pos = s > T(0);
    nr = pos ? s * rs * P.inv_div : T(0);
    w = pos ? rs * P.div : T(0);
}
#if defined(__CUDA_ARCH__)
template <>
__device__ __forceinline__ void norm_finish<float>(float s, const Params<float>& P, float& nr, float& w, bool& pos) {
    float rs;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rs) : "f"(fmaxf(s, 1.17549435e-38f)));
    pos = s >= 1.17549435e-38f;
    nr = pos ? s * rs * P.inv_div : 0.0f;
    w = pos ? rs * P.div : 0.0f;
}
#endif

#ifndef PYTVB_TVNORM_UNROLL
#define PYTVB_TVNORM_UNROLL 64   // row loop of sweep 1: fully unrolled
#endif
// Sweep 1 over rows i0 .. i0+R-1 of one quad column: w = 1/|D x| (0 where the norm is 0) into `w_plane`, optionally
// the norms (inf where 0) into `n_plane`; returns the sum of the norms.  FAC: the time component carries a per-voxel
// factor (mask_static or a weight map); without it the weight is uniform.  Rows past the image (last strip) recompute
// the last row and are not stored: the row loop has no branches.
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, int R, bool TS, bool FAC>
PYTVB_HD T strip_rows_tv_norm_impl(T* w_plane, T* n_plane, const DualPlane<T>& pl, const Params<T>& P, int i0, int j0) {
    static_assert(SCHEME != CENTRAL, "row-marching sweeps are for the one-sided and hybrid schemes");
    typedef Comp<SCHEME, Z_ON, T_ON> C;
    constexpr bool FWD = C::NEED_FWD, BWD = C::NEED_BWD;
    const int Nj = P.Nj, Ni = P.Ni;
    int o = i0 * Nj + j0;
    T xc[VEC], db[VEC];            // row i; x_i - x_{i-1}
    ld_into<T, VEC>(xc, pl.c + o);
    if (BWD) {
        T up[VEC];
        ld_into<T, VEC>(up, pl.c + (i0 > 0 ? o - Nj : o));
#pragma unroll
        for (int e = 0; e < VEC; ++e) db[e] = xc[e] - up[e];
    }
    const bool has_l = j0 > 0, has_r = j0 + VEC < Nj;
    const T rz2 = P.srz * P.srz, rt2 = P.srt * P.srt;
    T sum = T(0);
    constexpr int UNR = PYTVB_TVNORM_UNROLL;
#pragma unroll(UNR)
    for (int r = 0; r < R; ++r) {
        const int i = i0 + r;
        const bool live = r == 0 || i < Ni;
        const int on = i < Ni - 1 ? o + Nj : o;
        T xn[VEC], df[VEC], s[VEC];
        if (FWD || r + 1 < R) {
            ld_into<T, VEC>(xn, pl.c + on);
#pragma unroll
            for (int e = 0; e < VEC; ++e) df[e] = xn[e] - xc[e];
        }
        // (plain loads here: with the lane exchange of sweep 2 this sweep measured 20 % slower - it is not L1-bound)
        const T cl = (BWD && has_l) ? pl.c[o - 1] : xc[0], cr = (FWD && has_r) ? pl.c[o + VEC] : xc[VEC - 1];
        if (FWD) {
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                const T jf = (e + 1 < VEC ? xc[e + 1 < VEC ? e + 1 : e] : cr) - xc[e];
                s[e] = df[e] * df[e];
                s[e] += jf * jf;
            }
        }
        if (BWD) {
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                const T jb = xc[e] - (e > 0 ? xc[e > 0 ? e - 1 : 0] : cl);
                if (FWD) s[e] += db[e] * db[e]; else s[e] = db[e] * db[e];
                s[e] += jb * jb;
            }
        }
        if (Z_ON) {
            T q[VEC];
            if (FWD) {
                T zp[VEC];
                ld_into<T, VEC>(zp, pl.zp + o);
#pragma unroll
                for (int e = 0; e < VEC; ++e) { const T d = zp[e] - xc[e]; q[e] = d * d; }
            }
            if (BWD) {
                T zm[VEC];
                ld_into<T, VEC>(zm, pl.zm + o);
#pragma unroll
                for (int e = 0; e < VEC; ++e) { const T d = xc[e] - zm[e]; if (FWD) q[e] += d * d; else q[e] = d * d; }
            }
#pragma unroll
            for (int e = 0; e < VEC; ++e) s[e] += rz2 * q[e];
        }
        if (T_ON) {
            T q[VEC];
            if (FWD) {
                T tp[VEC];
                ld_into<T, VEC>(tp, pl.tp + o);
#pragma unroll
                for (int e = 0; e < VEC; ++e) { const T d = tp[e] - xc[e]; q[e] = d * d; }
            }
            if (BWD) {
                T tm[VEC];
                ld_into<T, VEC>(tm, pl.tm + o);
#pragma unroll
                for (int e = 0; e < VEC; ++e) { const T d = xc[e] - tm[e]; if (FWD) q[e] += d * d; else q[e] = d * d; }
            }
            if constexpr (FAC) {
                T fac[VEC];
                const int il = i < Ni ? i : Ni - 1;
                if constexpr (TS) time_factor<T, VEC>(fac, P, pl.ts, il, j0, o); else static_factor<T, VEC>(fac, P, il, j0);
#pragma unroll
                for (int e = 0; e < VEC; ++e) { const T wt = P.srt * fac[e]; s[e] += (wt * wt) * q[e]; }
            } else {
#pragma unroll
                for (int e = 0; e < VEC; ++e) s[e] += rt2 * q[e];
            }
        }
        Pack<T, VEC> w, n;
        T rowsum = T(0);
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            T nr; bool pos;
            norm_finish<T>(s[e], P, nr, w.v[e], pos);
            n.v[e] = pos ? nr : T(INFINITY);
            rowsum += nr;
        }
        if (live) {
            sum += rowsum;
            if (w_plane) st_pack<T, VEC>(w_plane + o, w);
            if (n_plane) st_pack<T, VEC>(n_plane + o, n);
        }
        if (r + 1 < R) {
#pragma unroll
            for (int e = 0; e < VEC; ++e) { if (BWD) db[e] = df[e]; xc[e] = xn[e]; }
            o = on;
        }
    }
    return sum;
}
// FAC must be true when the problem has a mask_static or a weight map (the launcher decides; TS implies FAC).
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, int R, bool TS = false, bool FAC = true>
PYTVB_HD T strip_rows_tv_norm(T* w_plane, T* n_plane, const DualPlane<T>& pl, const Params<T>& P, int i0, int j0) {
    return strip_rows_tv_norm_impl<T, VEC, SCHEME, Z_ON, T_ON, R, TS && T_ON, (FAC || TS) && T_ON>(w_plane, n_plane, pl, P, i0, j0);
}

#ifndef PYTVB_TVGRAD_UNROLL
#define PYTVB_TVGRAD_UNROLL 1    // row loop of sweep 2 stays a loop: unrolled, the compiler hoists the ten row loads of every row and needs 200+ registers
#endif
// Sweep 2 over rows i0 .. i0+R-1 of one quad column: the sub-gradient from x and w.
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, int R, bool TS, bool FAC>
PYTVB_HD void strip_rows_G_impl(T* g_plane, const GradPlane<T>& pl, const Params<T>& P, int i0, int j0, bool wrow) {
    const unsigned lanes = sweep_lanes();
    static_assert(SCHEME != CENTRAL, "row-marching sweeps are for the one-sided and hybrid schemes");
    const int Nj = P.Nj, Ni = P.Ni;
    int o = i0 * Nj + j0;
    T xc[VEC], wc[VEC], ti[VEC];     // row i of x and w; the row term between rows i-1 and i
    ld_into<T, VEC>(xc, pl.x + o);
    ld_into<T, VEC>(wc, pl.w + o);
    {
        T xu[VEC], wu[VEC];
        const int ou = i0 > 0 ? o - Nj : o;
        ld_into<T, VEC>(xu, pl.x + ou);
        ld_into<T, VEC>(wu, pl.w + ou);
#pragma unroll
        for (int e = 0; e < VEC; ++e) ti[e] = (xc[e] - xu[e]) * pair_w<T, SCHEME>(wu[e], wc[e]);
    }
    const bool has_l = j0 > 0, has_r = j0 + VEC < Nj;
    const T k2 = P.inv_div * P.inv_div;
    constexpr int UNR = PYTVB_TVGRAD_UNROLL;
#pragma unroll(UNR)
    for (int r = 0; r < R; ++r) {
        const int i = i0 + r;
        const bool live = r == 0 || i < Ni;
        const int on = i < Ni - 1 ? o + Nj : o;
        T xn[VEC], wn[VEC], g[VEC];
        ld_into<T, VEC>(xn, pl.x + on);
        ld_into<T, VEC>(wn, pl.w + on);
        // ---- rows
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            const T tn = (xn[e] - xc[e]) * pair_w<T, SCHEME>(wc[e], wn[e]);
            g[e] = ti[e] - tn;
            ti[e] = tn;
        }
        // ---- columns: VEC + 1 terms for VEC voxels
        {
            T xl, xr, wl, wr;
            row_neighbours<T>(xl, xr, pl.x + o, xc[0], xc[VEC - 1], has_l, has_r, VEC, wrow, lanes, true, true);
            row_neighbours<T>(wl, wr, pl.w + o, wc[0], wc[VEC - 1], has_l, has_r, VEC, wrow, lanes, true, true);
            T tj = (xc[0] - xl) * pair_w<T, SCHEME>(wl, wc[0]);
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                const T xe = e + 1 < VEC ? xc[e + 1 < VEC ? e + 1 : e] : xr, we = e + 1 < VEC ? wc[e + 1 < VEC ? e + 1 : e] : wr;
                const T tn = (xe - xc[e]) * pair_w<T, SCHEME>(wc[e], we);
                g[e] += tj - tn;
                tj = tn;
            }
        }
        if (Z_ON) {
            T xm[VEC], xp[VEC], wm[VEC], wp[VEC];
            ld_into<T, VEC>(xm, pl.xzm + o);  ld_into<T, VEC>(xp, pl.xzp + o);
            ld_into<T, VEC>(wm, pl.wzm + o);  ld_into<T, VEC>(wp, pl.wzp + o);
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                const T v = (xc[e] - xm[e]) * pair_w<T, SCHEME>(wm[e], wc[e]) - (xp[e] - xc[e]) * pair_w<T, SCHEME>(wc[e], wp[e]);
                g[e] += P.srz * v;
            }
        }
        if (T_ON) {
            T xm[VEC], xp[VEC], wm[VEC], wp[VEC], wq[VEC];
            ld_into<T, VEC>(xm, pl.xtm + o);  ld_into<T, VEC>(xp, pl.xtp + o);
            ld_into<T, VEC>(wm, pl.wtm + o);  ld_into<T, VEC>(wp, pl.wtp + o);
#pragma unroll
            for (int e = 0; e < VEC; ++e) wq[e] = wc[e];
            if constexpr (TS) {   // along t the inverse norms travel with their voxel's scale (see strip_quad_G_impl)
                scale_by<T, VEC>(wm, pl.ts_m, o); scale_by<T, VEC>(wq, pl.ts_c, o); scale_by<T, VEC>(wp, pl.ts_p, o);
            }
            T fac[VEC];
            if constexpr (FAC) static_factor<T, VEC>(fac, P, i < Ni ? i : Ni - 1, j0);
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                const T v = (xc[e] - xm[e]) * pair_w<T, SCHEME>(wm[e], wq[e]) - (xp[e] - xc[e]) * pair_w<T, SCHEME>(wq[e], wp[e]);
                if constexpr (FAC) g[e] += (P.srt * v) * fac[e]; else g[e] += P.srt * v;
            }
        }
        if (live) {
            Pack<T, VEC> pk;
#pragma unroll
            for (int e = 0; e < VEC; ++e) pk.v[e] = g[e] * k2;
            st_pack<T, VEC>(g_plane + o, pk);
        }
        if (r + 1 < R) {
#pragma unroll
            for (int e = 0; e < VEC; ++e) { xc[e] = xn[e]; wc[e] = wn[e]; }
            o = on;
        }
    }
}
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, int R, bool TS = false, bool FAC = true>
PYTVB_HD void strip_rows_G(T* g_plane, const GradPlane<T>& pl, const Params<T>& P, int i0, int j0, bool wrow = false) {
    strip_rows_G_impl<T, VEC, SCHEME, Z_ON, T_ON, R, TS && T_ON, FAC && T_ON>(g_plane, pl, P, i0, j0, wrow);
}

// ---- centred scheme, row-marching form.  Rows only: the centred differences along the rows come from a rolling window
// of registers; columns, z and t keep the per-row code.
// Sweep 1.
template <typename T, int VEC, bool Z_ON, bool T_ON, int R, bool TS, bool FAC>
PYTVB_HD T strip_rows_tv_norm_central(T* w_plane, T* n_plane, const DualPlane<T>& pl, const Params<T>& P, int i0, int j0) {
    const int Nj = P.Nj, Ni = P.Ni;
    int o = i0 * Nj + j0;
    T xu[VEC], xc[VEC];            // rows i-1 (clamped) and i
    ld_into<T, VEC>(xc, pl.c + o);
    ld_into<T, VEC>(xu, pl.c + (i0 > 0 ? o - Nj : o));
    const bool has_l = j0 > 0, has_r = j0 + VEC < Nj;
    const T wz = P.srz * pl.fz, wz2 = wz * wz, wtu = P.srt * pl.ft, wt2u = wtu * wtu;
    T sum = T(0);
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int i = i0 + r;
        const bool live = r == 0 || i < Ni;
        const int on = i < Ni - 1 ? o + Nj : o;
        T xn[VEC], s[VEC];
        ld_into<T, VEC>(xn, pl.c + on);
        const T fi = (i > 0 && i < Ni - 1) ? T(1) : T(0);
        const T cl = has_l ? pl.c[o - 1] : xc[0], cr = has_r ? pl.c[o + VEC] : xc[VEC - 1];
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            const int j = j0 + e;
            const T fj = (j > 0 && j < Nj - 1) ? T(1) : T(0);
            const T di = fi * (xn[e] - xu[e]);
            const T dj = fj * ((e + 1 < VEC ? xc[e + 1 < VEC ? e + 1 : e] : cr) - (e > 0 ? xc[e > 0 ? e - 1 : 0] : cl));
            s[e] = di * di;
            s[e] += dj * dj;
        }
        if (Z_ON) {
            T zp[VEC], zm[VEC];
            ld_into<T, VEC>(zp, pl.zp + o);
            ld_into<T, VEC>(zm, pl.zm + o);
#pragma unroll
            for (int e = 0; e < VEC; ++e) { const T d = zp[e] - zm[e]; s[e] += wz2 * (d * d); }
        }
        if (T_ON) {
            T tp[VEC], tm[VEC];
            ld_into<T, VEC>(tp, pl.tp + o);
            ld_into<T, VEC>(tm, pl.tm + o);
            if constexpr (FAC) {
                T fac[VEC];
                const int il = i < Ni ? i : Ni - 1;
                if constexpr (TS) time_factor<T, VEC>(fac, P, pl.ts, il, j0, o); else static_factor<T, VEC>(fac, P, il, j0);
#pragma unroll
                for (int e = 0; e < VEC; ++e) { const T d = tp[e] - tm[e], wt = wtu * fac[e]; s[e] += (wt * wt) * (d * d); }
            } else {
#pragma unroll
                for (int e = 0; e < VEC; ++e) { const T d = tp[e] - tm[e]; s[e] += wt2u * (d * d); }
            }
        }
        Pack<T, VEC> w, n;
        T rowsum = T(0);
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            T nr; bool pos;
            norm_finish<T>(s[e], P, nr, w.v[e], pos);
            n.v[e] = pos ? nr : T(INFINITY);
            rowsum += nr;
        }
        if (live) {
            sum += rowsum;
            if (w_plane) st_pack<T, VEC>(w_plane + o, w);
            if (n_plane) st_pack<T, VEC>(n_plane + o, n);
        }
        if (r + 1 < R) {
#pragma unroll
            for (int e = 0; e < VEC; ++e) { xu[e] = xc[e]; xc[e] = xn[e]; }
            o = on;
        }
    }
    return sum;
}

// Sweep 2.  C_m = (x_{m+1} - x_{m-1}) * w_m for 1 <= m <= Ni-2 (0 on the first and last row);  G_rows(i) = C_{i-1} - C_{i+1}.
template <typename T, int VEC, bool Z_ON, bool T_ON, int R, bool TS>
PYTVB_HD void strip_rows_G_central(T* g_plane, const GradPlane<T>& pl, const Params<T>& P, int i0, int j0) {
    const int Nj = P.Nj, Ni = P.Ni;
    const int o0 = i0 * Nj + j0;
    auto row = [&](int m) { return o0 + ((m < 0 ? 0 : (m > Ni - 1 ? Ni - 1 : m)) - i0) * Nj; };   // offset of row m, clamped
    auto valid = [&](int m) { return m >= 1 && m <= Ni - 2; };
    T xc[VEC], xp[VEC], Cm[VEC], Cc[VEC];     // rows i and i+1 of x; C_{i-1}, C_i
    ld_into<T, VEC>(xc, pl.x + o0);
    ld_into<T, VEC>(xp, pl.x + row(i0 + 1));
    {
        T xm2[VEC], xm1[VEC], wm1[VEC], w0[VEC];
        ld_into<T, VEC>(xm2, pl.x + row(i0 - 2));
        ld_into<T, VEC>(xm1, pl.x + row(i0 - 1));
        ld_into<T, VEC>(wm1, pl.w + row(i0 - 1));
        ld_into<T, VEC>(w0, pl.w + o0);
        const T vm = valid(i0 - 1) ? T(1) : T(0), vc = valid(i0) ? T(1) : T(0);
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            Cm[e] = vm * ((xc[e] - xm2[e]) * wm1[e]);
            Cc[e] = vc * ((xp[e] - xm1[e]) * w0[e]);
        }
    }
    int o = o0;
    constexpr int UNR = PYTVB_TVGRAD_UNROLL;
#pragma unroll(UNR)
    for (int r = 0; r < R; ++r) {
        const int i = i0 + r;
        if (r == 0 || i < Ni) {
            T x2[VEC], wn[VEC], g[VEC];
            ld_into<T, VEC>(x2, pl.x + row(i + 2));
            ld_into<T, VEC>(wn, pl.w + row(i + 1));
            const T vn = valid(i + 1) ? T(1) : T(0);
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                const T Cn = vn * ((x2[e] - xc[e]) * wn[e]);
                g[e] = Cm[e] - Cn;
                Cm[e] = Cc[e];
                Cc[e] = Cn;
                xc[e] = xp[e];
                xp[e] = x2[e];
            }
            strip_quad_G_impl<T, VEC, CENTRAL, Z_ON, T_ON, TS && T_ON, false>(g_plane, pl, P, i, j0, o, g);
            o += Nj;
        }
    }
}

}  // namespace pytvb

// Per-thread code of the Chambolle-Pock pass pair that finishes the in-plane and time terms of the adjoint in the dual pass
// (cp_adj.cu): A' (cp_dual_adj_kernel) and B' (cp_primal_adj_kernel).  __host__ __device__ like strip_core.cuh, so that
// tests/emul runs it tile by tile on the CPU; the tile's shared arrays are passed in.
//
// Tile of A': one z-plane x all M frames x ADJ_R rows x TWq quads (adj_tile_quads).  A thread walks the rows of one quad
// column of one frame.  Per row: adj_row_update computes the new y of its quad (strip_quad_cp_dual_y) and publishes what its
// column and frame neighbours need; after the CTA's barrier adj_row_finish gathers them, forms the column and time terms of
// the row and finishes the row term of the row before (one-row lag: it needs I_B of this row).  y is updated in place, so A'
// never reads y outside its tile.  On the first and last row of a tile (adj_edge_row) A' stores nothing and B' computes the
// whole adjoint from y (strip_quad_DT); on the first and last quad column (adj_edge_col) A' stores rows + time and B' adds the
// column term (adj_prefix sums the columns last).  Both passes derive the edges from the same geometry.
#pragma once
#include "strip_core.cuh"

#ifndef PYTVB_STRIP_R
#define PYTVB_STRIP_R 4   // image rows walked by one thread in the generation-2 kernels
#endif
#ifndef PYTVB_ADJ_R
#define PYTVB_ADJ_R 32    // rows of an A' tile: 2 of every ADJ_R rows are edges
#endif

namespace pytvb {

constexpr int ADJ_R = PYTVB_ADJ_R;
constexpr int ADJ_MAXM = 8;          // frames a tile spans: up to 8, larger M keeps the two-pass kernels
constexpr int ADJ_THREADS = 256;     // threads of an A' tile (CTA_THREADS)
static_assert(ADJ_R % PYTVB_STRIP_R == 0, "the L21 partial sums follow the row groups of cp_dual_strip_kernel");

// Quads per frame and row of an A' tile: the 256 threads over the M frames.
PYTVB_HD int adj_tile_quads(int M) { return M == 1 ? 256 : (M == 2 ? 128 : (M <= 4 ? 64 : 32)); }

// Whether A' leaves row i to B' / leaves the column term of quad column qj (tq = qj % TWq) to B'.
PYTVB_HD bool adj_edge_row(int i, int Ni) { return (i % ADJ_R == 0 && i > 0) || (i % ADJ_R == ADJ_R - 1 && i < Ni - 1); }
PYTVB_HD bool adj_edge_col(int tq, int TWq, int j0, int vec, int Nj) { return (tq == 0 && j0 > 0) || (tq == TWq - 1 && j0 + vec < Nj); }

// One row's buffer of the tile's shared arrays, AdjSlots<VEC>::value * ADJ_THREADS values at `b`: J_F first / last and J_B first
// element of every quad ([ADJ_THREADS] each), then time-scaled T_F and T_B ([VEC][ADJ_THREADS] each).
template <int VEC> struct AdjSlots { static constexpr int value = 3 + 2 * VEC; };
template <typename T, int VEC>
struct AdjShared {
    T* b;
    PYTVB_HD T& jf0(int k) const { return b[k]; }
    PYTVB_HD T& jf1(int k) const { return b[ADJ_THREADS + k]; }
    PYTVB_HD T& jb0(int k) const { return b[2 * ADJ_THREADS + k]; }
    PYTVB_HD T& tf(int e, int k) const { return b[(3 + e) * ADJ_THREADS + k]; }
    PYTVB_HD T& tb(int e, int k) const { return b[(3 + VEC + e) * ADJ_THREADS + k]; }
};

// State of one A' thread.
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON>
struct AdjThread {
    static constexpr int ND = Comp<SCHEME, Z_ON, T_ON>::ND;
    DualPlane<T, T> pl;
    MirrorPlanes<T> mir;
    T* qp;                                          // plane (z, t) of q
    int t, tq, j0, TWq;
    bool act, cedge;
    T at, bt;                                       // time factors of the adjoint at frame t
    T yv[ND][VEC], tsc[VEC];                        // the new y of the current row; time scale at the quad
    T cIFm[VEC], cIF[VEC], cIB[VEC], cCol[VEC], cT[VEC];   // carried from row k = i-1: I_F at k-1 and k, I_B at k, column and time terms at k
    T g;                                            // L21 of the current group of PYTVB_STRIP_R rows
    double l21;
};

template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, bool MIR>
PYTVB_HD void adj_thread_init(AdjThread<T, VEC, SCHEME, Z_ON, T_ON>& s, const ImgView<T>& Xb, T* y, T* qd, const Params<T>& P, const MirrorBufs<T>& mb,
                              int z, int cb, int tid, int TWq, int W) {
    s.TWq = TWq;
    s.t = tid / TWq;
    s.tq = tid - s.t * TWq;
    const int qj = cb * TWq + s.tq;
    s.j0 = qj * VEC;
    s.act = s.t < P.M && qj < W;
    const int tc = s.t < P.M ? s.t : P.M - 1;
    s.pl = make_dual_plane<T, SCHEME, T>(Xb, y, P, z, tc);
    s.mir = MirrorPlanes<T>{nullptr, nullptr};
    if constexpr (MIR) s.mir = mirror_planes<T>(mb, P, z, tc);
    s.qp = qd + (long long)z * P.sZ + (long long)tc * P.sT;
    s.cedge = adj_edge_col(s.tq, TWq, s.j0, VEC, P.Nj);
    s.at = s.bt = T(0);
    if (T_ON) {
        adj_factors<T, SCHEME>(s.at, s.bt, tc, P.M, P.t_fwd_fallback != 0);
        s.at *= P.srt;
        s.bt *= P.srt;
    }
#pragma unroll
    for (int e = 0; e < VEC; ++e) s.cIFm[e] = s.cIF[e] = s.cIB[e] = s.cCol[e] = s.cT[e] = T(0);
    s.g = T(0);
    s.l21 = 0.0;
}

// Finishes row k's prefix from the carried values, b_p = I_B at k+1 (clamped to k at the image's last row), and stores it
// unless k is an edge row.
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON>
PYTVB_HD void adj_finish_row(AdjThread<T, VEC, SCHEME, Z_ON, T_ON>& s, const Params<T>& P, int k, const T* ib_next) {
    constexpr bool NF = (SCHEME != DOWNWIND), NB = (SCHEME != UPWIND), CTR = (SCHEME == CENTRAL);
    T a, b;
    adj_factors<T, SCHEME>(a, b, k, P.Ni, false);
    Pack<T, VEC> pk;
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
        const T f_m = NF ? (k > 0 ? s.cIFm[e] : s.cIF[e]) : T(0);
        const T f_c = (!CTR && NF) ? s.cIF[e] : T(0);
        const T b_c = (!CTR && NB) ? s.cIB[e] : T(0);
        const T b_p = NB ? ib_next[e] : T(0);
        const T rows = adj_term<T, SCHEME>(a, b, f_m, f_c, b_c, b_p, false);
        pk.v[e] = s.cedge ? adj_rows_t<T, T_ON>(rows, s.cT[e]) : adj_prefix<T, T_ON>(rows, s.cCol[e], s.cT[e]);
    }
    if (!adj_edge_row(k, P.Ni)) st_pack<T, VEC>(s.qp + k * P.Nj + s.j0, pk);
}

// The next row's dual field and image row (row i+1 of y, row i+2 of xbar) to L2, before row i: the barrier of every row
// leaves one row of loads per warp in flight, too few for the HBM without it.  Device only.
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON>
PYTVB_HD void adj_prefetch_next(const AdjThread<T, VEC, SCHEME, Z_ON, T_ON>& s, const Params<T>& P, int i) {
#if defined(__CUDA_ARCH__)
    const int Nj = P.Nj, o = i * Nj + s.j0;
#pragma unroll
    for (int k = 0; k < Comp<SCHEME, Z_ON, T_ON>::ND; ++k) asm volatile("prefetch.global.L2 [%0];" ::"l"(s.pl.y + (long long)k * P.sC + o + Nj));
    asm volatile("prefetch.global.L2 [%0];" ::"l"(s.pl.c + (i + 2 < P.Ni ? o + 2 * Nj : o + Nj)));
#else
    (void)s; (void)P; (void)i;
#endif
}

// Phase 1 of row i: the dual update of the quad, its L21 partial (grouped like cp_dual_strip_kernel's per-thread sums), and
// the values its neighbours need into the shared buffer.
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, bool TS, bool MIR>
PYTVB_HD void adj_row_update(AdjThread<T, VEC, SCHEME, Z_ON, T_ON>& s, const Params<T>& P, int i, const AdjShared<T, VEC>& sh, int tid, T sig, T lam) {
    typedef Comp<SCHEME, Z_ON, T_ON> C;
    if (!s.act) return;
    const int Nj = P.Nj, o = i * Nj + s.j0;
    s.g += strip_quad_cp_dual_y<T, VEC, SCHEME, Z_ON, T_ON, T, TS, MIR>(s.yv, s.pl, P, i, s.j0, o, i > 0 ? o - Nj : o, i < P.Ni - 1 ? o + Nj : o, sig,
                                                                       lam, s.mir);
    if (i % PYTVB_STRIP_R == PYTVB_STRIP_R - 1 || i == P.Ni - 1) {
        s.l21 += (double)s.g * (double)P.inv_div;
        s.g = T(0);
    }
    sh.jf0(tid) = s.yv[C::J_F][0];
    sh.jf1(tid) = s.yv[C::J_F][VEC - 1];
    sh.jb0(tid) = s.yv[C::J_B][0];
    if (T_ON) {
#pragma unroll
        for (int e = 0; e < VEC; ++e) s.tsc[e] = T(1);
        if constexpr (TS) {
            const Pack<T, VEC> sc = ld_pack<T, VEC>(s.pl.ts + o);
#pragma unroll
            for (int e = 0; e < VEC; ++e) s.tsc[e] = sc.v[e];
        }
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            sh.tf(e, tid) = TS ? mul_rn(s.yv[C::T_F][e], s.tsc[e]) : s.yv[C::T_F][e];
            sh.tb(e, tid) = TS ? mul_rn(s.yv[C::T_B][e], s.tsc[e]) : s.yv[C::T_B][e];
        }
    }
}

// Phase 2 of row i (after the barrier): column and time terms of row i from the neighbours' values, row i-1 finished
// (first = row i is the tile's first row), the carried values moved on.
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, bool TS>
PYTVB_HD void adj_row_finish(AdjThread<T, VEC, SCHEME, Z_ON, T_ON>& s, const Params<T>& P, int i, bool first, const AdjShared<T, VEC>& sh, int tid) {
    typedef Comp<SCHEME, Z_ON, T_ON> C;
    constexpr bool NF = (SCHEME != DOWNWIND), NB = (SCHEME != UPWIND), CTR = (SCHEME == CENTRAL);
    constexpr bool HB = (SCHEME == HYBRID || SCHEME == DOWNWIND);
    if (!s.act) return;
    const int Nj = P.Nj, TWq = s.TWq;
    T col[VEC], tt[VEC];
    {
        T jb[VEC];
#pragma unroll
        for (int e = 0; e < VEC; ++e) jb[e] = (SCHEME == HYBRID) ? s.yv[C::J_B][e] : T(0);
        const bool has_l = s.j0 > 0 && s.tq > 0, has_r = s.j0 + VEC < Nj && s.tq < TWq - 1;   // neighbours inside the tile
        const T jf_l = (NF && has_l) ? sh.jf1(tid - 1) : T(0);
        const T jf_r = (CTR && has_r) ? sh.jf0(tid + 1) : T(0);
        const T jb_r = (HB && has_r) ? sh.jb0(tid + 1) : T(0);
        adj_cols<T, VEC, SCHEME>(col, s.yv[C::J_F], jb, jf_l, jf_r, jb_r, s.j0, Nj);
    }
    if (T_ON) {
        const bool tfb = P.t_fwd_fallback != 0, up_form = !CTR || tfb;
        T ifs[VEC], f_m[VEC], f_c[VEC], b_c[VEC], b_p[VEC], fac[VEC];
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            ifs[e] = TS ? mul_rn(s.yv[C::I_F][e], s.tsc[e]) : s.yv[C::I_F][e];   // the clamped operand of strip_quad_DT
            f_m[e] = NF ? (s.t > 0 ? sh.tf(e, tid - TWq) : ifs[e]) : T(0);
            f_c[e] = (up_form && NF) ? sh.tf(e, tid) : T(0);
            b_c[e] = (!CTR && NB) ? sh.tb(e, tid) : T(0);
            b_p[e] = (NB && !(CTR && tfb)) ? (s.t < P.M - 1 ? sh.tb(e, tid + TWq) : ifs[e]) : T(0);
        }
        static_factor<T, VEC>(fac, P, i, s.j0);
        adj_time<T, VEC, SCHEME>(tt, f_m, f_c, b_c, b_p, fac, s.at, s.bt, tfb);
    } else {
        zero_into<T, VEC>(tt);
    }
    if (!first) adj_finish_row(s, P, i - 1, s.yv[C::I_B]);
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
        s.cIFm[e] = s.cIF[e];
        s.cIF[e] = s.yv[C::I_F][e];
        s.cIB[e] = s.yv[C::I_B][e];
        s.cCol[e] = col[e];
        s.cT[e] = tt[e];
    }
}

// After the tile's last row: the image's last row has no row below, so it is finished here.
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON>
PYTVB_HD void adj_tile_end(AdjThread<T, VEC, SCHEME, Z_ON, T_ON>& s, const Params<T>& P, int i_end) {
    if (s.act && i_end == P.Ni) adj_finish_row(s, P, P.Ni - 1, s.cIB);
}

// B' at one quad: D^T y = (q + z term) * inv_div, with the column term added on A's edge columns and the whole adjoint from
// y on its edge rows, then the prox of cp_primal_update (VARIANT 0 ROF, 2 weighted L2, 3 L1; see strip_quad_cp_primal).
// Edge rows are warp-uniform in cp_primal_adj_kernel; an edge column is one lane of a warp, so its column loads are issued by
// every lane, from q where the lane does not need them (an L1 hit), instead of in a divergent branch.
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, int VARIANT, bool WM, bool TS, bool MIR>
PYTVB_HD T adj_quad_primal(const PrimalPlane<T, T>& pl, const T* qd, T* x, T* xbar, const T* x0, const T* w, const Params<T>& P, int i, int j0,
                           bool cedge, T tau, T c1, T theta, T tau_x0, MirrorPlanes<T> mir) {
    typedef Comp<SCHEME, Z_ON, T_ON> C;
    constexpr bool NF = (SCHEME != DOWNWIND), CTR = (SCHEME == CENTRAL), HB = (SCHEME == HYBRID || SCHEME == DOWNWIND);
    const int o = i * P.Nj + j0;
    T dty[VEC];
    if (adj_edge_row(i, P.Ni)) {
        strip_quad_DT<T, VEC, SCHEME, Z_ON, T_ON, false, T, TS>(dty, pl, P, i, j0, o, i > 0 ? o - P.Nj : o, i < P.Ni - 1 ? o + P.Nj : o);
    } else {
        const T* qo = qd + pl.img + o;
        const T* yJ_F = pl.y + (long long)C::J_F * P.sC + o;
        const T* yJ_B = pl.y + (long long)C::J_B * P.sC + o;
        const bool l = cedge && NF && j0 > 0, rf = cedge && CTR && j0 + VEC < P.Nj, rb = cedge && HB && j0 + VEC < P.Nj;
        T jf[VEC], jb[VEC];
        ld_into<T, VEC>(jf, cedge ? yJ_F : qo);
        if (SCHEME == HYBRID) ld_into<T, VEC>(jb, cedge ? yJ_B : qo); else zero_into<T, VEC>(jb);
        T jf_l = *(l ? yJ_F - 1 : qo), jf_r = *(rf ? yJ_F + VEC : qo), jb_r = *(rb ? yJ_B + VEC : qo);
        jf_l = l ? jf_l : T(0); jf_r = rf ? jf_r : T(0); jb_r = rb ? jb_r : T(0);
        const Pack<T, VEC> pre = ld_pack<T, VEC>(qo);
        T zt[VEC], cols[VEC];
        if (Z_ON) strip_quad_DT_z<T, VEC, SCHEME, Z_ON, T_ON, false, T>(zt, pl, P, o); else zero_into<T, VEC>(zt);
        adj_cols<T, VEC, SCHEME>(cols, jf, jb, jf_l, jf_r, jb_r, j0, P.Nj);
#pragma unroll
        for (int e = 0; e < VEC; ++e) dty[e] = adj_finish<T, Z_ON>(cedge ? add_rn(pre.v[e], cols[e]) : pre.v[e], zt[e], P.inv_div);
    }
    return cp_primal_update<T, VEC, Z_ON, VARIANT, MIR, WM>(dty, x, xbar, x0, pl.img + o, o, tau, c1, theta, tau_x0, mir, w);
}

}  // namespace pytvb

// TEST INFRASTRUCTURE ONLY - never linked into libpytv_b200.so.
// Host emulation of one Chambolle-Pock iteration in two forms, for a bitwise comparison:
//   split = 0: the two-pass kernels, cp_dual_strip_kernel + cp_primal_strip_kernel / cp_primal_data_strip_kernel
//              (strip_quad_cp_dual, strip_quad_cp_primal);
//   split = 1: the adjoint-split pair of cp_adj.cu, cp_dual_adj_kernel walked CTA by CTA (every thread's row update, then,
//              after the "barrier", every thread's row finish, with the tile's shared arrays on the host) and
//              cp_primal_adj_kernel quad by quad (adj_core.cuh).
// The template parameters are chosen as by the launchers.  All pointers (problem descriptor included) are HOST pointers.
#include <stdarg.h>

#include <vector>

#include "../../pytv-4d_b200/csrc/host_common.cuh"
#include "../../pytv-4d_b200/csrc/adj_core.cuh"

namespace pytvb {
static char g_err[512];
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
}  // namespace pytvb
using namespace pytvb;

namespace {

constexpr int R = PYTVB_STRIP_R;

template <typename T> struct IArgs {
    Params<T> P; ImgView<T> Xb; FieldView<T> Y; T* y; T* q; T* x; T* xbar; const T* x0; const T* w; T sig, lam, tau, theta; int term, split;
    MirrorBufs<T> mA, mB; double* sums;
};

template <typename T, int VEC, int SCHEME, bool Z, bool TT, bool TS, bool MIR>
double pass_A(const IArgs<T>& a) {
    const Params<T>& P = a.P;
    double s = 0;
    if (!a.split) {
        for (int z = 0; z < P.Nz; ++z)
            for (int t = 0; t < P.M; ++t) {
                const DualPlane<T, T> pl = make_dual_plane<T, SCHEME, T>(a.Xb, a.y, P, z, t);
                MirrorPlanes<T> mir{nullptr, nullptr};
                if constexpr (MIR) mir = mirror_planes<T>(a.mA, P, z, t);
                for (int strip = 0; strip < (P.Ni + R - 1) / R; ++strip)
                    for (int j0 = 0; j0 < P.Nj; j0 += VEC) {
                        T l21 = T(0);    // one thread's partial sum, as in the kernel
                        for (int r = 0; r < R; ++r) {
                            const int i = strip * R + r;
                            if (i < P.Ni) {
                                const int o = i * P.Nj + j0, o_up = i > 0 ? o - P.Nj : o, o_dn = i < P.Ni - 1 ? o + P.Nj : o;
                                l21 += strip_quad_cp_dual<T, VEC, SCHEME, Z, TT, T, TS, MIR>(pl, P, i, j0, o, o_up, o_dn, a.sig, a.lam, mir);
                            }
                        }
                        s += (double)l21 * (double)P.inv_div;
                    }
            }
        return s;
    }
    const int TWq = adj_tile_quads(P.M), W = (P.Nj + VEC - 1) / VEC, ncb = (W + TWq - 1) / TWq;
    std::vector<AdjThread<T, VEC, SCHEME, Z, TT>> th(ADJ_THREADS);
    std::vector<T> sm(2 * AdjSlots<VEC>::value * ADJ_THREADS, T(0));
    for (int i0 = 0; i0 < P.Ni; i0 += ADJ_R)
        for (int z = 0; z < P.Nz; ++z)
            for (int cb = 0; cb < ncb; ++cb) {
                const int nrows = ADJ_R < P.Ni - i0 ? ADJ_R : P.Ni - i0;
                for (int tid = 0; tid < ADJ_THREADS; ++tid)
                    adj_thread_init<T, VEC, SCHEME, Z, TT, MIR>(th[tid], a.Xb, a.y, a.q, P, a.mA, z, cb, tid, TWq, W);
                for (int r = 0; r < nrows; ++r) {
                    const AdjShared<T, VEC> sh{sm.data() + (r & 1) * AdjSlots<VEC>::value * ADJ_THREADS};
                    for (int tid = 0; tid < ADJ_THREADS; ++tid)
                        adj_row_update<T, VEC, SCHEME, Z, TT, TS, MIR>(th[tid], P, i0 + r, sh, tid, a.sig, a.lam);
                    for (int tid = 0; tid < ADJ_THREADS; ++tid) adj_row_finish<T, VEC, SCHEME, Z, TT, TS>(th[tid], P, i0 + r, r == 0, sh, tid);
                }
                for (int tid = 0; tid < ADJ_THREADS; ++tid) {
                    adj_tile_end(th[tid], P, i0 + nrows);
                    s += th[tid].l21;
                }
            }
    return s;
}

template <typename T, int VEC, int SCHEME, bool Z, bool TT, int VARIANT, bool WM, bool TS, bool MIR>
double pass_B(const IArgs<T>& a) {
    const Params<T>& P = a.P;
    const T c1 = VARIANT == 0 ? T(1) / (T(1) + a.tau) : T(0), tx = VARIANT == 0 ? T(-1) : a.tau;
    const int TWq = adj_tile_quads(P.M);
    double s = 0;
    for (int z = 0; z < P.Nz; ++z)
        for (int t = 0; t < P.M; ++t) {
            const PrimalPlane<T, T> pl = make_primal_plane<T, SCHEME, Z, TT, T>(a.Y, P, z, t);
            MirrorPlanes<T> mir{nullptr, nullptr};
            if constexpr (MIR) mir = mirror_planes<T>(a.mB, P, z, t);
            for (int strip = 0; strip < (P.Ni + R - 1) / R; ++strip)
                for (int j0 = 0; j0 < P.Nj; j0 += VEC) {
                    const bool cedge = adj_edge_col((j0 / VEC) % TWq, TWq, j0, VEC, P.Nj);
                    T fid = T(0);
                    for (int r = 0; r < R; ++r) {
                        const int i = strip * R + r;
                        if (i >= P.Ni) continue;
                        const int o = i * P.Nj + j0, o_up = i > 0 ? o - P.Nj : o, o_dn = i < P.Ni - 1 ? o + P.Nj : o;
                        if (a.split)
                            fid += adj_quad_primal<T, VEC, SCHEME, Z, TT, VARIANT, WM, TS, MIR>(pl, a.q, a.x, a.xbar, a.x0, a.w, P, i, j0, cedge, a.tau, c1,
                                                                                                a.theta, tx, mir);
                        else
                            fid += strip_quad_cp_primal<T, VEC, SCHEME, Z, TT, VARIANT, false, T, TS, MIR, WM>(a.x, a.xbar, a.x0, pl, P, i, j0, o, o_up, o_dn,
                                                                                                            a.tau, c1, a.theta, tx, mir, a.w);
                    }
                    s += (double)fid;
                }
        }
    return s;
}

template <typename T, int VEC, int SCHEME, bool Z, bool TT, int VARIANT, bool WM>
void iterate(const IArgs<T>& a) {
    const bool ts = TT && a.P.tscale, mA = Z && (a.mA.prev || a.mA.next), mB = Z && (a.mB.prev || a.mB.next);
    if (ts && mA) a.sums[0] = pass_A<T, VEC, SCHEME, Z, TT, TT, Z>(a);
    else if (ts) a.sums[0] = pass_A<T, VEC, SCHEME, Z, TT, TT, false>(a);
    else if (mA) a.sums[0] = pass_A<T, VEC, SCHEME, Z, TT, false, Z>(a);
    else a.sums[0] = pass_A<T, VEC, SCHEME, Z, TT, false, false>(a);
    if (ts && mB) a.sums[1] = pass_B<T, VEC, SCHEME, Z, TT, VARIANT, WM, TT, Z>(a);
    else if (ts) a.sums[1] = pass_B<T, VEC, SCHEME, Z, TT, VARIANT, WM, TT, false>(a);
    else if (mB) a.sums[1] = pass_B<T, VEC, SCHEME, Z, TT, VARIANT, WM, false, Z>(a);
    else a.sums[1] = pass_B<T, VEC, SCHEME, Z, TT, VARIANT, WM, false, false>(a);
}

template <typename T, int VEC, int SCHEME, bool Z, bool TT> struct EIter {
    static int run(const IArgs<T>& a) {
        if (a.term == PYTVB_DATA_L2 && !a.w) iterate<T, VEC, SCHEME, Z, TT, 0, false>(a);
        else if (a.term == PYTVB_DATA_L2) iterate<T, VEC, SCHEME, Z, TT, 2, true>(a);
        else if (a.w) iterate<T, VEC, SCHEME, Z, TT, 3, true>(a);
        else iterate<T, VEC, SCHEME, Z, TT, 3, false>(a);
        return 0;
    }
};

template <typename T>
int run(const pytvb_problem* pb, int split, int term, const void* w, void* xbar, void* y, void* q, void* x, const void* x0, const void* ilo,
        const void* ihi, const void* flo, const void* fhi, void* const* mir, double lam, double sigma, double tau, double theta, int force_scalar,
        double* sums) {
    const Axes ax = axes_of(pb);
    IArgs<T> a;
    a.P = make_params<T>(pb);
    a.Xb = ImgView<T>{(const T*)xbar, (const T*)ilo, (const T*)ihi, 1};
    a.Y = FieldView<T>{(const T*)y, (const T*)flo, (const T*)fhi};
    a.y = (T*)y; a.q = (T*)q; a.x = (T*)x; a.xbar = (T*)xbar; a.x0 = (const T*)x0; a.w = (const T*)w;
    a.sig = (T)sigma * a.P.inv_div; a.lam = (T)lam; a.tau = (T)tau; a.theta = (T)theta;
    a.term = term; a.split = split;
    a.mA = MirrorBufs<T>{(T*)mir[0], (T*)mir[1]};
    a.mB = MirrorBufs<T>{(T*)mir[2], (T*)mir[3]};
    a.sums = sums;
    const int vec = (force_scalar || pb->Nj % VecOf<T>::value) ? 1 : VecOf<T>::value;
    return dispatch<EIter, T>(vec, pb->scheme, ax.z_on, ax.t_on, a);
}

}  // namespace

// One iteration (dual pass on xbar, y; primal pass on x, xbar) in the two-pass (split = 0) or the adjoint-split form (split = 1,
// q = the prefix image).  ilo / ihi: image halo planes, flo / fhi: field halo planes (or NULL); mir[0..1]: the neighbours'
// field halo planes the dual pass stores into, mir[2..3]: their image halo planes for the primal pass (or NULL).
// sums[0] = L21(D xbar), sums[1] = the fidelity partial sum.
extern "C" int pytvb_emulate_adj(const pytvb_problem* pb, int split, int term, const void* w, void* xbar, void* y, void* q, void* x, const void* x0,
                                 const void* ilo, const void* ihi, const void* flo, const void* fhi, void* const* mir, double lam, double sigma,
                                 double tau, double theta, int force_scalar, double* sums) {
    if (check_problem(pb)) return -1;
    if (split && pb->M > ADJ_MAXM) {
        set_error("M > %d", ADJ_MAXM);
        return -1;
    }
    return pb->dtype == PYTVB_F32 ? run<float>(pb, split, term, w, xbar, y, q, x, x0, ilo, ihi, flo, fhi, mir, lam, sigma, tau, theta, force_scalar, sums)
                                  : run<double>(pb, split, term, w, xbar, y, q, x, x0, ilo, ihi, flo, fhi, mir, lam, sigma, tau, theta, force_scalar, sums);
}

extern "C" const char* pytvb_emulate_adj_error(void) { return g_err; }

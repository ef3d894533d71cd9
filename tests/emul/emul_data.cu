// TEST INFRASTRUCTURE ONLY - never linked into libpytv_b200.so.
// Host emulation of cp_primal_data_strip_kernel (pytv-4d_b200/csrc/cp_data.cu): the primal pass with the L1 / weighted-L2
// data terms, i.e. strip_quad_cp_primal<..., VARIANT 2 | 3, ..., WM> walked strip by strip and row by row like the kernel,
// with the same choice of template parameters as its launcher.  All pointers (problem descriptor included) are HOST pointers.
#include <stdarg.h>

#include "../../pytv-4d_b200/csrc/host_common.cuh"
#include "../../pytv-4d_b200/csrc/strip_core.cuh"

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

constexpr int R = 4;   // rows per strip, as PYTVB_STRIP_R

template <typename T> struct DArgs {
    Params<T> P; FieldView<T> Y; T* x; T* xbar; const T* x0; const T* w; T tau, theta; int term; MirrorBufs<T> mb; double* sum;
};

template <typename T, int VEC, int SCHEME, bool Z, bool TT, int VARIANT, bool WM, bool TS, bool MIR>
void walk(const DArgs<T>& a) {
    const Params<T>& P = a.P;
    double s = 0;
    for (int z = 0; z < P.Nz; ++z)
        for (int t = 0; t < P.M; ++t) {
            const PrimalPlane<T, T> pl = make_primal_plane<T, SCHEME, Z, TT, T>(a.Y, P, z, t);
            MirrorPlanes<T> mir{nullptr, nullptr};
            if constexpr (MIR) mir = mirror_planes<T>(a.mb, P, z, t);
            for (int strip = 0; strip < (P.Ni + R - 1) / R; ++strip)
                for (int j0 = 0; j0 < P.Nj; j0 += VEC) {
                    T fid = T(0);    // one thread's partial sum, as in the kernel
                    for (int r = 0; r < R; ++r) {
                        const int i = strip * R + r;
                        if (i < P.Ni) {
                            const int o = i * P.Nj + j0, o_up = i > 0 ? o - P.Nj : o, o_dn = i < P.Ni - 1 ? o + P.Nj : o;
                            fid += strip_quad_cp_primal<T, VEC, SCHEME, Z, TT, VARIANT, false, T, TS, MIR, WM>(a.x, a.xbar, a.x0, pl, P, i, j0, o, o_up, o_dn,
                                                                                                            a.tau, T(0), a.theta, a.tau, mir, a.w);
                        }
                    }
                    s += (double)fid;
                }
        }
    *a.sum = s;
}

template <typename T, int VEC, int SCHEME, bool Z, bool TT, int VARIANT, bool WM>
void select_ts_mir(const DArgs<T>& a) {
    const bool ts = TT && a.P.tscale, mir = Z && (a.mb.prev || a.mb.next);
    if (ts && mir) walk<T, VEC, SCHEME, Z, TT, VARIANT, WM, TT, Z>(a);
    else if (ts) walk<T, VEC, SCHEME, Z, TT, VARIANT, WM, TT, false>(a);
    else if (mir) walk<T, VEC, SCHEME, Z, TT, VARIANT, WM, false, Z>(a);
    else walk<T, VEC, SCHEME, Z, TT, VARIANT, WM, false, false>(a);
}

template <typename T, int VEC, int SCHEME, bool Z, bool TT> struct EData {
    static int run(const DArgs<T>& a) {
        if (a.term == PYTVB_DATA_L2) select_ts_mir<T, VEC, SCHEME, Z, TT, 2, true>(a);
        else if (a.w) select_ts_mir<T, VEC, SCHEME, Z, TT, 3, true>(a);
        else select_ts_mir<T, VEC, SCHEME, Z, TT, 3, false>(a);
        return 0;
    }
};

template <typename T>
int run(const pytvb_problem* pb, int term, const void* w, const void* y, void* x, void* xbar, const void* x0, const void* lo, const void* hi, void* mp,
        void* mn, double tau, double theta, int force_scalar, double* sum) {
    const Axes ax = axes_of(pb);
    DArgs<T> a;
    a.P = make_params<T>(pb);
    a.Y = FieldView<T>{(const T*)y, (const T*)lo, (const T*)hi};
    a.x = (T*)x; a.xbar = (T*)xbar; a.x0 = (const T*)x0; a.w = (const T*)w;
    a.tau = (T)tau; a.theta = (T)theta; a.term = term;
    a.mb = MirrorBufs<T>{(T*)mp, (T*)mn};
    a.sum = sum;
    const int vec = (force_scalar || pb->Nj % VecOf<T>::value) ? 1 : VecOf<T>::value;
    return dispatch<EData, T>(vec, pb->scheme, ax.z_on, ax.t_on, a);
}

}  // namespace

// One primal pass with data term `term` (PYTVB_DATA_L2 needs a weight map); in = y, x / xbar updated in place, sum = the
// fidelity partial sum (sum w (x - x0)^2 or sum w |x - x0|); mp / mn = the neighbours' image halo planes or NULL.
extern "C" int pytvb_emulate_data(const pytvb_problem* pb, int term, const void* w, const void* y, void* x, void* xbar, const void* x0, const void* lo,
                                  const void* hi, void* mp, void* mn, double tau, double theta, int force_scalar, double* sum) {
    if (check_problem(pb)) return -1;
    if (!(term == PYTVB_DATA_L1 || (term == PYTVB_DATA_L2 && w))) {
        set_error("term must be L1, or L2 with a weight map");
        return -1;
    }
    double dummy = 0;
    if (!sum) sum = &dummy;
    return pb->dtype == PYTVB_F32 ? run<float>(pb, term, w, y, x, xbar, x0, lo, hi, mp, mn, tau, theta, force_scalar, sum)
                                  : run<double>(pb, term, w, y, x, xbar, x0, lo, hi, mp, mn, tau, theta, force_scalar, sum);
}

extern "C" const char* pytvb_emulate_data_error(void) { return g_err; }

// Chambolle-Pock primal pass (B) of the ROF-form iteration with other data terms: per-voxel weighted L2 and (weighted) L1.
// Only the point-wise prox changes, so the iteration stays at two passes.  Split from cp.cu so that the ROF / README kernels
// keep their signatures and the translation units compile in parallel.
#include <stdlib.h>

#include "host_common.cuh"
#include "kernels2.cuh"

#ifndef PYTVB_STRIP_R
#define PYTVB_STRIP_R 4   // image rows walked by one thread in the generation-2 kernels
#endif

using namespace pytvb;

namespace pytvb {

// Same row loop as cp_primal_strip_kernel; VARIANT 2 (weighted L2) or 3 (L1), see strip_quad_cp_primal.  WM: a weight map
// is read (a template parameter, not a null check: see strip_raw_diffs_impl).  The prox is point-wise: no weight halos.
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, int VARIANT, bool WM, int R, bool TS = false, bool MIR = false>
__global__ void __launch_bounds__(CTA_THREADS, PYTVB_PRIMAL_MINB) cp_primal_data_strip_kernel(FieldView<T> Y, T* __restrict__ x, T* __restrict__ xbar,
                                                                           const T* __restrict__ x0, const T* __restrict__ w,
                                                                           double* __restrict__ partial, Params<T> P, T tau, T theta, Tiling tl,
                                                                           MirrorBufs<T> mb) {
    const QuadIdx q = decode_quad(tl, (P.Ni + R - 1) / R, VEC);
    T fid = T(0);
    if (q.active) {
        const PrimalPlane<T, T> pl = make_primal_plane<T, SCHEME, Z_ON, T_ON, T>(Y, P, q.z, q.t);
        MirrorPlanes<T> mir{nullptr, nullptr};
        if constexpr (MIR) mir = mirror_planes<T>(mb, P, q.z, q.t);
        const int i0 = q.i * R;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = i0 + r;
            if (i < P.Ni) {
                const int o = i * P.Nj + q.j0;
                const int o_up = i > 0 ? o - P.Nj : o;
                const int o_dn = i < P.Ni - 1 ? o + P.Nj : o;
                fid += strip_quad_cp_primal<T, VEC, SCHEME, Z_ON, T_ON, VARIANT, false, T, TS, MIR, WM>(x, xbar, x0, pl, P, i, q.j0, o, o_up, o_dn, tau,
                                                                                                       T(0), theta, tau, mir, w);
            }
        }
    }
    if (partial) {
        const double bs = block_sum((double)fid);
        store_or_finish(bs, partial, P);
    }
}

}  // namespace pytvb

namespace {

template <typename T> struct DataArgs {
    FieldView<T> Y; T* x; T* xbar; const T* x0; const T* w; double* partial; Params<T> P; T tau, theta; int term; cudaStream_t st; long long* nb;
    T* mir_prev; T* mir_next;
};

// TS / MIR are instantiated only where the axis exists (TS = TT, MIR = Z), as in cp.cu
template <typename T, int VEC, int SCHEME, bool Z, bool TT, int VARIANT, bool WM>
void launch_data(const DataArgs<T>& a, const Tiling& tl) {
    constexpr int R = PYTVB_STRIP_R;
    const bool ts = TT && a.P.tscale, mir = Z && (a.mir_prev || a.mir_next);
    const MirrorBufs<T> mb{a.mir_prev, a.mir_next};
    const unsigned nb = (unsigned)tl.nblocks;
    if (ts && mir)
        cp_primal_data_strip_kernel<T, VEC, SCHEME, Z, TT, VARIANT, WM, R, TT, Z><<<nb, CTA_THREADS, 0, a.st>>>(a.Y, a.x, a.xbar, a.x0, a.w, a.partial, a.P, a.tau, a.theta, tl, mb);
    else if (ts)
        cp_primal_data_strip_kernel<T, VEC, SCHEME, Z, TT, VARIANT, WM, R, TT, false><<<nb, CTA_THREADS, 0, a.st>>>(a.Y, a.x, a.xbar, a.x0, a.w, a.partial, a.P, a.tau, a.theta, tl, mb);
    else if (mir)
        cp_primal_data_strip_kernel<T, VEC, SCHEME, Z, TT, VARIANT, WM, R, false, Z><<<nb, CTA_THREADS, 0, a.st>>>(a.Y, a.x, a.xbar, a.x0, a.w, a.partial, a.P, a.tau, a.theta, tl, mb);
    else
        cp_primal_data_strip_kernel<T, VEC, SCHEME, Z, TT, VARIANT, WM, R, false, false><<<nb, CTA_THREADS, 0, a.st>>>(a.Y, a.x, a.xbar, a.x0, a.w, a.partial, a.P, a.tau, a.theta, tl, mb);
}

template <typename T, int VEC, int SCHEME, bool Z, bool TT> struct LaunchPrimalData {
    static int run(const DataArgs<T>& a) {
        const Tiling tl = make_strip_tiling<PYTVB_STRIP_R>(a.P.Nj, a.P.Ni, a.P.M, a.P.Nz, VEC);
        if (int rc = check_grid(tl)) return rc;
        if (a.term == PYTVB_DATA_L2) launch_data<T, VEC, SCHEME, Z, TT, 2, true>(a, tl);       // the caller routes L2 without a map to ROF
        else if (a.w) launch_data<T, VEC, SCHEME, Z, TT, 3, true>(a, tl);
        else launch_data<T, VEC, SCHEME, Z, TT, 3, false>(a, tl);
        count_launches(1);
        PYTVB_CUDA(cudaGetLastError());
        *a.nb = tl.nblocks;
        return PYTVB_OK;
    }
};

template <typename T>
int run_primal_data(const pytvb_problem* pb, int term, const void* w, const void* y, void* x, void* xbar, const void* x0, double tau, double theta,
                    double* d_fid, const void* lo, const void* hi, void* mir_prev, void* mir_next, void* ws, cudaStream_t st) {
    const Axes ax = axes_of(pb);
    DataArgs<T> a;
    a.Y = FieldView<T>{(const T*)y, (const T*)lo, (const T*)hi};
    a.x = (T*)x; a.xbar = (T*)xbar; a.x0 = (const T*)x0; a.w = (const T*)w;
    a.partial = d_fid ? reduce_partials(ws) : nullptr;
    a.P = make_params<T>(pb);
    arm_reduction(a.P, ws, d_fid);
    a.tau = (T)tau; a.theta = (T)theta;
    a.term = term;
    a.mir_prev = (T*)mir_prev; a.mir_next = (T*)mir_next;
    a.st = st;
    long long nb = 0;
    a.nb = &nb;
    const int vec = pick_vec<T>(pb, {y, x, xbar, x0, w, lo, hi, mir_prev, mir_next});
    if (int rc = dispatch<LaunchPrimalData, T>(vec, pb->scheme, ax.z_on, ax.t_on, a)) return rc;
    return d_fid ? finish_reduction(a.partial, nb, d_fid, st) : PYTVB_OK;
}

}  // namespace

extern "C" {

int pytvb_cp_primal_data(const pytvb_problem* pb, int data_term, const void* data_weight, const void* y, void* x, void* xbar, const void* x0,
                         double tau, double theta, double* d_fid_or_null, const void* halo_lo, const void* halo_hi, void* mirror_prev,
                         void* mirror_next, void* ws, void* stream) {
    if (int rc = check_problem(pb)) return rc;
    PYTVB_REQUIRE(data_term == PYTVB_DATA_L2 || data_term == PYTVB_DATA_L1, "data_term must be PYTVB_DATA_L2 (0) or PYTVB_DATA_L1 (1)");
    if (data_term == PYTVB_DATA_L2 && !data_weight)    // unweighted L2 is the ROF form
        return pytvb_cp_primal_p2p(pb, 0, y, x, xbar, x0, tau, theta, d_fid_or_null, halo_lo, halo_hi, mirror_prev, mirror_next, ws, stream);
    PYTVB_REQUIRE(y && x && xbar && x0, "y, x, xbar and x0 must not be NULL");
    PYTVB_REQUIRE(!d_fid_or_null || ws, "a reduction workspace is required when d_fid is requested");
    if (int rc = check_halos(pb, axes_of(pb).z_on, true, halo_lo, halo_hi)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    return pb->dtype == PYTVB_F32
               ? run_primal_data<float>(pb, data_term, data_weight, y, x, xbar, x0, tau, theta, d_fid_or_null, halo_lo, halo_hi, mirror_prev, mirror_next, ws, st)
               : run_primal_data<double>(pb, data_term, data_weight, y, x, xbar, x0, tau, theta, d_fid_or_null, halo_lo, halo_hi, mirror_prev, mirror_next, ws, st);
}

}  // extern "C"

// Chambolle-Pock iteration with the in-plane and time terms of the adjoint finished in the dual pass.
//
// Pass A' (cp_dual_adj_kernel) computes the new dual field y exactly as cp_dual_strip_kernel does and, while the new y of a
// tile is still in registers, the part of D^T y that the tile holds: the row, column and time terms (adj_prefix).  It stores
// that prefix q (one image) next to y.  Pass B' (cp_primal_adj_kernel) adds the z term, the only one that needs other
// z-planes, and applies the unchanged prox.  Per voxel and iteration at Nd = 8 that is 72 + 28 bytes instead of 68 + 48: B'
// reads q and the two z components instead of all Nd components.  Tiles, edges and the per-thread code: adj_core.cuh.
#include <stdlib.h>

#include "host_common.cuh"
#include "kernels2.cuh"
#include "adj_core.cuh"

using namespace pytvb;

namespace pytvb {

static_assert(ADJ_THREADS == CTA_THREADS, "an A' tile is one CTA");

struct AdjTiling {
    int TWq, W, ncb, nz;
    FastDiv d_ncb, d_nz;
    long long nblocks;
};
inline AdjTiling make_adj_tiling(int Nj, int Ni, int M, int nz, int vec) {
    AdjTiling t;
    t.TWq = adj_tile_quads(M);
    t.W = (Nj + vec - 1) / vec;
    t.ncb = (t.W + t.TWq - 1) / t.TWq;
    t.nz = nz;
    t.d_ncb = make_fastdiv((unsigned)t.ncb);
    t.d_nz = make_fastdiv((unsigned)nz);
    t.nblocks = (long long)t.ncb * nz * ((Ni + ADJ_R - 1) / ADJ_R);
    return t;
}

// CTAs are numbered column block fastest, then z, then row strip: the z-neighbour planes of xbar stay in L2.
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, bool TS, bool MIR>
__global__ void __launch_bounds__(CTA_THREADS, PYTVB_DUAL_MINB) cp_dual_adj_kernel(ImgView<T> Xb, T* __restrict__ y, T* __restrict__ qd,
                                                                                  double* __restrict__ partial, Params<T> P, T sig, T lam,
                                                                                  AdjTiling tl, MirrorBufs<T> mb) {
    __shared__ T sm[2][AdjSlots<T_ON ? VEC : 0>::value * CTA_THREADS];   // one buffer per row parity
    unsigned b = blockIdx.x, cb, zi;
    tl.d_ncb.divmod(b, b, cb);
    tl.d_nz.divmod(b, b, zi);
    const int i0 = (int)b * ADJ_R, nrows = min(ADJ_R, P.Ni - i0), tid = threadIdx.x;
    AdjThread<T, VEC, SCHEME, Z_ON, T_ON> s;
    adj_thread_init<T, VEC, SCHEME, Z_ON, T_ON, MIR>(s, Xb, y, qd, P, mb, (int)zi, (int)cb, tid, tl.TWq, tl.W);
    for (int r = 0; r < nrows; ++r) {
        const int bf = r & 1;
        const AdjShared<T, VEC> sh{sm[bf]};
        if (s.act && r + 1 < nrows) adj_prefetch_next(s, P, i0 + r);
        adj_row_update<T, VEC, SCHEME, Z_ON, T_ON, TS, MIR>(s, P, i0 + r, sh, tid, sig, lam);
        __syncthreads();
        adj_row_finish<T, VEC, SCHEME, Z_ON, T_ON, TS>(s, P, i0 + r, r == 0, sh, tid);
    }
    adj_tile_end(s, P, i0 + nrows);
    if (partial) {
        const double bs = block_sum(s.l21);
        store_or_finish(bs, partial, P);
    }
}

// B' (adj_quad_primal), row loop and tiling of cp_primal_strip_kernel.
template <typename T, int VEC, int SCHEME, bool Z_ON, bool T_ON, int VARIANT, bool WM, int R, bool TS, bool MIR>
__global__ void __launch_bounds__(CTA_THREADS, PYTVB_PRIMAL_MINB) cp_primal_adj_kernel(FieldView<T> Y, const T* __restrict__ qd, T* __restrict__ x,
                                                                                      T* __restrict__ xbar, const T* __restrict__ x0,
                                                                                      const T* __restrict__ w, double* __restrict__ partial,
                                                                                      Params<T> P, T tau, T c1, T theta, T tau_x0, Tiling tl,
                                                                                      int twq, MirrorBufs<T> mb) {
    const QuadIdx q = decode_quad(tl, (P.Ni + R - 1) / R, VEC);
    T fid = T(0);
    if (q.active) {
        const PrimalPlane<T, T> pl = make_primal_plane<T, SCHEME, Z_ON, T_ON, T>(Y, P, q.z, q.t);
        MirrorPlanes<T> mir{nullptr, nullptr};
        if constexpr (MIR) mir = mirror_planes<T>(mb, P, q.z, q.t);
        const bool cedge = adj_edge_col((q.j0 / VEC) & (twq - 1), twq, q.j0, VEC, P.Nj);
        const int i0 = q.i * R;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = i0 + r;
            if (i < P.Ni)
                fid += adj_quad_primal<T, VEC, SCHEME, Z_ON, T_ON, VARIANT, WM, TS, MIR>(pl, qd, x, xbar, x0, w, P, i, q.j0, cedge, tau, c1, theta, tau_x0,
                                                                                         mir);
        }
    }
    if (partial) {
        const double bs = block_sum((double)fid);
        store_or_finish(bs, partial, P);
    }
}

}  // namespace pytvb

namespace {

template <typename T> struct AdjDualArgs { ImgView<T> Xb; T* y; T* q; double* partial; Params<T> P; T sig, lam; cudaStream_t st; long long* nb; T* mir_prev; T* mir_next; };

// TS / MIR are instantiated only where the axis exists (TS = TT, MIR = Z), as in cp.cu
template <typename T, int VEC, int SCHEME, bool Z, bool TT> struct LaunchDualAdj {
    static int run(const AdjDualArgs<T>& a) {
        const AdjTiling tl = make_adj_tiling(a.P.Nj, a.P.Ni, a.P.M, a.P.Nz, VEC);
        PYTVB_REQUIRE(tl.nblocks > 0 && tl.nblocks < 2147483647LL, "grid of %lld CTAs is out of range", tl.nblocks);
        const bool ts = TT && a.P.tscale, mir = Z && (a.mir_prev || a.mir_next);
        const MirrorBufs<T> mb{a.mir_prev, a.mir_next};
        const unsigned nb = (unsigned)tl.nblocks;
        if (ts && mir) cp_dual_adj_kernel<T, VEC, SCHEME, Z, TT, TT, Z><<<nb, CTA_THREADS, 0, a.st>>>(a.Xb, a.y, a.q, a.partial, a.P, a.sig, a.lam, tl, mb);
        else if (ts) cp_dual_adj_kernel<T, VEC, SCHEME, Z, TT, TT, false><<<nb, CTA_THREADS, 0, a.st>>>(a.Xb, a.y, a.q, a.partial, a.P, a.sig, a.lam, tl, mb);
        else if (mir) cp_dual_adj_kernel<T, VEC, SCHEME, Z, TT, false, Z><<<nb, CTA_THREADS, 0, a.st>>>(a.Xb, a.y, a.q, a.partial, a.P, a.sig, a.lam, tl, mb);
        else cp_dual_adj_kernel<T, VEC, SCHEME, Z, TT, false, false><<<nb, CTA_THREADS, 0, a.st>>>(a.Xb, a.y, a.q, a.partial, a.P, a.sig, a.lam, tl, mb);
        count_launches(1);
        PYTVB_CUDA(cudaGetLastError());
        *a.nb = tl.nblocks;
        return PYTVB_OK;
    }
};

template <typename T> struct AdjPrimalArgs {
    FieldView<T> Y; const T* q; T* x; T* xbar; const T* x0; const T* w; double* partial; Params<T> P; T tau, theta; int term; cudaStream_t st;
    long long* nb; T* mir_prev; T* mir_next;
};

template <typename T, int VEC, int SCHEME, bool Z, bool TT, int VARIANT, bool WM>
void launch_primal_adj(const AdjPrimalArgs<T>& a, const Tiling& tl) {
    constexpr int R = PYTVB_STRIP_R;
    const bool ts = TT && a.P.tscale, mir = Z && (a.mir_prev || a.mir_next);
    const MirrorBufs<T> mb{a.mir_prev, a.mir_next};
    const unsigned nb = (unsigned)tl.nblocks;
    // ROF: c1 = 1/(1+tau) and the data term's step is tau; the other data terms take c1 = 0 (unused), as cp_primal_data_strip_kernel
    const T c1 = VARIANT == 0 ? T(1) / (T(1) + a.tau) : T(0), tx = VARIANT == 0 ? T(-1) : a.tau;
    const int twq = adj_tile_quads(a.P.M);
#define PYTVB_ADJ_B(TSV, MIRV)                                                                                                                  \
    cp_primal_adj_kernel<T, VEC, SCHEME, Z, TT, VARIANT, WM, R, TSV, MIRV><<<nb, CTA_THREADS, 0, a.st>>>(a.Y, a.q, a.x, a.xbar, a.x0, a.w, a.partial, \
                                                                                                      a.P, a.tau, c1, a.theta, tx, tl, twq, mb)
    if (ts && mir) PYTVB_ADJ_B(TT, Z);
    else if (ts) PYTVB_ADJ_B(TT, false);
    else if (mir) PYTVB_ADJ_B(false, Z);
    else PYTVB_ADJ_B(false, false);
#undef PYTVB_ADJ_B
}

template <typename T, int VEC, int SCHEME, bool Z, bool TT> struct LaunchPrimalAdj {
    static int run(const AdjPrimalArgs<T>& a) {
        const Tiling tl = make_strip_tiling<PYTVB_STRIP_R>(a.P.Nj, a.P.Ni, a.P.M, a.P.Nz, VEC);
        if (int rc = check_grid(tl)) return rc;
        if (a.term == PYTVB_DATA_L2 && !a.w) launch_primal_adj<T, VEC, SCHEME, Z, TT, 0, false>(a, tl);
        else if (a.term == PYTVB_DATA_L2) launch_primal_adj<T, VEC, SCHEME, Z, TT, 2, true>(a, tl);
        else if (a.w) launch_primal_adj<T, VEC, SCHEME, Z, TT, 3, true>(a, tl);
        else launch_primal_adj<T, VEC, SCHEME, Z, TT, 3, false>(a, tl);
        count_launches(1);
        PYTVB_CUDA(cudaGetLastError());
        *a.nb = tl.nblocks;
        return PYTVB_OK;
    }
};

template <typename T>
int run_dual_adj(const pytvb_problem* pb, const void* xbar, void* y, void* q, double lam, double sigma, double* d_l21, const void* lo, const void* hi,
                 void* mir_prev, void* mir_next, void* ws, cudaStream_t st) {
    const Axes ax = axes_of(pb);
    AdjDualArgs<T> a;
    a.Xb = ImgView<T>{(const T*)xbar, (const T*)lo, (const T*)hi, 1};
    a.y = (T*)y;
    a.q = (T*)q;
    a.partial = d_l21 ? reduce_partials(ws) : nullptr;
    a.P = make_params<T>(pb);
    arm_reduction(a.P, ws, d_l21);
    a.sig = (T)sigma * a.P.inv_div;
    a.lam = (T)lam;
    a.mir_prev = (T*)mir_prev; a.mir_next = (T*)mir_next;
    a.st = st;
    long long nb = 0;
    a.nb = &nb;
    const int vec = pick_vec<T>(pb, {xbar, y, q, lo, hi, mir_prev, mir_next});
    if (int rc = dispatch<LaunchDualAdj, T>(vec, pb->scheme, ax.z_on, ax.t_on, a)) return rc;
    return d_l21 ? finish_reduction(a.partial, nb, d_l21, st) : PYTVB_OK;
}

template <typename T>
int run_primal_adj(const pytvb_problem* pb, int term, const void* w, const void* y, const void* q, void* x, void* xbar, const void* x0, double tau,
                   double theta, double* d_fid, const void* lo, const void* hi, void* mir_prev, void* mir_next, void* ws, cudaStream_t st) {
    const Axes ax = axes_of(pb);
    AdjPrimalArgs<T> a;
    a.Y = FieldView<T>{(const T*)y, (const T*)lo, (const T*)hi};
    a.q = (const T*)q;
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
    const int vec = pick_vec<T>(pb, {y, q, x, xbar, x0, w, lo, hi, mir_prev, mir_next});
    if (int rc = dispatch<LaunchPrimalAdj, T>(vec, pb->scheme, ax.z_on, ax.t_on, a)) return rc;
    return d_fid ? finish_reduction(a.partial, nb, d_fid, st) : PYTVB_OK;
}

}  // namespace

extern "C" {

int pytvb_cp_dual_adj_p2p(const pytvb_problem* pb, const void* xbar, void* y, void* q, double lam, double sigma, double* d_l21_or_null,
                          const void* halo_lo, const void* halo_hi, void* mirror_prev, void* mirror_next, void* ws, void* stream) {
    if (int rc = check_problem(pb)) return rc;
    PYTVB_REQUIRE(xbar && y && q, "xbar, y and q must not be NULL");
    PYTVB_REQUIRE(pb->M <= ADJ_MAXM, "M = %lld: the dual pass with the adjoint prefix spans at most %d frames", (long long)pb->M, ADJ_MAXM);
    PYTVB_REQUIRE(!d_l21_or_null || ws, "a reduction workspace is required when d_l21 is requested");
    PYTVB_REQUIRE(lam >= 0, "lam must be >= 0");
    if (int rc = check_halos(pb, axes_of(pb).z_on, false, halo_lo, halo_hi)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    return pb->dtype == PYTVB_F32 ? run_dual_adj<float>(pb, xbar, y, q, lam, sigma, d_l21_or_null, halo_lo, halo_hi, mirror_prev, mirror_next, ws, st)
                                  : run_dual_adj<double>(pb, xbar, y, q, lam, sigma, d_l21_or_null, halo_lo, halo_hi, mirror_prev, mirror_next, ws, st);
}

int pytvb_cp_dual_adj(const pytvb_problem* pb, const void* xbar, void* y, void* q, double lam, double sigma, double* d_l21_or_null, const void* halo_lo,
                      const void* halo_hi, void* ws, void* stream) {
    return pytvb_cp_dual_adj_p2p(pb, xbar, y, q, lam, sigma, d_l21_or_null, halo_lo, halo_hi, nullptr, nullptr, ws, stream);
}

int pytvb_cp_primal_adj_p2p(const pytvb_problem* pb, int data_term, const void* data_weight, const void* y, const void* q, void* x, void* xbar,
                            const void* x0, double tau, double theta, double* d_fid_or_null, const void* halo_lo, const void* halo_hi,
                            void* mirror_prev, void* mirror_next, void* ws, void* stream) {
    if (int rc = check_problem(pb)) return rc;
    PYTVB_REQUIRE(data_term == PYTVB_DATA_L2 || data_term == PYTVB_DATA_L1, "data_term must be PYTVB_DATA_L2 (0) or PYTVB_DATA_L1 (1)");
    PYTVB_REQUIRE(y && q && x && xbar && x0, "y, q, x, xbar and x0 must not be NULL");
    PYTVB_REQUIRE(pb->M <= ADJ_MAXM, "M = %lld: the dual pass with the adjoint prefix spans at most %d frames", (long long)pb->M, ADJ_MAXM);
    PYTVB_REQUIRE(!d_fid_or_null || ws, "a reduction workspace is required when d_fid is requested");
    if (int rc = check_halos(pb, axes_of(pb).z_on, true, halo_lo, halo_hi)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    return pb->dtype == PYTVB_F32 ? run_primal_adj<float>(pb, data_term, data_weight, y, q, x, xbar, x0, tau, theta, d_fid_or_null, halo_lo, halo_hi,
                                                          mirror_prev, mirror_next, ws, st)
                                  : run_primal_adj<double>(pb, data_term, data_weight, y, q, x, xbar, x0, tau, theta, d_fid_or_null, halo_lo, halo_hi,
                                                           mirror_prev, mirror_next, ws, st);
}

int pytvb_cp_primal_adj(const pytvb_problem* pb, int data_term, const void* data_weight, const void* y, const void* q, void* x, void* xbar,
                        const void* x0, double tau, double theta, double* d_fid_or_null, const void* halo_lo, const void* halo_hi, void* ws,
                        void* stream) {
    return pytvb_cp_primal_adj_p2p(pb, data_term, data_weight, y, q, x, xbar, x0, tau, theta, d_fid_or_null, halo_lo, halo_hi, nullptr, nullptr, ws,
                                   stream);
}

}  // extern "C"

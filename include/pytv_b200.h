/* pytv_b200 - C ABI of the B200-native total-variation hot path (drop-in for PyTV-4D's GPU path).
 *
 * The reference (PyTV-4D v1.1.2) has no FFI: its boundary is the Python module API
 *     pytv/tv_GPU.py:47,142,217,290            tv_hybrid / tv_downwind / tv_upwind / tv_central
 *     pytv/tv_operators_GPU.py:134,253,362,471 D_hybrid / D_downwind / D_upwind / D_central
 *     pytv/tv_operators_GPU.py:583,719,828,938 D_T_hybrid / D_T_downwind / D_T_upwind / D_T_central
 *     pytv/tv_operators_GPU.py:46              compute_L21_norm
 *     README.md:139-158                        the Chambolle-Pock loop users build from the above
 * Each entry point below names the reference function it replaces.  The Python package binds them with
 * ctypes (pytv-4d_b200/_lib.py); INTEGRATION.md shows the binding a maintainer of the reference would add.
 *
 * Conventions
 *  - every data pointer is a DEVICE pointer on the current CUDA device unless the name ends in `_host`;
 *    arrays are dense, C order: images (Nz, M, Ni, Nj), gradient fields (Nz, Nd, M, Ni, Nj);
 *  - `stream` is a cudaStream_t passed as void* (NULL = default stream); calls only enqueue work, they do
 *    not synchronise (except the *_host entry points, which return finished results);
 *  - every function returns 0 on success, a negative pytvb_status otherwise; pytvb_last_error() gives the
 *    message for the calling thread;
 *  - there is no CPU fallback: without a CUDA device every compute entry point fails with PYTVB_ERR_CUDA.
 *
 * Slabs (multi-GPU): a call may describe one contiguous z-slab [z_offset, z_offset+Nz) of a volume with
 * Nz_global planes.  Planes just outside the slab are passed as halo pointers; they may be NULL on the
 * sides where the slab touches the volume boundary (or when the z axis is off).
 */
#ifndef PYTV_B200_H
#define PYTV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PYTVB_VERSION 101 /* 0.1.1: pytvb_problem grew time_scale_lo / time_scale_hi; the single-launch iteration was removed */

typedef enum { PYTVB_OK = 0, PYTVB_ERR_ARG = -1, PYTVB_ERR_CUDA = -2 } pytvb_status;

/* discretisation schemes (reference README.md:20-26) */
typedef enum { PYTVB_UPWIND = 0, PYTVB_DOWNWIND = 1, PYTVB_CENTRAL = 2, PYTVB_HYBRID = 3 } pytvb_scheme;
typedef enum { PYTVB_F32 = 0, PYTVB_F64 = 1 } pytvb_dtype;

/* Geometry and regularisation weights shared by all calls: the keyword arguments every reference function
 * takes (tv_operators_GPU.py:134: reg_z_over_reg, reg_time, mask_static, factor_reg_static). */
typedef struct pytvb_problem {
    int32_t scheme;             /* pytvb_scheme */
    int32_t dtype;              /* pytvb_dtype of every image / field pointer */
    int64_t Nz, M, Ni, Nj;      /* local extents (the reference requires Ni == Nj; this library does not) */
    int64_t z_offset;           /* global index of local plane 0 (0 for a whole volume) */
    int64_t Nz_global;          /* planes of the whole volume (== Nz for a whole volume) */
    double reg_z_over_reg;      /* weight of the z differences, sqrt applied inside; <= 0 or NaN: z axis off */
    double reg_time;            /* weight of the time differences; <= 0: time axis off */
    double factor_reg_static;   /* time weight multiplier where mask_static is set */
    const uint8_t* mask_static; /* device (Ni, Nj) bytes, nonzero = static pixel; NULL = none */
    const void* time_scale;     /* EXTENSION (reference TODO, README.md:258): device (Nz, M, Ni, Nj) array of `dtype`, the per-voxel factor
                                 * of the time component(s) = sqrt of a weight map; multiplies on top of mask_static; NULL = none. */
    const void* time_scale_lo;  /* slabs with z halos, pytvb_tv only: the (M, Ni, Nj) plane of time_scale at local z = -1 / z = Nz (the */
    const void* time_scale_hi;  /* gradient norm of the neighbouring plane enters the sub-gradient); NULL where the slab touches the volume edge */
} pytvb_problem;

int pytvb_version(void);
/* Identifies the SOURCES the library was built from: the first 16 hex digits of the sha256 over csrc/*.cu, *.cuh and this header (in
 * sorted order), passed in by the build (Makefile / __graft_entry__.build); "unknown" for any other build.  Ties recorded profiles
 * (profiles/traffic.json) to a build without depending on the bytes of the binary, which differ from one nvcc run to the next. */
const char* pytvb_build_id(void);
const char* pytvb_last_error(void);
/* Number of CUDA kernels this library has launched in the calling process (diagnostics / benchmarks). */
uint64_t pytvb_launch_count(void);

/* Number of difference components Nd (tv_operators_CPU.py:110-114 hybrid: 4/6/8; :256-260 others: 2/3/4). */
int pytvb_num_components(const pytvb_problem* pb);

/* Scratch sizes.  `reduce`: needed by every call that produces a scalar; `tv`: needed by pytvb_tv (a few bytes when the
 * single-sweep kernel takes the problem, an (Nz+2)-plane inverse-norm field for the two-sweep fallback).
 * The reduce workspace must be ZERO-INITIALISED before its first use (cudaMemset once after the allocation): its first 64 bytes
 * hold the arrival counter of the reductions that pytvb_tv and pytvb_gd_update finish inside the kernel (the last CTA sums the
 * partials: one launch per call); every call leaves the counter at zero.  One workspace serves one stream at a time. */
size_t pytvb_reduce_workspace_bytes(const pytvb_problem* pb);
size_t pytvb_tv_workspace_bytes(const pytvb_problem* pb);

/* D_<scheme>(img) (tv_operators_GPU.py:134,253,362,471): x (Nz,M,Ni,Nj) -> D (Nz,Nd,M,Ni,Nj).
 * halo_lo / halo_hi: image plane (M,Ni,Nj) at local z = -1 / z = Nz. */
int pytvb_D(const pytvb_problem* pb, const void* x, void* D, const void* halo_lo, const void* halo_hi, void* stream);

/* D_T_<scheme>(field) (tv_operators_GPU.py:583,719,828,938): p (Nz,Nd,M,Ni,Nj) -> out (Nz,M,Ni,Nj).
 * halo_lo: plane (M,Ni,Nj) of the forward-type z component (upwind/central: the z component) at z = -1;
 * halo_hi: plane of the backward-type z component (downwind/central: the z component) at z = Nz. */
int pytvb_DT(const pytvb_problem* pb, const void* p, void* out, const void* halo_lo, const void* halo_hi, void* stream);

/* compute_L21_norm(D_img, return_array) (tv_operators_GPU.py:46): d_sum[0] = sum_v |D_v|_2 (device double);
 * norms (Nz,M,Ni,Nj) optional.  Nd is explicit because the function takes any field. */
int pytvb_l21(const pytvb_problem* pb, const void* D, int64_t Nd, void* norms_or_null, double* d_sum, void* ws, void* stream);

/* img[~mask] = 0 in place (tv_GPU.py:79-80).  mask: bytes, full volume or one (Ni,Nj) plane. */
int pytvb_apply_mask(const pytvb_problem* pb, void* x, const uint8_t* mask, int mask_is_plane, void* stream);

/* tv_<scheme>(img) (tv_GPU.py:47,142,217,290): d_tv[0] = TV (device double), G = the reference's
 * sub-gradient, norms_or_null = gradient norms with inf where zero (return_grad_norms).
 * halo_lo2 / halo_hi2: TWO image planes each (2,M,Ni,Nj): z = -2,-1 and z = Nz, Nz+1.
 * One launch: a z-marching tile kernel reads x once (TMA into shared-memory windows) and writes G once (8 bytes per voxel;
 * csrc/tile_core.cuh, tile2_core.cuh).  The two-sweep form (inverse norms through a workspace) remains for the cases the tile
 * kernel does not take: more than 16 coupled time frames, and the centred scheme on a length-2 z or time axis.
 * x, G, norms and the halo buffers aligned to 16 bytes and Nj divisible by 4 (float) / 2 (double) select the vector path. */
int pytvb_tv(const pytvb_problem* pb, const void* x, void* G, void* norms_or_null, double* d_tv, const void* halo_lo2,
             const void* halo_hi2, void* ws_reduce, void* ws_tv, void* stream);

/* One step of the README's sub-gradient descent (README.md:120-123), fused: x <- x - step * ((x - x0) + lam * G) with G from
 * pytvb_tv, and d_fid_or_null[0] = sum (x_new - x0)^2 (the data term of the loss, README.md:123). */
int pytvb_gd_update(const pytvb_problem* pb, void* x, const void* x0, const void* G, double step, double lam, double* d_fid_or_null, void* ws,
                    void* stream);

/* TV value only, d_tv[0] = L21(D_<scheme>(x)) without materialising D or the sub-gradient (one read of x):
 * the TV term of a primal energy / duality gap.  halos: as pytvb_D (ONE image plane each side). */
int pytvb_tv_value(const pytvb_problem* pb, const void* x, double* d_tv, const void* halo_lo, const void* halo_hi, void* ws, void* stream);

/* Fused Chambolle-Pock iteration = pass A + pass B (reference: user loop README.md:145-157).
 * Pass A (dual):    y <- proj_{|.|_2 <= lam}( y + sigma * D(xbar) )           [README.md:149-151]
 *                   d_l21_or_null[0] = L21(D(xbar))  (the TV term of the loss, README.md:157)
 * halos: as pytvb_D (planes of xbar). */
int pytvb_cp_dual(const pytvb_problem* pb, const void* xbar, void* y, double lam, double sigma, double* d_l21_or_null,
                  const void* halo_lo, const void* halo_hi, void* ws, void* stream);

/* Pass B (primal), ROF form: x <- (x - tau D^T y + tau x0) / (1 + tau); xbar <- x_new + theta (x_new - x_old);
 *                   d_fid_or_null[0] = sum (x_new - x0)^2.   halos: as pytvb_DT (planes of y). */
int pytvb_cp_primal_rof(const pytvb_problem* pb, const void* y, void* x, void* xbar, const void* x0, double tau, double theta,
                        double* d_fid_or_null, const void* halo_lo, const void* halo_hi, void* ws, void* stream);

/* Pass B, README form (README.md:148,154): y_f <- (y_f + sigma_A (x - x0)) / (1 + sigma_A);
 *                   x <- x - tau y_f - tau D^T y_tv;  d_fid_or_null[0] = sum (x_new - x0)^2. */
int pytvb_cp_primal_readme(const pytvb_problem* pb, const void* y_tv, void* x, void* y_f, const void* x0, double tau,
                           double sigma_A, double* d_fid_or_null, const void* halo_lo, const void* halo_hi, void* ws,
                           void* stream);

/* Multi-GPU without an exchange step ("peer-memory halo push"): the same passes, but the kernel stores the boundary
 * planes a z-neighbour will read as its halos a second time, directly into that neighbour's halo buffer.
 * mirror_prev / mirror_next: peer-mapped DEVICE pointers (CUDA IPC / symmetric memory; NVLink) to one (M, Ni, Nj) plane in the
 * previous / next rank, or NULL.  Pass A pushes the backward-type z component of local plane 0 (the previous rank's field
 * halo_hi) and the forward-type z component of the last plane (the next rank's field halo_lo); pass B pushes plane 0 / the last
 * plane of the image the next dual pass differentiates (xbar for variant 0, x for variant 1) into the neighbours' image halo_hi /
 * halo_lo.  The caller separates the passes with a cross-rank barrier on the stream (no data moves in it). */
int pytvb_cp_dual_p2p(const pytvb_problem* pb, const void* xbar, void* y, double lam, double sigma, double* d_l21_or_null,
                      const void* halo_lo, const void* halo_hi, void* mirror_prev, void* mirror_next, void* ws, void* stream);
int pytvb_cp_primal_p2p(const pytvb_problem* pb, int variant, const void* y, void* x, void* aux, const void* x0, double tau, double c2,
                        double* d_fid_or_null, const void* halo_lo, const void* halo_hi, void* mirror_prev, void* mirror_next, void* ws,
                        void* stream);

/* Pass B of the ROF-form iteration with another data term: sum_v w_v phi(x_v - x0_v), phi = 0.5 r^2 (L2) or |r| (L1).
 * With v = x - tau D^T y:   L2: x <- (v + tau w x0) / (1 + tau w)
 *                           L1: x <- x0 + sign(v - x0) max(|v - x0| - tau w, 0)   (soft threshold)
 * then xbar <- x_new + theta (x_new - x_old).  Pass A (pytvb_cp_dual) is unchanged.
 * data_weight: device (Nz, M, Ni, Nj) array of `dtype`, >= 0, or NULL (w = 1).  L2 without a weight map is pytvb_cp_primal_rof.
 * d_fid_or_null[0] = sum_v w_v (x_new - x0)^2 (L2) or sum_v w_v |x_new - x0| (L1).
 * mirror_prev / mirror_next: as pytvb_cp_primal_p2p (NULL: no peer push).  halos: as pytvb_DT. */
typedef enum { PYTVB_DATA_L2 = 0, PYTVB_DATA_L1 = 1 } pytvb_data_term;
int pytvb_cp_primal_data(const pytvb_problem* pb, int data_term, const void* data_weight, const void* y, void* x, void* xbar,
                         const void* x0, double tau, double theta, double* d_fid_or_null, const void* halo_lo, const void* halo_hi,
                         void* mirror_prev, void* mirror_next, void* ws, void* stream);

/* The same iteration with the adjoint split between the passes: fewer bytes per voxel, results bitwise equal to
 * pytvb_cp_dual followed by pytvb_cp_primal_rof (data_term L2, no weight) or pytvb_cp_primal_data.  M <= 8.
 * q: device (Nz, M, Ni, Nj) array of `dtype`, scratch written by the dual pass and read by the primal pass of the same
 * iteration (the in-plane and time part of D^T y).  Other arguments: as pytvb_cp_dual_p2p, and as pytvb_cp_primal_data for
 * the primal pass; halos and mirrors keep their meaning.  The non-_p2p forms push nothing. */
int pytvb_cp_dual_adj(const pytvb_problem* pb, const void* xbar, void* y, void* q, double lam, double sigma, double* d_l21_or_null,
                      const void* halo_lo, const void* halo_hi, void* ws, void* stream);
int pytvb_cp_dual_adj_p2p(const pytvb_problem* pb, const void* xbar, void* y, void* q, double lam, double sigma, double* d_l21_or_null,
                          const void* halo_lo, const void* halo_hi, void* mirror_prev, void* mirror_next, void* ws, void* stream);
int pytvb_cp_primal_adj(const pytvb_problem* pb, int data_term, const void* data_weight, const void* y, const void* q, void* x, void* xbar,
                        const void* x0, double tau, double theta, double* d_fid_or_null, const void* halo_lo, const void* halo_hi, void* ws,
                        void* stream);
int pytvb_cp_primal_adj_p2p(const pytvb_problem* pb, int data_term, const void* data_weight, const void* y, const void* q, void* x, void* xbar,
                            const void* x0, double tau, double theta, double* d_fid_or_null, const void* halo_lo, const void* halo_hi,
                            void* mirror_prev, void* mirror_next, void* ws, void* stream);

/* Half-precision STORAGE of the dual field (SURVEY 8f-4): float32 images and arithmetic, y kept as IEEE half in the
 * same (Nz, Nd, M, Ni, Nj) layout, normalised to the unit ball (the array holds y / lam).  Halves the dominant
 * traffic: 4(3Nd+5) -> 6Nd+20 bytes per voxel (68 instead of 116 for Nd = 8).  NOT within the 1e-5 parity
 * tolerance (max error ~3e-4 on [0,1] images after 200 iterations): an opt-in mode.  ROF form only.  Field halo planes
 * are half precision too. */
int pytvb_cp_dual_f16y(const pytvb_problem* pb, const void* xbar, void* y_half, double lam, double sigma, double* d_l21_or_null,
                       const void* halo_lo, const void* halo_hi, void* ws, void* stream);
int pytvb_cp_primal_rof_f16y(const pytvb_problem* pb, const void* y_half, void* x, void* xbar, const void* x0, double lam, double tau,
                             double theta, double* d_fid_or_null, const void* halo_lo_half, const void* halo_hi_half, void* ws, void* stream);

/* ---- host-buffer entry points: what a caller without device memory management binds -------------------
 * tv_<scheme> with numpy-style HOST arrays in and out (the reference's default call: numpy in, numpy out,
 * tv_GPU.py:129-139).  Copies x to the device, runs pytvb_tv, copies G (and norms) back, returns TV. */
int pytvb_tv_host(const pytvb_problem* pb_host_mask /* mask_static and time_scale are HOST pointers here */, const void* x_host, void* G_host,
                  void* norms_host_or_null, double* tv_out);

/* Streaming Chambolle-Pock denoiser with device-resident state (x, xbar, y) and HOST data in / out. */
typedef struct pytvb_cp_solver pytvb_cp_solver;
int pytvb_cp_create(const pytvb_problem* pb_host_mask, double lam, double sigma, double tau, double theta, pytvb_cp_solver** out);
/* (Re)start from x0_host: x = xbar = x0, y = 0. */
int pytvb_cp_reset_host(pytvb_cp_solver* s, const void* x0_host);
/* One iteration against the data x0_host (uploaded in the call); the current x is downloaded to x_host_or_null
 * and energy_out[0] = 0.5 |x - x0|^2 + lam L21(D xbar_old).  Synchronous. */
int pytvb_cp_step_host(pytvb_cp_solver* s, const void* x0_host, void* x_host_or_null, double* energy_out);
int pytvb_cp_destroy(pytvb_cp_solver* s);

#ifdef __cplusplus
}
#endif
#endif /* PYTV_B200_H */

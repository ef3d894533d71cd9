"""Many time frames, on the host: which implementation of tv the library picks beyond 8 and 16 coupled frames (host logic of
kernels_tile.cuh / tv_path.cuh, through the emulation harness and the C ABI), and the per-thread code of those paths - the tile
kernel with one strip per frame (TI = 2), the two-sweep fallback, the two-pass Chambolle-Pock strip code - run on the host against
the float64 oracle.  tests/test_gpu_many_frames.py runs the same regimes through the real launches and relies on the table pinned
here for which path each of its cases takes."""
import ctypes

import numpy as np
import pytest

import emul_helper as em
from oracle import tv_oracle as orc
from pytv_b200 import _lib

SCHEMES = orc.SCHEMES
DTYPES = [np.float32, np.float64]


def _tv_ws_bytes(shape, dtype, reg_time, mask=None):
    keep = None if mask is None else np.ascontiguousarray(mask.astype(np.uint8))
    pb = _lib.make_problem("hybrid", _lib.F32 if dtype == np.float32 else _lib.F64, shape, 1.0, reg_time, 2.0,
                           keep.ctypes.data if keep is not None else None)
    return _lib.lib().pytvb_tv_workspace_bytes(ctypes.byref(pb))


# ------------------------------------------------------------------ 5. path selection at every threshold
# (form, strips per frame, useful rows per tile) the library picks on a 1024 x 1024 plane with the time axis on, M = 1 .. 16;
# form 1 = two phases per plane (tile_core.cuh), 2 = one phase (tile2_core.cuh).  The static-mask factors cost shared memory:
# with them M = 2 and M = 4 take the two-phase form.  Beyond 8 frames a CTA holds one strip of 4 rows per frame (TI = 2).
TILE_TABLE = {
    False: {1: (2, 16, 62), 2: (2, 8, 30), 3: (2, 5, 18), 4: (2, 4, 14), 5: (2, 3, 10), 6: (2, 2, 6), 7: (2, 2, 6), 8: (1, 2, 6),
            9: (2, 1, 2), 10: (2, 1, 2), 11: (2, 1, 2), 12: (2, 1, 2), 13: (2, 1, 2), 14: (1, 1, 2), 15: (1, 1, 2), 16: (1, 1, 2)},
    True: {1: (2, 16, 62), 2: (1, 8, 30), 3: (2, 5, 18), 4: (1, 4, 14), 5: (2, 3, 10), 6: (2, 2, 6), 7: (2, 2, 6), 8: (1, 2, 6),
           9: (2, 1, 2), 10: (2, 1, 2), 11: (2, 1, 2), 12: (2, 1, 2), 13: (2, 1, 2), 14: (1, 1, 2), 15: (1, 1, 2), 16: (1, 1, 2)},
}


@pytest.mark.parametrize("mask", [False, True], ids=["nomask", "mask_static"])
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_tile_form_table_up_to_sixteen_frames(dtype, mask):
    """Form and tile of the single-sweep kernel at every frame count it takes; the float64 tile has the same bytes per row as
    the float32 one (half the columns), so both precisions share the table."""
    vec = 4 if dtype == np.float32 else 2
    for M in range(1, 17):
        shape = (8, M, 1024, 1024)
        ms = np.ones((1024, 1024), bool) if mask else None
        g = em.tile_geometry(shape, dtype, reg_time=0.5, mask_static=ms, fac=2.0)
        form, strips, TI = TILE_TABLE[mask][M]
        assert (g["form"], g["strips"], g["TI"]) == (form, strips, TI), (M, g)
        assert g["FC"] == M and g["nthreads"] == 32 * M * strips and g["TJ"] == 32 * vec - 2 * vec
        assert 0 < g["smem"] <= g["smem_limit"]
        assert _tv_ws_bytes(shape, dtype, 0.5, ms) == 256


@pytest.mark.parametrize("mask", [False, True], ids=["nomask", "mask_static"])
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("Ni,Nj", [(7, 124), (10, 121), (1024, 1024)])
def test_nine_to_sixteen_frames_take_one_strip_per_frame(Ni, Nj, dtype, mask):
    """M = 9 .. 16: one strip of 4 rows per frame, 2 useful rows per tile, 32 M threads; the form does not depend on the image
    size; the single-sweep kernel needs only the 256-byte tv workspace."""
    for M in range(9, 17):
        shape = (6, M, Ni, Nj)
        ms = np.ones((Ni, Nj), bool) if mask else None
        g = em.tile_geometry(shape, dtype, reg_time=0.5, mask_static=ms, fac=2.0)
        assert g["form"] == TILE_TABLE[mask][M][0], (M, g)
        assert (g["strips"], g["TI"], g["FC"], g["nthreads"]) == (1, 2, M, 32 * M), (M, g)
        assert g["smem"] <= g["smem_limit"]
        assert g["nblocks"] == -(-Ni // 2) * -(-Nj // g["TJ"]) * g["nzc"] and g["Lz"] * g["nzc"] >= 6
        assert _tv_ws_bytes(shape, dtype, 0.5, ms) == 256


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("M", [17, 18, 24, 32, 50])
def test_more_than_sixteen_coupled_frames_fall_back_to_two_sweeps(M, dtype):
    """Beyond 16 coupled frames a CTA would need more than 512 threads: form 0, and the tv workspace holds the inverse-norm field of
    the slab plus one plane on each side."""
    shape = (5, M, 10, 124)
    es = np.dtype(dtype).itemsize
    for ms in (None, np.ones((10, 124), bool)):
        assert em.tile_geometry(shape, dtype, reg_time=0.5, mask_static=ms, fac=2.0)["form"] == 0
        assert _tv_ws_bytes(shape, dtype, 0.5, ms) == (5 + 2) * M * 10 * 124 * es + 256


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("M", [9, 16, 17, 32, 100])
def test_without_the_time_axis_the_tile_kernel_takes_any_frame_count(M, dtype):
    """reg_time = 0: the frames are independent 3-D volumes; a CTA holds one frame (FC = 1) and the grid has one tile group per
    frame (nfg = M)."""
    shape = (8, M, 10, 124)
    g = em.tile_geometry(shape, dtype, reg_time=0.0)
    assert g["form"] in (1, 2) and g["FC"] == 1 and g["smem"] <= g["smem_limit"]
    assert g["nblocks"] == -(-10 // g["TI"]) * -(-124 // g["TJ"]) * M * g["nzc"]
    assert _tv_ws_bytes(shape, dtype, 0.0) == 256


# ------------------------------------------------------------------ 6. the per-thread code at many frames, on the host
@pytest.fixture(params=[(0, 0, 0), (1, 4, 1), (1, 4, 2)], ids=["library", "tile-lz4-form1", "tile-lz4-form2"])
def tile(request):
    """The tile kernel with the geometry the library chooses, and with 4-plane z chunks in either form (z-chunk seams inside the
    5-plane volumes below).  Frame counts the kernel cannot take run the two-sweep fallback in every setting."""
    old = em.GEN
    em.GEN = 3
    em.set_tile(*request.param)
    yield request.param
    em.GEN = old
    em.set_tile(0, 0, 0)


def _weights(rs, shape, on):
    Nz, M, Ni, Nj = shape
    kw = dict(reg_z_over_reg=0.7, reg_time=0.3)
    if on:
        kw.update(mask_static=rs.rand(1, 1, Ni, Nj) > 0.5, factor_reg_static=2.0, time_weight=3.0 * rs.rand(*shape))
    return kw


@pytest.mark.parametrize("weights", [False, True], ids=["plain", "mask_time_weight"])
@pytest.mark.parametrize("M", [9, 12, 16, 17])
@pytest.mark.parametrize("scheme", SCHEMES)
def test_emulated_tv_at_many_frames(scheme, M, weights, tile):
    """tv, G and the norms of the emulated kernels against the oracle: odd and even image heights across the 2-row tiles, a row
    one column past the float64 tile width (and the float32 one: 124 = 120 + 4), an odd row length for the scalar form."""
    rs = np.random.RandomState(100 + M)
    for Ni, Nj in ((7, 124), (10, 61)):
        shape = (5, M, Ni, Nj)
        x = rs.rand(*shape)
        kw = _weights(rs, shape, weights)
        tv_o, G_o, n_o = orc.tv(x.copy(), scheme, return_grad_norms=True, **kw)
        for scalar in (False, True):
            tv, G, n = em.tv(x, scheme, scalar=scalar, **kw)
            assert tv == pytest.approx(tv_o, rel=1e-13), (shape, scalar)
            np.testing.assert_allclose(G, G_o, rtol=0, atol=1e-12)
            np.testing.assert_allclose(n, n_o, rtol=0, atol=1e-13)


@pytest.mark.parametrize("M", [12, 16, 17])
@pytest.mark.parametrize("scheme", SCHEMES)
def test_emulated_slabs_with_time_weight_halos(scheme, M, tile):
    """Three z-slabs with their 2-plane image halos and the weight map's neighbouring planes (time_scale_lo / _hi) reproduce the
    whole volume.  Beyond 16 frames the library refuses a weight map on slabs with halos; the same slabs without one run the
    fallback."""
    rs = np.random.RandomState(7 + M)
    Nz, Ni, Nj = 6, 7, 124
    shape = (Nz, M, Ni, Nj)
    x = rs.rand(*shape)
    kw = _weights(rs, shape, True)
    W = kw["time_weight"]
    if M > 16:
        kw.pop("time_weight")
    tv_o, G_o, n_o = orc.tv(x.copy(), scheme, return_grad_norms=True, **kw)
    tv_sum = 0.0
    for a, b in ((0, 2), (2, 3), (3, Nz)):
        lo2 = np.full((2, M, Ni, Nj), np.nan)
        hi2 = np.full((2, M, Ni, Nj), np.nan)
        for k in (1, 2):
            if a - k >= 0:
                lo2[2 - k] = x[a - k]
            if b + k - 1 < Nz:
                hi2[k - 1] = x[b + k - 1]
        kws = dict(kw)
        halos = None
        if M <= 16:
            kws["time_weight"] = W[a:b]
            halos = (W[a - 1] if a > 0 else None, W[b] if b < Nz else None)
        tvs, Gs, ns = em.tv(np.ascontiguousarray(x[a:b]), scheme, lo=lo2 if a > 0 else None, hi=hi2 if b < Nz else None, z_offset=a, Nz_global=Nz,
                            time_scale_halos=halos, **kws)
        np.testing.assert_allclose(Gs, G_o[a:b], rtol=0, atol=1e-12)
        np.testing.assert_allclose(ns, n_o[a:b], rtol=0, atol=1e-13)
        tv_sum += tvs
    assert tv_sum == pytest.approx(tv_o, rel=1e-13)


@pytest.mark.parametrize("scalar", [False, True], ids=["vec", "scalar"])
@pytest.mark.parametrize("M", [9, 12, 16, 17])
@pytest.mark.parametrize("scheme", SCHEMES)
def test_emulated_cp_iteration_at_many_frames(scheme, M, scalar):
    """One Chambolle-Pock iteration of both forms through the two-pass strip code (what CPSolver runs beyond 8 frames) from a
    random state, y non-zero also where the adjoint must ignore it; mask_static and a time-weight map on."""
    old = em.GEN
    em.GEN = 3
    try:
        rs = np.random.RandomState(200 + M)
        shape = (3, M, 7, 62)
        x0 = rs.rand(*shape)
        kw = _weights(rs, shape, True)
        Nd = orc.num_components(scheme, 3, M, 0.7, 0.3)
        y = 0.2 * rs.randn(3, Nd, *shape[1:])
        x = x0 + 0.1 * rs.randn(*shape)
        xbar = x + 0.01 * rs.randn(*shape)
        y_f = 0.1 * rs.randn(*shape)
        for variant in (0, 1):
            yy, xx = y.copy(), x.copy()
            if variant == 0:
                x_ref, aux_ref, y_ref, e_ref = orc.cp_rof_step(x.copy(), xbar.copy(), x0, y.copy(), scheme, lam=0.1, sigma=0.5, tau=0.07, theta=0.9, **kw)
                aux = xbar.copy()
                l21 = em.cp_dual(xbar, yy, scheme, 0.1, 0.5, scalar=scalar, **kw)
                fid = em.cp_primal(yy, xx, aux, x0, scheme, 0.07, 0.9, 0, scalar=scalar, **kw)
            else:
                x_ref, aux_ref, y_ref, e_ref = orc.cp_readme_step(x.copy(), x0, y_f.copy(), y.copy(), scheme, lam=0.1, sigma_D=0.5, sigma_A=0.8, tau=0.07,
                                                                  **kw)
                aux = y_f.copy()
                l21 = em.cp_dual(x, yy, scheme, 0.1, 0.5, scalar=scalar, **kw)
                fid = em.cp_primal(yy, xx, aux, x0, scheme, 0.07, 0.8, 1, scalar=scalar, **kw)
            np.testing.assert_allclose(yy, y_ref, rtol=0, atol=1e-13)
            np.testing.assert_allclose(xx, x_ref, rtol=0, atol=1e-13)
            np.testing.assert_allclose(aux, aux_ref, rtol=0, atol=1e-13)
            assert 0.5 * fid + 0.1 * l21 == pytest.approx(e_ref, rel=1e-12)
    finally:
        em.GEN = old

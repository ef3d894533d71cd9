"""Many time frames on the GPU: tv and the Chambolle-Pock solver against the float64 oracle on both sides of every frame-count
switch of the library (see tests/test_many_frames_host.py for the table of which path takes which M):
  tv: the tile kernel with several strips per frame (M <= 8), with one strip of 2 useful rows per frame (M = 9 .. 16, both forms),
      the two-sweep fallback (M >= 17), and 32 independent frames (reg_time = 0);
  slabs with a time-weight map and its halo planes (time_scale_lo / _hi), and the refusal of that combination beyond 16 frames;
  CP: the adjoint-split pass pair (M <= 8) with its tile seams inside the image, the two-pass kernels (M > 8), the data terms,
      the README form and half-precision dual storage.
Tolerances: float64 1e-12 .. 1e-13 (summation order only); float32 the north-star values against the float64 oracle on the same
float32 data - tv and energies 1e-5 relative, fields 1e-5 absolute, the sub-gradient within 1e-5 or 3 x the float32 oracle's own
error where the norms are tiny (_assert_G_float32)."""
import ctypes

import numpy as np
import pytest
import torch

import data_term_oracle as dto
import emul_helper as em
import pytv_b200 as pytv
from oracle import tv_oracle as orc
from pytv_b200 import _dev, _lib
from test_gpu_parity import _assert_G_float32

pytestmark = pytest.mark.gpu
SCHEMES = orc.SCHEMES
DTYPES = [np.float32, np.float64]
DT_IDS = ["f32", "f64"]


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"


def _tv(scheme):
    return getattr(pytv.tv_GPU, "tv_" + scheme)


def _path(shape, dtype, kw):
    """The tv implementation the library takes for a whole volume (host geometry of kernels_tile.cuh)."""
    g = em.tile_geometry(shape, dtype, reg_z_over_reg=kw.get("reg_z_over_reg", 1.0), reg_time=kw.get("reg_time", 0.0),
                         mask_static=kw.get("mask_static"), fac=kw.get("factor_reg_static", 0.0))
    return "fallback" if g["form"] == 0 else "tile form %d, %d strip(s) x TI %d, FC %d" % (g["form"], g["strips"], g["TI"], g["FC"])


def _weights(rs, shape, kind):
    Nz, M, Ni, Nj = shape
    kw = dict(reg_z_over_reg=0.7, reg_time=0.3)
    if kind in ("mask", "both"):
        kw.update(mask_static=rs.rand(1, 1, Ni, Nj) > 0.5, factor_reg_static=2.0)
    if kind in ("time_weight", "both"):
        kw.update(time_weight=0.5 + rs.rand(*shape))
    return kw


def _check_tv(got, x, scheme, kw, dtype, what):
    """(tv, G, norms) of the library against the float64 oracle on the same (float32-rounded) data."""
    tv, G, n = got
    tv_o, G_o, n_o = orc.tv(x.astype(np.float64), scheme, return_grad_norms=True, **kw)
    if dtype == np.float64:
        assert float(tv) == pytest.approx(tv_o, rel=1e-13), what
        np.testing.assert_allclose(G, G_o, rtol=0, atol=1e-12, err_msg=what)
        np.testing.assert_allclose(n, n_o, rtol=0, atol=1e-13, err_msg=what)
    else:
        assert float(tv) == pytest.approx(tv_o, rel=1e-5), what
        _assert_G_float32(G, G_o, x, scheme, kw)
        np.testing.assert_allclose(n, n_o, rtol=0, atol=1e-5, err_msg=what)


# ------------------------------------------------------------------ 1. tv across the frame-count regimes
TV_M = [1, 2, 3, 4, 5, 8, 9, 12, 16, 17, 24, 32]


def test_the_frame_counts_cover_every_tv_path():
    """The M values below reach every tv implementation: several strips per frame, one strip per frame (TI = 2) in both forms of the
    tile kernel, and the two-sweep fallback, in both precisions."""
    for dtype in DTYPES:
        paths = {_path((5, M, 10, 124), dtype, dict(reg_time=0.3)) for M in TV_M}
        assert "fallback" in paths
        for form in (1, 2):
            assert any(p.startswith("tile form %d, 1 strip(s) x TI 2" % form) for p in paths), paths
        assert any(p.startswith("tile form 2, 3 strip(s)") for p in paths), paths


@pytest.mark.parametrize("weights", ["plain", "mask", "time_weight"])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("M", TV_M)
def test_tv_across_frame_regimes(M, dtype, weights):
    """tv, G and the norms for every scheme: Ni odd and even across the 2-row tiles, Nj = 124 one quad past the float32 tile width
    (120) and past twice the float64 one (60), odd Nj = 121 for the scalar form; 5 planes so that the z chunks have seams."""
    rs = np.random.RandomState(1000 + 10 * M + len(weights))
    for Ni, Nj in ((7, 124), (10, 124), (10, 121)):
        shape = (5, M, Ni, Nj)
        x = rs.rand(*shape).astype(dtype)
        kw = _weights(rs, shape, weights)
        path = _path(shape, dtype, kw)
        for scheme in SCHEMES:
            got = _tv(scheme)(x.copy(), return_grad_norms=True, **kw)
            _check_tv(got, x, scheme, kw, dtype, "%s %s %s" % (scheme, shape, path))


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("M", [5, 12, 24])
def test_tv_unaligned_view_takes_the_scalar_forms(M, dtype):
    """An image that starts one element past an aligned address: no tensor map, no vector loads (VEC = 1), in the multi-strip and
    one-strip tile kernel and the fallback; mask_static and a time-weight map on."""
    rs = np.random.RandomState(77 + M)
    shape = (5, M, 10, 124)
    tdt = torch.float32 if dtype == np.float32 else torch.float64
    x = rs.rand(*shape).astype(dtype)
    kw = _weights(rs, shape, "both")
    big = torch.empty(x.size + 1, dtype=tdt, device="cuda")
    xu = big[1:].view(shape)
    assert xu.data_ptr() % 16 != 0
    for scheme in SCHEMES:
        xu.copy_(torch.as_tensor(x))
        tv, G, n = _tv(scheme)(xu, return_grad_norms=True, return_pytorch_tensor=True, **kw)
        _check_tv((tv, G.cpu().numpy(), n.cpu().numpy()), x, scheme, kw, dtype, "%s unaligned %s" % (scheme, _path(shape, dtype, kw)))


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_tv_thirty_two_independent_frames(dtype):
    """reg_time = 0 at M = 32: the tile kernel with one frame per CTA and one tile group per frame, against the per-frame 3-D oracle."""
    rs = np.random.RandomState(32)
    for Ni, Nj in ((7, 124), (10, 121)):
        shape = (5, 32, Ni, Nj)
        x = rs.rand(*shape).astype(dtype)
        kw = dict(reg_z_over_reg=0.7, reg_time=0.0)
        path = _path(shape, dtype, kw)
        assert path.startswith("tile") and path.endswith("FC 1"), path
        for scheme in SCHEMES:
            got = _tv(scheme)(x.copy(), return_grad_norms=True, **kw)
            _check_tv(got, x, scheme, kw, dtype, "%s %s %s" % (scheme, shape, path))


# ------------------------------------------------------------------ 2. z-slabs with time-weight halos on one GPU
def _tv_call(pb, x, lo2, hi2):
    lib = _lib.lib()
    G, n, d = torch.empty_like(x), torch.empty_like(x), torch.zeros(1, dtype=torch.float64, device="cuda")
    wsr = _dev.reduce_workspace(pb, x.device)
    wst = torch.empty(lib.pytvb_tv_workspace_bytes(ctypes.byref(pb)), dtype=torch.uint8, device="cuda")
    _lib.check(lib.pytvb_tv(ctypes.byref(pb), _dev.ptr(x), _dev.ptr(G), _dev.ptr(n), _dev.ptr(d), _dev.ptr(lo2), _dev.ptr(hi2), _dev.ptr(wsr),
                            _dev.ptr(wst), _dev.stream_ptr()))
    torch.cuda.synchronize()
    return G, n, float(d[0])


def _halos2(x, a, b):
    Nz = x.shape[0]
    lo2 = torch.full((2,) + tuple(x.shape[1:]), float("nan"), dtype=x.dtype, device="cuda")
    hi2 = torch.full_like(lo2, float("nan"))
    for k in (1, 2):
        if a - k >= 0:
            lo2[2 - k] = x[a - k]
        if b + k - 1 < Nz:
            hi2[k - 1] = x[b + k - 1]
    return (lo2 if a > 0 else None), (hi2 if b < Nz else None)


SLABS = ((0, 2), (2, 3), (3, 7))


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("scheme", SCHEMES)
@pytest.mark.parametrize("M", [4, 12, 16])
def test_slabs_with_time_weight_halos_match_whole_volume_and_oracle(M, scheme, dtype):
    """Three z-slabs, each with its 2-plane image halos and the weight map's planes z = -1 and z = Nz (time_scale_lo / _hi): G and the
    norms bitwise those of the whole-volume call, which matches the oracle; the slab values add up to the whole one."""
    rs = np.random.RandomState(400 + M)
    tdt = torch.float32 if dtype == np.float32 else torch.float64
    did = _lib.F32 if dtype == np.float32 else _lib.F64
    Nz, Ni, Nj = 7, 10, 124
    shape = (Nz, M, Ni, Nj)
    xn = rs.rand(*shape).astype(dtype)
    W = 0.5 + rs.rand(*shape)
    msn = rs.rand(Ni, Nj) > 0.5
    rz, rt, fac = 0.7, 0.3, 2.0
    x = torch.as_tensor(xn).cuda()
    ts = torch.as_tensor(np.sqrt(W)).to(tdt).cuda()                     # the problem carries sqrt of the weight map
    ms = torch.as_tensor(msn.astype(np.uint8)).cuda()
    whole = _lib.make_problem(scheme, did, shape, rz, rt, fac, ms.data_ptr(), 0, Nz, ts.data_ptr())
    G_w, n_w, tv_w = _tv_call(whole, x, None, None)
    kw = dict(reg_z_over_reg=rz, reg_time=rt, mask_static=msn.reshape(1, 1, Ni, Nj), factor_reg_static=fac, time_weight=W)
    _check_tv((tv_w, G_w.cpu().numpy(), n_w.cpu().numpy()), xn, scheme, kw, dtype, "%s whole %s" % (scheme, _path(shape, dtype, kw)))
    tv_parts = 0.0
    for a, b in SLABS:
        pb = _lib.make_problem(scheme, did, (b - a, M, Ni, Nj), rz, rt, fac, ms.data_ptr(), a, Nz, ts[a].data_ptr())
        pb.time_scale_lo = ts[a - 1].data_ptr() if a > 0 else None
        pb.time_scale_hi = ts[b].data_ptr() if b < Nz else None
        lo2, hi2 = _halos2(x, a, b)
        G_s, n_s, tv_s = _tv_call(pb, x[a:b].contiguous(), lo2, hi2)
        assert torch.equal(G_s, G_w[a:b]) and torch.equal(n_s, n_w[a:b]), (a, b)
        tv_parts += tv_s
    assert tv_parts == pytest.approx(tv_w, rel=1e-12)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("scheme", SCHEMES)
def test_slabs_beyond_sixteen_frames(scheme, dtype):
    """M = 17: a weight map on slabs with z halos is refused (only the single-sweep kernel reads the map's halo planes); the same
    slabs without a map run the two-sweep fallback, bitwise equal to the whole volume and matching the oracle."""
    rs = np.random.RandomState(417)
    tdt = torch.float32 if dtype == np.float32 else torch.float64
    did = _lib.F32 if dtype == np.float32 else _lib.F64
    Nz, M, Ni, Nj = 7, 17, 10, 124
    shape = (Nz, M, Ni, Nj)
    xn = rs.rand(*shape).astype(dtype)
    msn = rs.rand(Ni, Nj) > 0.5
    rz, rt, fac = 0.7, 0.3, 2.0
    x = torch.as_tensor(xn).cuda()
    ts = torch.as_tensor(np.sqrt(0.5 + rs.rand(*shape))).to(tdt).cuda()
    ms = torch.as_tensor(msn.astype(np.uint8)).cuda()
    for a, b in SLABS:
        pb = _lib.make_problem(scheme, did, (b - a, M, Ni, Nj), rz, rt, fac, ms.data_ptr(), a, Nz, ts[a].data_ptr())
        pb.time_scale_lo = ts[a - 1].data_ptr() if a > 0 else None
        pb.time_scale_hi = ts[b].data_ptr() if b < Nz else None
        lo2, hi2 = _halos2(x, a, b)
        with pytest.raises(_lib.PytvError, match="time_scale on slabs with z halos needs the single-sweep kernel"):
            _tv_call(pb, x[a:b].contiguous(), lo2, hi2)
    whole = _lib.make_problem(scheme, did, shape, rz, rt, fac, ms.data_ptr(), 0, Nz)
    G_w, n_w, tv_w = _tv_call(whole, x, None, None)
    kw = dict(reg_z_over_reg=rz, reg_time=rt, mask_static=msn.reshape(1, 1, Ni, Nj), factor_reg_static=fac)
    assert _path(shape, dtype, kw) == "fallback"
    _check_tv((tv_w, G_w.cpu().numpy(), n_w.cpu().numpy()), xn, scheme, kw, dtype, "%s whole fallback" % scheme)
    tv_parts = 0.0
    for a, b in SLABS:
        pb = _lib.make_problem(scheme, did, (b - a, M, Ni, Nj), rz, rt, fac, ms.data_ptr(), a, Nz)
        lo2, hi2 = _halos2(x, a, b)
        G_s, n_s, tv_s = _tv_call(pb, x[a:b].contiguous(), lo2, hi2)
        assert torch.equal(G_s, G_w[a:b]) and torch.equal(n_s, n_w[a:b]), (a, b)
        tv_parts += tv_s
    assert tv_parts == pytest.approx(tv_w, rel=1e-12)


# ------------------------------------------------------------------ 3. Chambolle-Pock across the frame-count regimes
CP_M = [1, 2, 3, 5, 8, 9, 12, 17]


def _adj_tile_quads(M):
    """Quads per tile row of the adjoint-split dual pass (adj_core.cuh: adj_tile_quads)."""
    return 256 if M == 1 else (128 if M == 2 else (64 if M <= 4 else 32))


def _cp_shape(M, dtype, Nj=None):
    """33 rows (one past the 32-row tile) and, for the pass pair, one quad past the tile width: every tile class has an interior row
    seam and an interior column seam."""
    vec = 4 if dtype == np.float32 else 2
    return (3, M, 33, Nj if Nj is not None else (_adj_tile_quads(M) if M <= 8 else 32) * vec + vec)


def _cp_tol(dtype, iters=1):
    return dict(atol=1e-12 if iters == 1 else 1e-11, rel=1e-12) if dtype == np.float64 else dict(atol=1e-5, rel=1e-5)


def _cp_state(rs, shape, scheme, dtype):
    Nz, M, Ni, Nj = shape
    kw = _weights(rs, shape, "both")
    Nd = orc.num_components(scheme, Nz, M, kw["reg_z_over_reg"], kw["reg_time"])
    x0 = rs.rand(*shape).astype(dtype)
    x = (x0 + 0.1 * rs.randn(*shape)).astype(dtype)
    xbar = (x + 0.01 * rs.randn(*shape)).astype(dtype)
    y = (0.2 * rs.randn(Nz, Nd, M, Ni, Nj)).astype(dtype)      # non-zero also where the adjoint must ignore it
    return kw, x0, x, xbar, y


def _f64(*a):
    return [v.astype(np.float64) for v in a]


def _solver(x0, scheme, kw, M, **opts):
    s = pytv.CPSolver(x0, lam=0.1, scheme=scheme, sigma=0.5, tau=0.07, **dict(kw, **opts))
    assert s._adj == (M <= 8 and opts.get("variant", "rof") == "rof"), (M, s._adj)
    return s


def _close(a, b, atol, what):
    np.testing.assert_allclose(a.cpu().numpy() if isinstance(a, torch.Tensor) else a, b, rtol=0, atol=atol, err_msg=what)


def _cp_cases():
    cases = [pytest.param(M, None, id="M%d" % M) for M in CP_M]
    return cases + [pytest.param(5, 65, id="M5_scalar"), pytest.param(12, 65, id="M12_scalar")]


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("scheme", SCHEMES)
@pytest.mark.parametrize("M,Nj", _cp_cases())
def test_cp_one_iteration_from_a_random_state(M, Nj, scheme, dtype):
    """(a) ROF form, one iteration from a random (x, xbar, y) against orc.cp_rof_step: the pass pair for M <= 8, the two-pass kernels
    beyond; time-weight map and mask_static on; an odd row length for the scalar forms."""
    rs = np.random.RandomState(500 + M)
    shape = _cp_shape(M, dtype, Nj)
    kw, x0, x, xbar, y = _cp_state(rs, shape, scheme, dtype)
    s = _solver(x0, scheme, kw, M, theta=0.9)
    s.x.copy_(torch.as_tensor(x)); s.aux.copy_(torch.as_tensor(xbar)); s.y.copy_(torch.as_tensor(y))
    s.step()
    xr, xbr, yr, er = orc.cp_rof_step(*_f64(x, xbar, x0, y), scheme, lam=0.1, sigma=0.5, tau=0.07, theta=0.9, **kw)
    t = _cp_tol(dtype)
    what = "%s %s %s" % (scheme, shape, "pass pair" if s._adj else "two-pass")
    _close(s.y, yr, t["atol"], what)
    _close(s.x, xr, t["atol"], what)
    _close(s.aux, xbr, t["atol"], what)
    assert s.energy() == pytest.approx(er, rel=t["rel"]), what


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("scheme", SCHEMES)
@pytest.mark.parametrize("M", CP_M, ids=["M%d" % M for M in CP_M])
def test_cp_ten_iterations_energy_and_gap(M, scheme, dtype):
    """(b) Ten iterations from the start against the oracle: iterates, the energy of the last iteration, and the primal and dual
    energies of the duality gap (P = 0.5|x - x0|^2 + lam TV(x), D = 0.5|x0|^2 - 0.5|x0 - D^T y|^2)."""
    rs = np.random.RandomState(600 + M)
    shape = _cp_shape(M, dtype)
    kw, x0, _, _, _ = _cp_state(rs, shape, scheme, dtype)
    s = _solver(x0, scheme, kw, M, theta=1.0)
    s.step(10)
    x064 = x0.astype(np.float64)
    x, xb, y = x064.copy(), x064.copy(), np.zeros((shape[0], s.Nd) + shape[1:])
    for _ in range(10):
        x, xb, y, e = orc.cp_rof_step(x, xb, x064, y, scheme, lam=0.1, sigma=0.5, tau=0.07, theta=1.0, **kw)
    t = _cp_tol(dtype, 10)
    what = "%s %s %s" % (scheme, shape, "pass pair" if s._adj else "two-pass")
    _close(s.x, x, t["atol"], what)
    _close(s.aux, xb, t["atol"], what)
    _close(s.y, y, t["atol"], what)
    assert s.energy() == pytest.approx(e, rel=t["rel"]), what
    p, d, g = s.gap()
    p_o = 0.5 * np.sum((x - x064) ** 2) + 0.1 * orc.l21(orc.D(x, scheme, **kw))
    d_o = 0.5 * np.sum(x064 ** 2) - 0.5 * np.sum((x064 - orc.D_T(y, scheme, **kw)) ** 2)
    assert p == pytest.approx(p_o, rel=t["rel"]) and d == pytest.approx(d_o, rel=t["rel"]), what
    assert g == p - d and g > 0


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("scheme", SCHEMES)
@pytest.mark.parametrize("M", CP_M, ids=["M%d" % M for M in CP_M])
def test_cp_data_terms_across_frame_regimes(M, scheme, dtype):
    """(c) TV-L1 and weighted L2 (weights 0 on every third row: missing data), one iteration from a random state against
    data_term_oracle.cp_data_step."""
    rs = np.random.RandomState(700 + M)
    shape = _cp_shape(M, dtype)
    kw, x0, x, xbar, y = _cp_state(rs, shape, scheme, dtype)
    w = 2.0 * rs.rand(*shape)
    w[:, :, ::3] = 0
    w = w.astype(dtype)
    t = _cp_tol(dtype)
    for term, ww in (("l1", None), ("l2", w)):
        s = _solver(x0, scheme, kw, M, theta=0.9, data_term=term, data_weight=ww)
        s.x.copy_(torch.as_tensor(x)); s.aux.copy_(torch.as_tensor(xbar)); s.y.copy_(torch.as_tensor(y))
        s.step()
        xr, xbr, yr, er = dto.cp_data_step(*_f64(x, xbar, x0, y), term, None if ww is None else ww.astype(np.float64), scheme, lam=0.1, sigma=0.5,
                                           tau=0.07, theta=0.9, **kw)
        what = "%s %s %s %s" % (term, scheme, shape, "pass pair" if s._adj else "two-pass")
        _close(s.y, yr, t["atol"], what)
        _close(s.x, xr, t["atol"], what)
        _close(s.aux, xbr, t["atol"], what)
        assert s.energy() == pytest.approx(er, rel=t["rel"]), what


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("scheme", SCHEMES)
def test_cp_readme_form_at_twelve_frames(scheme, dtype):
    """(d) The README iteration (dual fidelity variable, no over-relaxation) at M = 12 against orc.cp_readme_step."""
    M = 12
    rs = np.random.RandomState(812)
    shape = _cp_shape(M, dtype)
    kw, x0, x, _, y = _cp_state(rs, shape, scheme, dtype)
    y_f = (0.1 * rs.randn(*shape)).astype(dtype)
    s = _solver(x0, scheme, kw, M, variant="readme", sigma_A=0.8)
    s.x.copy_(torch.as_tensor(x)); s.aux.copy_(torch.as_tensor(y_f)); s.y.copy_(torch.as_tensor(y))
    s.step()
    x64, x064, yf64, y64 = _f64(x, x0, y_f, y)
    xr, yfr, yr, er = orc.cp_readme_step(x64, x064, yf64, y64, scheme, lam=0.1, sigma_D=0.5, sigma_A=0.8, tau=0.07, **kw)
    t = _cp_tol(dtype)
    _close(s.y, yr, t["atol"], scheme)
    _close(s.x, xr, t["atol"], scheme)
    _close(s.aux, yfr, t["atol"], scheme)
    assert s.energy() == pytest.approx(er, rel=t["rel"]), scheme


# ------------------------------------------------------------------ 4. half-precision dual storage at M = 12
@pytest.mark.parametrize("scheme", SCHEMES)
def test_half_precision_dual_storage_at_twelve_frames(scheme):
    """y stored as y / lam in IEEE half through the two-pass kernels: equal, up to one half-ulp flip of y (which moves x by
    tau * lam * 2^-11 ~ 3.5e-6), to a float32 run whose dual field is rounded to half after every dual pass, over 3 iterations."""
    g = torch.Generator().manual_seed(12)
    x0 = torch.rand((6, 12, 32, 64), generator=g).cuda()
    kw = dict(lam=0.1, scheme=scheme, variant="rof", reg_time=0.25)
    emu = pytv.CPSolver(x0, **kw)
    assert not emu._adj
    for _ in range(3):
        emu._pass_A()
        emu.y.copy_(((emu.y / emu.lam).half().float()) * emu.lam)
        emu._pass_B()
    h3 = pytv.CPSolver(x0, dual_dtype=torch.float16, **kw)
    assert h3.y.dtype == torch.float16
    h3.step(3)
    assert float((h3.x - emu.x).abs().max()) < 3e-5

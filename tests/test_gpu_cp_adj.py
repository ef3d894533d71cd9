"""The Chambolle-Pock pass pair that finishes the in-plane and time terms of the adjoint in the dual pass
(pytvb_cp_dual_adj + pytvb_cp_primal_adj) against the two-pass entry points (pytvb_cp_dual + pytvb_cp_primal_rof /
pytvb_cp_primal_data): the iterates must be equal bit for bit, over several iterations, for every scheme and precision, the
time-axis options, tile edges (rows not a multiple of the 32-row tile, columns not a multiple of the column block, the
scalar path), M = 1 .. 8, slabs with halo planes and the peer-push schedule."""
import ctypes

import pytest
import torch

import p2p_schedule
from pytv_b200 import _dev, _lib, cp

pytestmark = pytest.mark.gpu
L2, L1 = 0, 1


def _state(shape, dtype, Nd, seed, halo):
    g = torch.Generator().manual_seed(seed)
    rnd = lambda *s: torch.rand(s, generator=g, dtype=torch.float64).to(dtype).cuda()
    Nz, M, Ni, Nj = shape
    st = dict(x0=rnd(*shape), y=torch.zeros((Nz, Nd, M, Ni, Nj), dtype=dtype, device="cuda"))
    st["x"], st["xbar"] = st["x0"].clone(), st["x0"].clone()
    st["w"] = rnd(*shape) * 2.0
    st["w"][..., 0, :] = 0.0                                  # missing data
    st["ts"] = rnd(*shape) + 0.5
    if halo:   # an interior slab: fixed image and field halo planes on both sides
        st["img_lo"], st["img_hi"] = rnd(M, Ni, Nj), rnd(M, Ni, Nj)
        st["fld_lo"], st["fld_hi"] = rnd(M, Ni, Nj) * 0.05, rnd(M, Ni, Nj) * 0.05
    return st


def _iterate(new, scheme, dtype, shape, iters=3, term=None, weight=False, rt=0.25, mask=False, tw=False, halo=False, lam=0.1):
    Nz, M, Ni, Nj = shape
    lib = _lib.lib()
    code = _lib.F32 if dtype == torch.float32 else _lib.F64
    z_on, t_on = True, M > 1 and rt > 0
    Nd = (4 + 2 * z_on + 2 * t_on) if scheme == "hybrid" else (2 + z_on + t_on)
    st = _state(shape, dtype, Nd, 5, halo)
    ms = None
    if mask:
        ms = (torch.arange(Ni * Nj, device="cuda").reshape(Ni, Nj) % 3 == 0).to(torch.uint8)
    pb = _lib.make_problem(scheme, code, shape, 0.7, rt, 2.0 if mask else 0.0, ms.data_ptr() if ms is not None else None, 1 if halo else 0,
                           Nz + 2 if halo else Nz, st["ts"].data_ptr() if tw else None)
    ws = _dev.reduce_workspace(pb, torch.device("cuda"))
    q = torch.full_like(st["x0"], float("nan"))
    scal = torch.zeros(2 * iters, dtype=torch.float64, device="cuda")
    P = lambda k: _dev.ptr(st.get(k))
    s = _dev.stream_ptr()
    sigma, tau, theta = 0.5, 0.07, 0.9
    w = P("w") if weight else None
    for it in range(iters):
        d1, d2 = _dev.ptr(scal[2 * it:2 * it + 1]), _dev.ptr(scal[2 * it + 1:2 * it + 2])
        if new:
            _lib.check(lib.pytvb_cp_dual_adj(ctypes.byref(pb), P("xbar"), P("y"), _dev.ptr(q), lam, sigma, d1, P("img_lo"), P("img_hi"), _dev.ptr(ws), s))
            _lib.check(lib.pytvb_cp_primal_adj(ctypes.byref(pb), L2 if term is None else term, w, P("y"), _dev.ptr(q), P("x"), P("xbar"), P("x0"), tau,
                                               theta, d2, P("fld_lo"), P("fld_hi"), _dev.ptr(ws), s))
        else:
            _lib.check(lib.pytvb_cp_dual(ctypes.byref(pb), P("xbar"), P("y"), lam, sigma, d1, P("img_lo"), P("img_hi"), _dev.ptr(ws), s))
            if term is None:
                _lib.check(lib.pytvb_cp_primal_rof(ctypes.byref(pb), P("y"), P("x"), P("xbar"), P("x0"), tau, theta, d2, P("fld_lo"), P("fld_hi"),
                                                   _dev.ptr(ws), s))
            else:
                _lib.check(lib.pytvb_cp_primal_data(ctypes.byref(pb), term, w, P("y"), P("x"), P("xbar"), P("x0"), tau, theta, d2, P("fld_lo"),
                                                    P("fld_hi"), None, None, _dev.ptr(ws), s))
    torch.cuda.synchronize()
    return st["x"], st["xbar"], st["y"], scal.cpu()


def _same(shape, scheme="hybrid", dtype=torch.float32, **kw):
    a = _iterate(False, scheme, dtype, shape, **kw)
    b = _iterate(True, scheme, dtype, shape, **kw)
    for u, v in zip(a[:3], b[:3]):
        assert torch.equal(u, v)
    assert bool(torch.isfinite(b[0]).all())
    # the L21 and fidelity partial sums: the same per-thread float partials, summed in another order in double
    assert torch.allclose(a[3], b[3], rtol=1e-12, atol=0.0)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("scheme", ["upwind", "downwind", "central", "hybrid"])
@pytest.mark.parametrize("shape", [(3, 4, 70, 520), (2, 3, 33, 130), (2, 8, 65, 100), (2, 8, 40, 300), (2, 6, 40, 264), (3, 1, 40, 1030),
                                   (2, 2, 31, 77)],
                         ids=["M4", "M3", "M8", "M8_two_blocks", "M6", "M1", "M2_scalar"])
def test_adj_pair_equals_two_pass(shape, scheme, dtype):
    _same(shape, scheme, dtype)


@pytest.mark.parametrize("scheme", ["upwind", "downwind", "central", "hybrid"])
@pytest.mark.parametrize("opts", [dict(mask=True), dict(tw=True), dict(mask=True, tw=True), dict(halo=True), dict(halo=True, tw=True)],
                         ids=["mask_static", "time_weight", "both", "halo", "halo_time_weight"])
def test_adj_pair_time_options_and_halos(scheme, opts):
    _same((3, 4, 67, 260), scheme, torch.float32, **opts)
    _same((2, 3, 35, 66), scheme, torch.float64, **opts)


@pytest.mark.parametrize("scheme", ["central", "hybrid"])
@pytest.mark.parametrize("term,weight", [(L2, True), (L1, False), (L1, True)], ids=["l2_weighted", "l1", "l1_weighted"])
def test_adj_pair_data_terms(scheme, term, weight):
    _same((3, 4, 67, 260), scheme, torch.float32, term=term, weight=weight, tw=True)
    _same((2, 2, 35, 66), scheme, torch.float64, term=term, weight=weight, halo=True)


def test_adj_pair_length_two_axes_and_one_row():
    for shape in ((2, 2, 1, 64), (2, 2, 2, 8), (3, 4, 64, 256)):
        for scheme in ("central", "hybrid", "upwind"):
            _same(shape, scheme, torch.float32)


def test_adj_rejects_more_than_eight_frames():
    pb = _lib.make_problem("hybrid", _lib.F32, (2, 9, 8, 8), 1.0, 0.1)
    x = torch.zeros((2, 9, 8, 8), device="cuda")
    with pytest.raises(_lib.PytvError):
        _lib.check(_lib.lib().pytvb_cp_dual_adj(ctypes.byref(pb), _dev.ptr(x), _dev.ptr(x), _dev.ptr(x), 0.1, 0.5, None, None, None, None,
                                                _dev.stream_ptr()))


class _AdjOps(cp.CudaOps):
    """The push schedule of tests/p2p_schedule.py with the adjoint-split passes (ROF form); one q image per y buffer."""

    def __init__(self):
        super().__init__()
        self.q = {}

    def _q(self, y):
        k = y.data_ptr()
        if k not in self.q:
            self.q[k] = torch.empty((y.shape[0],) + tuple(y.shape[2:]), dtype=y.dtype, device=y.device)
        return self.q[k]

    def cp_dual_p2p(self, pb, xbar, y, lam, sigma, d_l21, lo, hi, mirror_prev, mirror_next, ws):
        self.cp_dual_adj(pb, xbar, y, self._q(y), lam, sigma, d_l21, lo, hi, mirror_prev, mirror_next, ws)

    def cp_primal_p2p(self, variant, pb, y, x, aux, x0, tau, c2, d_fid, lo, hi, mirror_prev, mirror_next, ws):
        assert variant == "rof"
        self.cp_primal_adj(pb, "l2", None, y, self._q(y), x, aux, x0, tau, c2, d_fid, lo, hi, mirror_prev, mirror_next, ws)


@pytest.mark.parametrize("scheme", ["upwind", "downwind", "central", "hybrid"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
def test_adj_push_schedule_on_one_device(scheme, dtype):
    slabs, _ = p2p_schedule.run(_AdjOps(), torch.device("cuda", 0), scheme, "rof", dtype, shape=(7, 3, 70, 520), bounds=((0, 2), (2, 3), (3, 7)))
    _, whole = p2p_schedule.run(cp.CudaOps(), torch.device("cuda", 0), scheme, "rof", dtype, shape=(7, 3, 70, 520), bounds=((0, 2), (2, 3), (3, 7)))
    torch.cuda.synchronize()
    for a, b in zip(slabs, whole):
        assert torch.equal(a, b)


@pytest.mark.parametrize("opts", [dict(), dict(data_term="l1"), dict(data_weight="w")], ids=["rof", "l1", "l2_weighted"])
def test_solver_takes_the_adj_pair_and_matches_the_two_pass_entry_points(opts):
    shape = (4, 4, 96, 264)
    g = torch.Generator().manual_seed(3)
    x0 = torch.rand(shape, generator=g).cuda()
    if opts.get("data_weight") == "w":
        opts = dict(data_weight=torch.rand(shape, generator=g).cuda())
    s = cp.CPSolver(x0, lam=0.1, reg_time=0.1, **opts)
    assert s._adj and s.q is not None
    s.step(1)
    x, xbar, y = s.x.clone(), s.aux.clone(), s.y.clone()
    s.step(2)
    lib, st = _lib.lib(), _dev.stream_ptr()
    term = L1 if opts.get("data_term") == "l1" else L2
    w = opts.get("data_weight")
    for _ in range(2):
        _lib.check(lib.pytvb_cp_dual(ctypes.byref(s.pb), _dev.ptr(xbar), _dev.ptr(y), s.lam, s.sigma, None, None, None, _dev.ptr(s.ws), st))
        _lib.check(lib.pytvb_cp_primal_data(ctypes.byref(s.pb), term, _dev.ptr(s._dw) if w is not None else None, _dev.ptr(y), _dev.ptr(x),
                                            _dev.ptr(xbar), _dev.ptr(s.x0), s.tau, s.theta, None, None, None, None, None, _dev.ptr(s.ws), st))
    torch.cuda.synchronize()
    assert torch.equal(x, s.x) and torch.equal(xbar, s.aux) and torch.equal(y, s.y)
    assert not cp.CPSolver(torch.rand((2, 9, 16, 16)).cuda(), lam=0.1, reg_time=0.1)._adj      # M > 8: two-pass kernels
    assert not cp.CPSolver(x0, lam=0.1, variant="readme")._adj

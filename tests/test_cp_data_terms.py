"""The L1 and weighted-L2 data terms of the Chambolle-Pock solver, without a GPU: the numpy reference (prox optimality,
known answers), the per-quad CUDA code of the new primal pass run on the host (tests/emul/emul_data.cu) against it, the
sharded solver logic over gloo, and the argument check of the C entry point."""
import ctypes
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import data_term_oracle as dto  # noqa: E402
import emul_helper as em  # noqa: E402
from oracle import tv_oracle as orc  # noqa: E402
from pytv_b200 import _lib  # noqa: E402

SCHEMES = orc.SCHEMES
EMUL_SRC = os.path.join(ROOT, "tests", "emul", "emul_data.cu")
EMUL_SO = os.path.join(ROOT, "tests", "emul", "libpytvb_emul_data.so")
L1, L2 = 1, 0


_emul_data_handle = None


def _emul_data():
    """The host emulation library, built when a source is newer than it; loaded once per process."""
    global _emul_data_handle
    if _emul_data_handle is not None:
        return _emul_data_handle
    deps = [EMUL_SRC] + [os.path.join(ROOT, "pytv-4d_b200", "csrc", f) for f in ("core.cuh", "strip_core.cuh", "kernels.cuh", "host_common.cuh")]
    deps.append(os.path.join(ROOT, "include", "pytv_b200.h"))
    if not (os.path.exists(EMUL_SO) and all(os.path.getmtime(EMUL_SO) >= os.path.getmtime(d) for d in deps)):
        subprocess.run(["nvcc", "-O1", "-std=c++17", "-Xcompiler", "-fPIC", "-shared", "-gencode", "arch=compute_100a,code=sm_100a", EMUL_SRC, "-o",
                        EMUL_SO], check=True, cwd=os.path.dirname(EMUL_SRC))
    h = ctypes.CDLL(EMUL_SO)
    VP = ctypes.c_void_p
    h.pytvb_emulate_data.restype = ctypes.c_int
    h.pytvb_emulate_data.argtypes = [ctypes.POINTER(_lib.Problem), ctypes.c_int] + [VP] * 9 + [ctypes.c_double, ctypes.c_double, ctypes.c_int,
                                                                                              ctypes.POINTER(ctypes.c_double)]
    h.pytvb_emulate_data_error.restype = ctypes.c_char_p
    _emul_data_handle = h
    return h


@pytest.fixture(scope="module")
def emul_data():
    return _emul_data()


def _p(a):
    if a is None:
        return None
    return ctypes.c_void_p(a.data_ptr()) if isinstance(a, torch.Tensor) else a.ctypes.data_as(ctypes.c_void_p)


def emul_pass_B(h, term, w, y, x, xbar, x0, scheme, tau, theta, lo=None, hi=None, mp_=None, mn=None, z_offset=0, Nz_global=None, scalar=False,
                **kw):
    """One primal pass of the new kernel code on the host; x and xbar are updated in place; returns the fidelity partial sum."""
    pb, keep = em._problem(scheme, x.dtype, x.shape, kw.get("reg_z_over_reg", 1.0), kw.get("reg_time", 0.0), kw.get("mask_static", False),
                           kw.get("factor_reg_static", 0.0), z_offset, Nz_global, kw.get("time_weight"))
    s = ctypes.c_double(0)
    rc = h.pytvb_emulate_data(ctypes.byref(pb), term, _p(w), _p(np.ascontiguousarray(y)), _p(x), _p(xbar), _p(x0), _p(lo), _p(hi), _p(mp_), _p(mn),
                              tau, theta, int(scalar), ctypes.byref(s))
    assert rc == 0, h.pytvb_emulate_data_error()
    return s.value


def _fid(x, x0, term, w):
    r = (x - x0).astype(np.float64)
    w = np.ones_like(r) if w is None else np.broadcast_to(np.asarray(w, dtype=np.float64), r.shape)
    return float(np.sum(w * r * r)) if term == "l2" else float(np.sum(w * np.abs(r)))


# ------------------------------------------------------------------ the numpy reference
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("scheme", SCHEMES)
def test_oracle_l2_unit_weight_is_rof(scheme, dtype):
    rs = np.random.RandomState(3)
    shape = (3, 2, 6, 8)
    kw = dict(reg_z_over_reg=0.5, reg_time=0.25)
    x0 = rs.rand(*shape).astype(dtype)
    x, xb = (x0 + 0.1 * rs.randn(*shape)).astype(dtype), (x0 + 0.1 * rs.randn(*shape)).astype(dtype)
    y = (0.1 * rs.randn(shape[0], orc.num_components(scheme, 3, 2, 0.5, 0.25), *shape[1:])).astype(dtype)
    for w in (None, np.ones(shape)):
        a = dto.cp_data_step(x, xb, x0, y, "l2", w, scheme, lam=0.1, sigma=0.5, tau=0.07, theta=0.9, **kw)
        b = orc.cp_rof_step(x, xb, x0, y, scheme, lam=0.1, sigma=0.5, tau=0.07, theta=0.9, **kw)
        for u, v in zip(a[:3], b[:3]):
            assert u.dtype == v.dtype and np.array_equal(u, v)
        assert a[3] == b[3]


@pytest.mark.parametrize("scheme", SCHEMES)
def test_oracle_prox_optimality(scheme):
    """L2: (x - v) + tau w (x - x0) = 0;  L1: |x - v| <= tau w, with equality where x != x0 (v = x_old - tau D^T y_new)."""
    rs = np.random.RandomState(4)
    shape = (2, 3, 7, 6)
    x0 = rs.rand(*shape)
    x, xb = x0 + 0.2 * rs.randn(*shape), x0 + 0.2 * rs.randn(*shape)
    y = 0.2 * rs.randn(shape[0], orc.num_components(scheme, 2, 3), *shape[1:])
    w = rs.rand(*shape) * 3
    w[0, 0, :2] = 0
    tau = 0.1
    for term in ("l2", "l1"):
        xn, _, yn, _ = dto.cp_data_step(x, xb, x0, y, term, w, scheme, lam=0.15, sigma=0.5, tau=tau, theta=1.0)
        v = x - tau * orc.D_T(yn, scheme)
        if term == "l2":
            np.testing.assert_allclose((xn - v) + tau * w * (xn - x0), 0, atol=1e-14)
        else:
            assert np.all(np.abs(xn - v) <= tau * w + 1e-14)
            moved = xn != x0
            np.testing.assert_allclose(np.abs(xn - v)[moved], (tau * w)[moved], atol=1e-14)
            assert moved.any() and (~moved).any()


def test_oracle_inpainting_known_answer():
    """A constant image with garbage under a w = 0 hole: TV fills the hole with the constant."""
    c = 0.7
    x0 = np.full((1, 2, 12, 12), c)
    w = np.ones_like(x0)
    x0[0, :, 4:8, 3:9] = np.random.RandomState(5).rand(2, 4, 6) * 5
    w[0, :, 4:8, 3:9] = 0
    for term in ("l2", "l1"):
        x, _, _, _ = dto.run(x0, 1500, term, w, "hybrid", lam=0.1, sigma=0.5, tau=1.0 / 17.0, reg_time=0.5)
        np.testing.assert_allclose(x, c, atol=1e-5)


@pytest.mark.parametrize("h", [1.0, 7.0])
@pytest.mark.parametrize("lam,kept", [(0.2, True), (0.27, True), (0.31, False), (0.45, False)])
def test_oracle_tv_l1_impulse_threshold(h, lam, kept):
    """Upwind 2-D TV-L1: one interior impulse of height h costs (2 + sqrt 2) h of TV against h of fidelity, so it is kept for
    lam < 1 / (2 + sqrt 2) ~ 0.293 and removed above, whatever h (contrast invariance)."""
    x0 = np.zeros((1, 1, 9, 9))
    x0[0, 0, 4, 4] = h
    x, _, _, _ = dto.run(x0, 3000, "l1", None, "upwind", lam=lam, sigma=0.5, tau=1.0 / 9.0)
    np.testing.assert_allclose(x, x0 if kept else 0.0, atol=1e-3 * h)


# ------------------------------------------------------------------ the kernel code on the host
def _state(rs, shape, scheme, dtype, kw):
    Nz, M = shape[:2]
    x0 = rs.rand(*shape)
    x = x0 + 0.1 * rs.randn(*shape)
    xb = x + 0.01 * rs.randn(*shape)
    y = 0.2 * rs.randn(Nz, orc.num_components(scheme, Nz, M, kw.get("reg_z_over_reg", 1.0), kw.get("reg_time", 0.0)), *shape[1:])
    w = 2.0 * rs.rand(*shape)
    w[:, :, ::3] = 0
    return [a.astype(dtype) for a in (x0, x, xb, y)] + [w.astype(dtype)]


FORMS = [("l1", False), ("l1", True), ("l2", True)]


@pytest.mark.parametrize("scalar", [False, True], ids=["vec", "scalar"])
@pytest.mark.parametrize("weights", [False, True], ids=["plain", "tw_mask"])
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("scheme", SCHEMES)
def test_emulated_pass_B_matches_oracle(emul_data, scheme, dtype, weights, scalar):
    rs = np.random.RandomState(6)
    shape = (3, 3, 6, 8)
    kw = dict(reg_z_over_reg=0.6, reg_time=0.4)
    if weights:
        kw.update(mask_static=rs.rand(1, 1, 6, 8) > 0.5, factor_reg_static=3.0, time_weight=0.5 + rs.rand(*shape))
    x0, x, xb, y, w = _state(rs, shape, scheme, dtype, kw)
    tol = 1e-12 if dtype == np.float64 else 1e-5
    for term, use_w in FORMS:
        ww = w if use_w else None
        xr, xbr, yr, _ = dto.cp_data_step(x, xb, x0, y, term, ww, scheme, lam=0.1, sigma=0.5, tau=0.07, theta=0.9, **kw)
        xe, xbe = x.copy(), np.full_like(x, np.nan)
        fid = emul_pass_B(emul_data, L1 if term == "l1" else L2, ww, yr, xe, xbe, x0, scheme, 0.07, 0.9, scalar=scalar, **kw)
        np.testing.assert_allclose(xe, xr, atol=tol)
        np.testing.assert_allclose(xbe, xbr, atol=tol)
        assert fid == pytest.approx(_fid(xr, x0, term, ww), rel=10 * tol)


@pytest.mark.parametrize("scalar", [False, True], ids=["vec", "scalar"])
@pytest.mark.parametrize("scheme", SCHEMES)
def test_emulated_pass_B_slab_and_mirror_stores(emul_data, scheme, scalar):
    """Planes [1, 4) of a 5-plane volume with the field halos from the neighbours equal the whole-volume pass; the mirror
    stores put the slab's first / last xbar plane into the neighbours' image halo planes."""
    rs = np.random.RandomState(7)
    shape = (5, 2, 5, 12)
    kw = dict(reg_z_over_reg=0.5, reg_time=0.3)
    x0, x, xb, y, w = _state(rs, shape, scheme, np.float64, kw)
    tw = 0.5 + rs.rand(*shape)
    zf, zb = (4, 5) if scheme == "hybrid" else (2, 2)
    for term, use_w in FORMS:
        ww = w if use_w else None
        xa, xba = x.copy(), np.zeros_like(x)
        emul_pass_B(emul_data, L1 if term == "l1" else L2, ww, y, xa, xba, x0, scheme, 0.07, 1.0, time_weight=tw, scalar=scalar, **kw)
        xs, xbs = x[1:4].copy(), np.zeros_like(x[1:4])
        mp_, mn = np.full(shape[1:], np.nan), np.full(shape[1:], np.nan)
        emul_pass_B(emul_data, L1 if term == "l1" else L2, None if ww is None else np.ascontiguousarray(ww[1:4]), y[1:4], xs, xbs, x0[1:4].copy(),
                    scheme, 0.07, 1.0, lo=np.ascontiguousarray(y[0, zf]), hi=np.ascontiguousarray(y[4, zb]), mp_=mp_, mn=mn, z_offset=1, Nz_global=5,
                    time_weight=np.ascontiguousarray(tw[1:4]), scalar=scalar, **kw)
        assert np.array_equal(xs, xa[1:4]) and np.array_equal(xbs, xba[1:4])
        assert np.array_equal(mp_, xbs[0]) and np.array_equal(mn, xbs[-1])


def test_emulated_pass_B_odd_width(emul_data):
    """Nj = 7: every pointer takes the scalar path."""
    rs = np.random.RandomState(8)
    shape = (2, 2, 5, 7)
    for dtype in (np.float64, np.float32):
        x0, x, xb, y, w = _state(rs, shape, "hybrid", dtype, dict(reg_time=0.5))
        for term, use_w in FORMS:
            ww = w if use_w else None
            xr, xbr, yr, _ = dto.cp_data_step(x, xb, x0, y, term, ww, "hybrid", lam=0.1, sigma=0.5, tau=0.07, theta=1.0, reg_time=0.5)
            xe, xbe = x.copy(), np.zeros_like(x)
            emul_pass_B(emul_data, L1 if term == "l1" else L2, ww, yr, xe, xbe, x0, "hybrid", 0.07, 1.0, reg_time=0.5)
            np.testing.assert_allclose(xe, xr, atol=1e-12 if dtype == np.float64 else 1e-5)


# ------------------------------------------------------------------ sharded solver logic over gloo
class EmulDataOps(em.EmulOps):
    """EmulOps with the primal pass of the other data terms (the host emulation of cp_primal_data_strip_kernel)."""

    def cp_primal_data(self, pb, data_term, w, y, x, xbar, x0, tau, theta, d_fid, lo, hi, mirror_prev, mirror_next, ws):
        s = ctypes.c_double(0.0)
        rc = _emul_data().pytvb_emulate_data(ctypes.byref(pb), L1 if data_term == "l1" else L2, self._p(w), self._p(y), self._p(x), self._p(xbar),
                                             self._p(x0), self._p(lo), self._p(hi), mirror_prev, mirror_next, tau, theta, 0, ctypes.byref(s))
        assert rc == 0
        if d_fid is not None:
            d_fid[0] = s.value

    # what primal_energy / dual_energy need: the adjoint and the TV value of a slab with one halo plane per side
    def adjoint(self, pb, y, out, lo, hi):
        rc = em.emul().pytvb_emulate(8, ctypes.byref(pb), self._p(y), self._p(out), None, None, None, self._p(lo), self._p(hi), 0.0, 0.0, 0, 0, None)
        assert rc == 0

    def tv_value(self, pb, x, d_tv, lo, hi, ws):
        D = torch.empty((x.shape[0], em.nd_of(pb)) + tuple(x.shape[1:]), dtype=x.dtype)
        rc = em.emul().pytvb_emulate(7, ctypes.byref(pb), self._p(x), self._p(D), None, None, None, self._p(lo), self._p(hi), 0.0, 0.0, 0, 0, None)
        assert rc == 0
        d_tv[0] = float(torch.sqrt((D.double() ** 2).sum(dim=1)).sum())


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gloo_problem():
    rs = np.random.RandomState(19)
    Nz, M, N = 5, 2, 8
    x0 = rs.rand(Nz, M, N, N)
    w = 0.2 + 2 * rs.rand(Nz, M, N, N)
    return x0, w, dict(reg_z_over_reg=0.5, reg_time=0.25, lam=0.15, scheme="hybrid")


def _run_solver(x0, w, kw, term, n=4, **extra):
    import pytv_b200
    s = pytv_b200.CPSolver(x0, data_term=term, data_weight=w, ops=EmulDataOps(), **kw, **extra)
    energies = []
    for _ in range(n):
        s.step()
        energies.append(s.energy())
    return s, energies


def _gloo_worker(rank, world, port, term, use_w, overlap, out_dir):
    os.environ["PYTVB_OVERLAP"] = overlap
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    import pytv_b200
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        x0, w, kw = _gloo_problem()
        off, cnt = pytv_b200.partition_z(x0.shape[0], world)[rank]
        s, energies = _run_solver(x0[off:off + cnt], w[off:off + cnt] if use_w else None, kw, term, distributed=True)
        np.save(os.path.join(out_dir, "x_%d.npy" % rank), s.result())
        np.save(os.path.join(out_dir, "y_%d.npy" % rank), s.y.numpy())
        gap = s.gap()           # cross-rank reductions of the dual energy (sum; max of |D^T y| / w for L1)
        s.step()                # the diagnostics reuse the halo buffers: iterating on afterwards must still work
        e_after = s.energy()
        if rank == 0:
            np.save(os.path.join(out_dir, "energies.npy"), np.array(energies + list(gap) + [e_after]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("overlap", ["0", "1"], ids=["blocking", "overlap"])
@pytest.mark.parametrize("term,use_w", [("l1", False), ("l1", True), ("l2", True)], ids=["l1", "l1_w", "l2_w"])
def test_sharded_data_terms_equal_single_rank(tmp_path, emul_data, term, use_w, overlap):
    mp.spawn(_gloo_worker, args=(2, _free_port(), term, use_w, overlap, str(tmp_path)), nprocs=2, join=True)
    x = np.concatenate([np.load(tmp_path / ("x_%d.npy" % r)) for r in range(2)], axis=0)
    y = np.concatenate([np.load(tmp_path / ("y_%d.npy" % r)) for r in range(2)], axis=0)
    x0, w, kw = _gloo_problem()
    s, energies = _run_solver(x0, w if use_w else None, kw, term)
    assert np.array_equal(x, s.result()) and np.array_equal(y, s.y.numpy())
    e = np.load(tmp_path / "energies.npy")
    np.testing.assert_allclose(e[:4], energies, rtol=1e-13)
    p, d, g = s.gap()
    np.testing.assert_allclose(e[4:6], [p, d], rtol=1e-12)          # other summation grouping
    assert abs(e[6] - g) <= 1e-12 * abs(p) and g >= 0
    assert d == pytest.approx(dto.dual_energy(s.y.numpy(), x0, term, w if use_w else None, "hybrid", reg_z_over_reg=0.5, reg_time=0.25), rel=1e-12)
    assert p == pytest.approx(dto.primal_energy(s.result(), x0, term, w if use_w else None, "hybrid", 0.15, reg_z_over_reg=0.5, reg_time=0.25),
                              rel=1e-12)
    # and the single-rank run is the reference's iteration
    xr, _, _, er = dto.run(x0, 4, term, w if use_w else None, "hybrid", lam=0.15, sigma=0.5, tau=s.tau, theta=1.0, reg_z_over_reg=0.5, reg_time=0.25)
    np.testing.assert_allclose(s.result(), xr, atol=1e-13)
    assert energies[-1] == pytest.approx(er, rel=1e-12)
    s.step()
    assert e[7] == pytest.approx(s.energy(), rel=1e-13)


# ------------------------------------------------------------------ solver options and the C entry point (no compute)
def test_solver_rejects_bad_data_options():
    import pytv_b200
    x0 = np.random.RandomState(0).rand(2, 1, 4, 8)
    ops = EmulDataOps()
    with pytest.raises(ValueError):
        pytv_b200.CPSolver(x0, 0.1, data_term="huber", ops=ops)
    for bad in (-1.0, np.nan, np.inf):
        w = np.ones_like(x0)
        w[0, 0, 1, 1] = bad
        with pytest.raises(ValueError):
            pytv_b200.CPSolver(x0, 0.1, data_term="l1", data_weight=w, ops=ops)
    with pytest.raises(ValueError):
        pytv_b200.CPSolver(x0, 0.1, variant="readme", data_term="l1", ops=ops)
    with pytest.raises(ValueError):
        pytv_b200.CPSolver(x0, 0.1, data_weight=np.ones_like(x0), variant="readme", ops=ops)
    with pytest.raises(ValueError):
        pytv_b200.CPSolver(x0.astype(np.float32), 0.1, data_term="l1", dual_dtype=torch.float16, ops=ops)
    s = pytv_b200.CPSolver(x0, 0.1, data_weight=np.full((1, 1, 4, 8), 2.0), ops=ops)     # broadcast like time_weight
    assert tuple(s._dw.shape) == x0.shape and s._dw.dtype == torch.float64


def test_weight_that_rounds_to_zero_counts_as_missing():
    """A positive float64 weight below float32's range is stored as 0: the dual energy is then unbounded and is refused."""
    import pytv_b200
    x0 = np.random.RandomState(0).rand(2, 1, 4, 8).astype(np.float32)
    w = np.ones(x0.shape)
    w[1, 0, 2, 3] = 1e-50
    s = pytv_b200.CPSolver(x0, 0.1, data_term="l2", data_weight=w, ops=EmulDataOps())
    assert float(s._dw[1, 0, 2, 3]) == 0.0 and s._w_min == 0.0
    with pytest.raises(ValueError):
        s.gap()


def test_cabi_rejects_unknown_data_term():
    lib = _lib.lib()
    pb = _lib.make_problem("hybrid", _lib.F32, (2, 1, 8, 8))
    rc = lib.pytvb_cp_primal_data(ctypes.byref(pb), 2, None, None, None, None, None, 0.1, 1.0, None, None, None, None, None, None, None)
    assert rc == -1
    assert b"data_term" in lib.pytvb_last_error()

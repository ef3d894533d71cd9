"""Host emulation of the adjoint-split Chambolle-Pock pass pair (csrc/adj_core.cuh, run tile by tile by tests/emul/emul_adj.cu)
against the emulated two-pass iteration (strip_quad_cp_dual + strip_quad_cp_primal): x, xbar, y and the mirror stores must be
equal bit for bit over several iterations, the L21 and fidelity sums equal up to the order of their double additions.  Covers
every scheme in both precisions, mask_static and a time-weight map, tile edges (rows not a multiple of the 32-row tile, several
column blocks and a partial last one, the scalar path), M = 1 .. 8, slabs with halo planes, mirror stores and the data terms."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import emul_helper as em
from pytv_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL_SRC = os.path.join(ROOT, "tests", "emul", "emul_adj.cu")
EMUL_SO = os.path.join(ROOT, "tests", "emul", "libpytvb_emul_adj.so")
SCHEMES = ["upwind", "downwind", "central", "hybrid"]
L2, L1 = 0, 1

_handle = None


def _emul():
    """The host emulation library, built when a source is newer than it; loaded once per process."""
    global _handle
    if _handle is not None:
        return _handle
    deps = [EMUL_SRC] + [os.path.join(ROOT, "pytv-4d_b200", "csrc", f) for f in ("core.cuh", "strip_core.cuh", "adj_core.cuh", "kernels.cuh",
                                                                               "host_common.cuh")]
    deps.append(os.path.join(ROOT, "include", "pytv_b200.h"))
    if not (os.path.exists(EMUL_SO) and all(os.path.getmtime(EMUL_SO) >= os.path.getmtime(d) for d in deps)):
        subprocess.run(["nvcc", "-O1", "-std=c++17", "-Xcompiler", "-fPIC", "-shared", "-gencode", "arch=compute_100a,code=sm_100a", EMUL_SRC, "-o",
                        EMUL_SO], check=True, cwd=os.path.dirname(EMUL_SRC))
    h = ctypes.CDLL(EMUL_SO)
    VP = ctypes.c_void_p
    h.pytvb_emulate_adj.restype = ctypes.c_int
    h.pytvb_emulate_adj.argtypes = ([ctypes.POINTER(_lib.Problem), ctypes.c_int, ctypes.c_int] + [VP] * 10 + [ctypes.POINTER(VP)] +
                                    [ctypes.c_double] * 4 + [ctypes.c_int, ctypes.POINTER(ctypes.c_double)])
    h.pytvb_emulate_adj_error.restype = ctypes.c_char_p
    _handle = h
    return h


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _run(split, scheme, dtype, shape, iters=3, term=L2, weight=False, mask=False, tw=False, halo=False, mirrors=False, scalar=False, rt=0.25):
    Nz, M, Ni, Nj = shape
    rs = np.random.RandomState(7)
    rnd = lambda *s: rs.rand(*s).astype(dtype)
    x0 = rnd(*shape)
    x, xbar = x0.copy(), x0.copy()
    z_on, t_on = True, M > 1 and rt > 0
    Nd = (4 + 2 * z_on + 2 * t_on) if scheme == "hybrid" else (2 + z_on + t_on)
    y = np.zeros((Nz, Nd) + shape[1:], dtype=dtype)
    q = np.full(shape, np.nan, dtype=dtype)
    w = (rnd(*shape) * 2).astype(dtype) if weight else None
    if w is not None:
        w[..., 0, :] = 0
    ms = (np.arange(Ni * Nj).reshape(Ni, Nj) % 3 == 0) if mask else None
    twm = rnd(*shape) + 0.5 if tw else None
    pb, keep = em._problem(scheme, np.dtype(dtype), shape, 0.7, rt, ms, 2.0 if mask else 0.0, 1 if halo else 0, Nz + 2 if halo else Nz, twm)
    ilo = ihi = flo = fhi = None
    if halo:
        ilo, ihi, flo, fhi = rnd(M, Ni, Nj), rnd(M, Ni, Nj), rnd(M, Ni, Nj) * 0.05, rnd(M, Ni, Nj) * 0.05
    mir = [np.zeros((M, Ni, Nj), dtype=dtype) for _ in range(4)] if mirrors else [None] * 4
    mp = (ctypes.c_void_p * 4)(*[m.ctypes.data if m is not None else None for m in mir])
    h = _emul()
    sums = []
    for _ in range(iters):
        s = (ctypes.c_double * 2)()
        rc = h.pytvb_emulate_adj(ctypes.byref(pb), split, term, _p(w), _p(xbar), _p(y), _p(q), _p(x), _p(x0), _p(ilo), _p(ihi), _p(flo), _p(fhi), mp, 0.1,
                                 0.5, 0.07, 0.9, int(scalar), s)
        assert rc == 0, h.pytvb_emulate_adj_error()
        sums.append((s[0], s[1]))
    return x, xbar, y, [m for m in mir if m is not None], np.array(sums)


def _same(shape, scheme="hybrid", dtype=np.float32, **kw):
    a = _run(0, scheme, dtype, shape, **kw)
    b = _run(1, scheme, dtype, shape, **kw)
    for u, v in zip(a[:3], b[:3]):
        np.testing.assert_array_equal(u, v)
    for u, v in zip(a[3], b[3]):
        np.testing.assert_array_equal(u, v)
    assert np.isfinite(b[0]).all() and np.abs(b[2]).max() > 0
    np.testing.assert_allclose(a[4], b[4], rtol=1e-12, atol=0)


SHAPES = {"M4": (2, 4, 70, 264), "M3": (2, 3, 33, 264), "M8": (2, 8, 40, 136), "M6": (2, 6, 40, 264), "M1": (2, 1, 40, 1030),
          "M2_odd": (2, 2, 31, 77)}


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("scheme", SCHEMES)
@pytest.mark.parametrize("shape", list(SHAPES.values()), ids=list(SHAPES))
def test_split_equals_two_pass(shape, scheme, dtype):
    _same(shape, scheme, dtype)


@pytest.mark.parametrize("scheme", SCHEMES)
@pytest.mark.parametrize("opts", [dict(mask=True), dict(tw=True), dict(mask=True, tw=True), dict(halo=True), dict(halo=True, mirrors=True, tw=True),
                                  dict(scalar=True, tw=True)],
                         ids=["mask_static", "time_weight", "both", "halo", "halo_mirrors_time_weight", "scalar_time_weight"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
def test_split_time_options_halos_and_mirrors(scheme, opts, dtype):
    _same((3, 4, 67, 264), scheme, dtype, **opts)


@pytest.mark.parametrize("scheme", ["central", "hybrid", "downwind"])
@pytest.mark.parametrize("term,weight", [(L2, True), (L1, False), (L1, True)], ids=["l2_weighted", "l1", "l1_weighted"])
def test_split_data_terms(scheme, term, weight):
    _same((2, 4, 67, 264), scheme, np.float32, term=term, weight=weight, tw=True)
    _same((2, 3, 35, 136), scheme, np.float64, term=term, weight=weight, halo=True)


def test_split_short_axes():
    for shape in ((2, 2, 1, 64), (2, 2, 2, 8), (2, 5, 64, 520)):
        for scheme in SCHEMES:
            _same(shape, scheme, np.float32)

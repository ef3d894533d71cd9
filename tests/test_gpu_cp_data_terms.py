"""The L1 and weighted-L2 data terms of the Chambolle-Pock solver on the GPU (pytvb_cp_primal_data) against the numpy
reference, the unchanged ROF path, the duality gap and the stopping rules, known answers, graph capture and two GPUs."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import data_term_oracle as dto
import pytv_b200 as pytv
from oracle import tv_oracle as orc
from pytv_b200 import _lib

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCHEMES = orc.SCHEMES
FORMS = [("l1", False), ("l1", True), ("l2", True)]
FORM_IDS = ["l1", "l1_w", "l2_w"]


def _weights(rs, shape):
    w = 2.0 * rs.rand(*shape)
    w[:, :, ::3] = 0
    return w


@pytest.mark.parametrize("shape", [(3, 2, 5, 8), (1, 1, 7, 12), (2, 2, 1, 4), (2, 3, 6, 5), (4, 2, 33, 260)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("scheme", SCHEMES)
def test_cp_data_terms_match_oracle(scheme, dtype, shape):
    """One iteration from a random state and 10 iterations from the start, time weights and mask_static on."""
    rs = np.random.RandomState(41)
    Nz, M, Ni, Nj = shape
    x0 = rs.rand(*shape).astype(dtype)
    kw = dict(reg_z_over_reg=0.6, reg_time=0.4, mask_static=rs.rand(1, 1, Ni, Nj) > 0.5, factor_reg_static=3.0, time_weight=0.5 + rs.rand(*shape))
    Nd = orc.num_components(scheme, Nz, M, 0.6, 0.4)
    y = (0.2 * rs.randn(Nz, Nd, M, Ni, Nj)).astype(dtype)
    x = (x0 + 0.1 * rs.randn(*shape)).astype(dtype)
    xbar = (x + 0.01 * rs.randn(*shape)).astype(dtype)
    w = _weights(rs, shape).astype(dtype)
    f64 = dtype == np.float64
    atol1, atol10, rel = (1e-12, 1e-12, 1e-12) if f64 else (1e-5, 2e-5, 2e-5)
    for term, use_w in FORMS:
        ww = w if use_w else None
        s = pytv.CPSolver(x0, lam=0.1, scheme=scheme, sigma=0.5, tau=0.07, theta=0.9, data_term=term, data_weight=ww, **kw)
        s.x.copy_(torch.as_tensor(x))
        s.y.copy_(torch.as_tensor(y))
        s.aux.copy_(torch.as_tensor(xbar))
        xr, xbr, yr, er = dto.cp_data_step(x.copy(), xbar.copy(), x0, y.copy(), term, ww, scheme, lam=0.1, sigma=0.5, tau=0.07, theta=0.9, **kw)
        s.step()
        np.testing.assert_allclose(s.y.cpu().numpy(), yr, atol=atol1)
        np.testing.assert_allclose(s.x.cpu().numpy(), xr, atol=atol1)
        np.testing.assert_allclose(s.aux.cpu().numpy(), xbr, atol=atol1)
        assert s.energy() == pytest.approx(er, rel=rel)
        s = pytv.CPSolver(x0, lam=0.1, scheme=scheme, sigma=0.5, tau=1.0 / 17.0, data_term=term, data_weight=ww, **kw)
        s.step(10)
        xr, xbr, yr, er = dto.run(x0, 10, term, ww, scheme, lam=0.1, sigma=0.5, tau=1.0 / 17.0, **kw)
        np.testing.assert_allclose(s.x.cpu().numpy(), xr, atol=atol10)
        np.testing.assert_allclose(s.aux.cpu().numpy(), xbr, atol=atol10)
        np.testing.assert_allclose(s.y.cpu().numpy(), yr, atol=atol10)
        assert s.energy() == pytest.approx(er, rel=rel)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("scheme", SCHEMES)
def test_cp_data_slab_with_halos_equals_whole_volume(scheme, dtype):
    """Pass B on planes [1, 4) of a 5-plane volume, field halos taken from the neighbouring planes: bitwise the whole-volume pass."""
    g = torch.Generator().manual_seed(5)
    Nz, M, Ni, Nj = 5, 3, 20, 64
    shape = (Nz, M, Ni, Nj)
    dt_id = _lib.F32 if dtype == torch.float32 else _lib.F64
    Nd = orc.num_components(scheme, Nz, M, 0.5, 0.3)
    x0 = torch.rand(shape, generator=g, dtype=torch.float64).to(dtype).cuda()
    y = (0.2 * torch.randn((Nz, Nd) + shape[1:], generator=g, dtype=torch.float64)).to(dtype).cuda()
    w = (2 * torch.rand(shape, generator=g, dtype=torch.float64)).to(dtype).cuda()
    ts = (0.5 + torch.rand(shape, generator=g, dtype=torch.float64)).sqrt().to(dtype).cuda()
    zf, zb = (4, 5) if scheme == "hybrid" else (2, 2)
    ops = pytv.cp.CudaOps()
    for term, use_w in FORMS:
        ww = w if use_w else None
        xa, xba = x0 + 0.1, torch.zeros_like(x0)
        pb = _lib.make_problem(scheme, dt_id, shape, 0.5, 0.3, time_scale_ptr=ts.data_ptr())
        ws = ops.workspace(pb, x0.device)
        da = torch.zeros(1, dtype=torch.float64, device="cuda")
        ops.cp_primal_data(pb, term, ww, y, xa, xba, x0, 0.07, 1.0, da, None, None, None, None, ws)
        xs, xbs = (x0 + 0.1)[1:4].contiguous(), torch.zeros_like(x0[1:4])
        pbs = _lib.make_problem(scheme, dt_id, (3, M, Ni, Nj), 0.5, 0.3, z_offset=1, Nz_global=Nz, time_scale_ptr=ts[1].data_ptr())
        ops.cp_primal_data(pbs, term, None if ww is None else ww[1:4], y[1:4], xs, xbs, x0[1:4], 0.07, 1.0, None, y[0, zf].contiguous(),
                           y[4, zb].contiguous(), None, None, ws)
        torch.cuda.synchronize()
        assert torch.equal(xs, xa[1:4]) and torch.equal(xbs, xba[1:4])
        r = (xa - x0).double()
        r = r * r if term == "l2" else r.abs()
        assert float(da) == pytest.approx(float((r if ww is None else r * ww.double()).sum()), rel=1e-5)


@pytest.mark.parametrize("scheme", SCHEMES)
def test_unweighted_l2_is_the_rof_solver(scheme):
    g = torch.Generator().manual_seed(7)
    x0 = torch.rand(4, 3, 24, 40, generator=g, dtype=torch.float64).cuda()
    kw = dict(lam=0.1, scheme=scheme, reg_time=0.25)
    a = pytv.CPSolver(x0, **kw).step(10)
    b = pytv.CPSolver(x0, data_term="l2", **kw).step(10)
    assert torch.equal(a.x, b.x) and torch.equal(a.aux, b.aux) and torch.equal(a.y, b.y) and a.energy() == b.energy()
    c = pytv.CPSolver(x0, data_weight=torch.ones_like(x0), **kw).step(10)
    torch.testing.assert_close(c.x, a.x, atol=1e-14, rtol=0)
    torch.testing.assert_close(c.aux, a.aux, atol=1e-14, rtol=0)
    assert c.energy() == pytest.approx(a.energy(), rel=1e-14)
    assert c.gap()[1] == pytest.approx(a.gap()[1], rel=1e-12)


@pytest.mark.parametrize("term,use_w,lam", [("l2", True, 0.1), ("l1", False, 0.6), ("l1", True, 0.6)], ids=["l2_w", "l1", "l1_w"])
def test_gap_matches_oracle_and_solve_converges(term, use_w, lam):
    rs = np.random.RandomState(1)
    x0 = rs.rand(2, 2, 16, 16)
    w = 0.5 + rs.rand(*x0.shape) if use_w else None
    kw = dict(reg_time=0.25)
    s = pytv.CPSolver(x0, lam=lam, scheme="hybrid", data_term=term, data_weight=w, **kw)
    s.step(50)
    p, d, gap = s.gap()
    x = s.result()
    assert p == pytest.approx(dto.primal_energy(x, x0, term, w, "hybrid", lam, **kw), rel=1e-12)
    assert d == pytest.approx(dto.dual_energy(s.y.cpu().numpy(), x0, term, w, "hybrid", **kw), rel=1e-12)
    assert gap >= 0
    info = pytv.CPSolver(x0, lam=lam, scheme="hybrid", data_term=term, data_weight=w, **kw).solve(max_iter=4000, tol=5e-4)
    assert info["converged"] and info["criterion"] == "gap" and info["gap"] >= 0


def test_zero_weight_inpainting_and_energy_stopping():
    """w = 0 under a hole: no duality gap (gap() raises), solve() stops on the energy change, and a constant image with garbage
    under the hole comes back constant."""
    c = 0.7
    x0 = np.full((1, 2, 12, 12), c)
    w = np.ones_like(x0)
    x0[0, :, 4:8, 3:9] = np.random.RandomState(5).rand(2, 4, 6) * 5
    w[0, :, 4:8, 3:9] = 0
    for term in ("l2", "l1"):
        s = pytv.CPSolver(x0, lam=0.1, scheme="hybrid", tau=1.0 / 17.0, reg_time=0.5, data_term=term, data_weight=w)
        with pytest.raises(ValueError):
            s.gap()
        s.step(1500)
        np.testing.assert_allclose(s.result(), c, atol=1e-5)
    rs = np.random.RandomState(2)
    x0 = rs.rand(2, 2, 16, 16)
    w = rs.rand(*x0.shape)
    w[:, :, 5:9, 5:9] = 0
    for term in ("l2", "l1"):
        info = pytv.CPSolver(x0, lam=0.3, scheme="hybrid", data_term=term, data_weight=w).solve(max_iter=5000, tol=1e-7)
        assert info["converged"] and info["criterion"] == "energy" and info["relative_change"] <= 1e-7


@pytest.mark.parametrize("h", [1.0, 7.0])
@pytest.mark.parametrize("lam,kept", [(0.2, True), (0.45, False)])
def test_tv_l1_impulse_known_answer(h, lam, kept):
    """Upwind 2-D TV-L1 keeps an interior impulse below lam = 1 / (2 + sqrt 2) and removes it above, whatever its height."""
    x0 = np.zeros((1, 1, 9, 9))
    x0[0, 0, 4, 4] = h
    s = pytv.CPSolver(x0, lam=lam, scheme="upwind", tau=1.0 / 9.0, data_term="l1").step(3000)
    np.testing.assert_allclose(s.result(), x0 if kept else 0.0, atol=1e-3 * h)


def test_graph_replay_equals_eager():
    rs = np.random.RandomState(9)
    x0 = rs.rand(3, 2, 32, 48).astype(np.float32)
    w = rs.rand(*x0.shape).astype(np.float32)
    for term in ("l1", "l2"):
        a = pytv.CPSolver(x0, lam=0.2, reg_time=0.25, data_term=term, data_weight=w)
        b = pytv.CPSolver(x0, lam=0.2, reg_time=0.25, data_term=term, data_weight=w).capture_graph(4)
        a.step(8)
        b.step(8)
        assert torch.equal(a.x, b.x) and torch.equal(a.aux, b.aux) and torch.equal(a.y, b.y)
        assert a.energy() == b.energy()


# ------------------------------------------------------------------ two GPUs
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _problem():
    g = torch.Generator().manual_seed(3)
    x0 = torch.rand(12, 3, 64, 64, generator=g)
    w = torch.rand(12, 3, 64, 64, generator=g) * 2 + 0.1
    return x0, w


def _worker(rank, world, port, comm, term, out_dir):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    import pytv_b200
    os.environ["PYTVB_OVERLAP"] = "0"
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        x0, w = _problem()
        off, cnt = pytv_b200.partition_z(12, world)[rank]
        s = pytv_b200.CPSolver(x0[off:off + cnt].cuda(), lam=0.1, reg_time=0.25, distributed=True, comm=comm, data_term=term,
                               data_weight=w[off:off + cnt].cuda())
        assert (s._peer is not None) == (comm == "p2p")
        energies = []
        for _ in range(5):
            s.step()
            energies.append(s.energy())
        energies.extend(s.gap())
        s.step(2)
        np.save(os.path.join(out_dir, "x_%d.npy" % rank), s.result())
        if rank == 0:
            np.save(os.path.join(out_dir, "e.npy"), np.array(energies))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("term", ["l1", "l2"])
@pytest.mark.parametrize("comm", ["nccl", "p2p"])
def test_two_gpu_sharded_data_terms_equal_single_gpu(tmp_path, comm, term):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    mp.spawn(_worker, args=(2, _free_port(), comm, term, str(tmp_path)), nprocs=2, join=True)
    x = np.concatenate([np.load(tmp_path / ("x_%d.npy" % r)) for r in range(2)], axis=0)
    x0, w = _problem()
    s = pytv.CPSolver(x0.cuda(), lam=0.1, reg_time=0.25, data_term=term, data_weight=w.cuda())
    energies = []
    for _ in range(5):
        s.step()
        energies.append(s.energy())
    energies.extend(s.gap())
    s.step(2)
    np.testing.assert_array_equal(x, s.result())
    e = np.load(tmp_path / "e.npy")
    np.testing.assert_allclose(e[:5], energies[:5], rtol=1e-12)
    np.testing.assert_allclose(e[5:7], energies[5:7], rtol=1e-9)

"""A/B of one Chambolle-Pock iteration on the C4 slab: the two-pass form (pytvb_cp_dual + pytvb_cp_primal_rof) against the
form that finishes the in-plane and time terms of the adjoint in the dual pass (pytvb_cp_dual_adj + pytvb_cp_primal_adj).

    python scripts/bench_cp_adj.py [--steps 20] [--rounds 5] [--warmup 3] [--out FILE]

Slab (128, 4, 1024, 1024) float32, hybrid scheme, reg_time = 2^-5 (Nd = 8), as bench.py's C4.  Both forms run in one process
from the same state and alternate round by round; each round times `steps` iterations of one form with CUDA events around
every pass.  Algorithmic bytes per voxel: two-pass 68 + 48; split 72 + 28 with the tile edges of csrc/adj_core.cuh counted
apart: on an edge row the dual pass stores no q (-4) and the primal pass reads the Nd components instead of q (+20); on an
edge column it also reads J_F and J_B (+8; the three single neighbour values it reads there are not counted).  The working
set (~60 GB) is far larger than the L2.  After the rounds both forms have run the same iterations and x, xbar and y must be equal bit for bit.  Prints one JSON
object.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ADJ_R = 32   # rows of a dual-pass tile (csrc/adj_core.cuh)


def _power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        return out[0] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def edge_fractions(M, Ni, Nj, vec=4):
    """Shares of voxels on an edge row, and on an edge column but not an edge row (adj_core.cuh: adj_edge_row / adj_edge_col)."""
    twq = 256 if M == 1 else (128 if M == 2 else (64 if M <= 4 else 32))
    rows = [(i % ADJ_R == 0 and i > 0) or (i % ADJ_R == ADJ_R - 1 and i < Ni - 1) for i in range(Ni)]
    cols = []
    for qj in range((Nj + vec - 1) // vec):
        tq, j0 = qj % twq, qj * vec
        cols.append((tq == 0 and j0 > 0) or (tq == twq - 1 and j0 + vec < Nj))
    n_r, n_c = sum(rows), sum(cols)
    nq = len(cols)
    return n_r / Ni, n_c * (Ni - n_r) / (Ni * nq)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="iterations per timed round")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--slab", type=int, nargs=4, default=[128, 4, 1024, 1024])
    ap.add_argument("--out", default=None, help="also write the JSON here")
    args = ap.parse_args()

    import torch
    from pytv_b200 import _dev, _lib

    if not torch.cuda.is_available():
        raise SystemExit("bench_cp_adj.py needs a CUDA device")
    shape = tuple(args.slab)
    Nz, M, Ni, Nj = shape
    V = Nz * M * Ni * Nj
    lib = _lib.lib()
    torch.manual_seed(0)
    x0 = torch.rand(shape, device="cuda") + 0.05 * torch.randn(shape, device="cuda")
    pb = _lib.make_problem("hybrid", _lib.F32, shape, 1.0, 2.0 ** -5)
    Nd = lib.pytvb_num_components(ctypes.byref(pb))
    lam, sigma, tau, theta = 0.1, 0.5, 1.0 / (4.0 * 2 + 4.0 + 1.0), 1.0
    st = _dev.stream_ptr()

    def state():
        return dict(x=x0.clone(), xbar=x0.clone(), y=torch.zeros((Nz, Nd) + shape[1:], device="cuda"), ws=_dev.reduce_workspace(pb, x0.device),
                    scal=torch.zeros(2, dtype=torch.float64, device="cuda"))

    old, new = state(), state()
    q = torch.empty_like(x0)
    P = _dev.ptr

    def pass_a(s, split):
        if split:
            _lib.check(lib.pytvb_cp_dual_adj(ctypes.byref(pb), P(s["xbar"]), P(s["y"]), P(q), lam, sigma, P(s["scal"][0:1]), None, None, P(s["ws"]), st))
        else:
            _lib.check(lib.pytvb_cp_dual(ctypes.byref(pb), P(s["xbar"]), P(s["y"]), lam, sigma, P(s["scal"][0:1]), None, None, P(s["ws"]), st))

    def pass_b(s, split):
        if split:
            _lib.check(lib.pytvb_cp_primal_adj(ctypes.byref(pb), 0, None, P(s["y"]), P(q), P(s["x"]), P(s["xbar"]), P(x0), tau, theta, P(s["scal"][1:2]),
                                               None, None, P(s["ws"]), st))
        else:
            _lib.check(lib.pytvb_cp_primal_rof(ctypes.byref(pb), P(s["y"]), P(s["x"]), P(s["xbar"]), P(x0), tau, theta, P(s["scal"][1:2]), None, None,
                                               P(s["ws"]), st))

    def run(s, split, n, timed):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * n + 1)] if timed else None
        if timed:
            ev[0].record()
        for k in range(n):
            pass_a(s, split)
            if timed:
                ev[2 * k + 1].record()
            pass_b(s, split)
            if timed:
                ev[2 * k + 2].record()
        torch.cuda.synchronize()
        if not timed:
            return None
        ta = sum(ev[2 * k].elapsed_time(ev[2 * k + 1]) for k in range(n)) / n
        tb = sum(ev[2 * k + 1].elapsed_time(ev[2 * k + 2]) for k in range(n)) / n
        return ta, tb

    run(old, False, args.warmup, False)
    run(new, True, args.warmup, False)
    f_row, f_col = edge_fractions(M, Ni, Nj)
    bytes_old = (4.0 * (2 * Nd + 1), 4.0 * (Nd + 4))
    bytes_new = (4.0 * (2 * Nd + 2) - 4.0 * f_row, 4.0 * 7 + 4.0 * (Nd - 3) * f_row + 8.0 * f_col)
    rounds = []
    for r in range(args.rounds):
        (oa, ob), (na, nb) = run(old, False, args.steps, True), run(new, True, args.steps, True)
        rounds.append(dict(round=r, two_pass=dict(pass_a_ms=oa, pass_b_ms=ob, iter_ms=oa + ob), split=dict(pass_a_ms=na, pass_b_ms=nb, iter_ms=na + nb),
                           speedup=(oa + ob) / (na + nb) - 1.0))
    equal = all(torch.equal(old[k], new[k]) for k in ("x", "xbar", "y"))

    def gbs(b, ms):
        return b * V / (ms * 1e-3) / 1e9

    it_old = [r["two_pass"]["iter_ms"] for r in rounds]
    it_new = [r["split"]["iter_ms"] for r in rounds]
    for r in rounds:
        r["two_pass"]["gbs"] = [gbs(bytes_old[0], r["two_pass"]["pass_a_ms"]), gbs(bytes_old[1], r["two_pass"]["pass_b_ms"])]
        r["split"]["gbs"] = [gbs(bytes_new[0], r["split"]["pass_a_ms"]), gbs(bytes_new[1], r["split"]["pass_b_ms"])]
    res = dict(device=torch.cuda.get_device_name(0), power_limit_and_max_sm_clock=_power_limit(), slab=list(shape), Nd=Nd, steps=args.steps,
               edge_row_fraction=f_row, edge_column_fraction=f_col, bytes_per_voxel=dict(two_pass=list(bytes_old), split=list(bytes_new)), rounds=rounds,
               two_pass_iter_ms=dict(min=min(it_old), max=max(it_old)), split_iter_ms=dict(min=min(it_new), max=max(it_new)),
               min_speedup=min(r["speedup"] for r in rounds), speedup_exceeds_spread=max(it_new) < min(it_old) - (max(it_old) - min(it_old)),
               bitwise_equal=equal)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if not equal:
        raise SystemExit("the two forms differ")


if __name__ == "__main__":
    main()

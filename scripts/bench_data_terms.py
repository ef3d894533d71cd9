"""Time one Chambolle-Pock iteration with each data term on the C4 slab: ROF (0.5|x - x0|^2), TV-L1, TV-L1 with a weight map
and weighted L2, alternating the four forms in one process so that they share the card's state.

    python scripts/bench_data_terms.py [--steps 20] [--rounds 5] [--out FILE]

Slab (128, 4, 1024, 1024) float32, hybrid scheme, reg_time = 2^-5 (Nd = 8), as bench.py's C4.  Per form: the median over
rounds of the mean time per iteration (CUDA events around `steps` iterations), the rate from the algorithmic bytes per
voxel (116 for ROF and L1: pass A reads xbar and y and writes y, pass B reads y, x, x0 and writes x, xbar; 120 with a weight
map, one more read), the ratio to ROF and whether it is within 1.03 x ROF x bytes / 116.  The working set (~100 GB) is far
larger than the L2, so no cache flush is needed between iterations.  Prints one JSON object.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FORMS = [("rof", "l2", False, 116), ("l1", "l1", False, 116), ("l1_weighted", "l1", True, 120), ("l2_weighted", "l2", True, 120)]


def _power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        return out[0] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="iterations per timed window")
    ap.add_argument("--rounds", type=int, default=5, help="alternating rounds over the four forms")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--slab", type=int, nargs=4, default=[128, 4, 1024, 1024])
    ap.add_argument("--out", default=None, help="also write the JSON here")
    args = ap.parse_args()

    import numpy as np
    import torch
    import pytv_b200 as pytv

    if not torch.cuda.is_available():
        raise SystemExit("bench_data_terms.py needs a CUDA device")
    torch.cuda.set_device(0)
    shape = tuple(args.slab)
    g = torch.Generator(device="cuda").manual_seed(1000)
    x0 = torch.rand(shape, generator=g, device="cuda") + 0.05 * torch.randn(shape, generator=g, device="cuda")
    w = 0.5 + torch.rand(shape, generator=g, device="cuda")
    solvers = {}
    for name, term, weighted, _ in FORMS:
        solvers[name] = pytv.CPSolver(x0, lam=0.1, scheme="hybrid", reg_time=2.0 ** -5, data_term=term, data_weight=w if weighted else None)
        assert solvers[name].Nd == 8
    del x0
    for s in solvers.values():
        s.step(args.warmup)
    torch.cuda.synchronize()
    times = {name: [] for name, *_ in FORMS}
    for _ in range(args.rounds):
        for name, *_ in FORMS:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            solvers[name].step(args.steps)
            b.record()
            b.synchronize()
            times[name].append(a.elapsed_time(b) / args.steps)
    voxels = float(np.prod(shape))
    rof_ms = float(np.median(times["rof"]))
    res = dict(device=torch.cuda.get_device_name(0), power_limit_and_max_sm_clock=_power_limit(), slab=list(shape), dtype="float32",
               scheme="hybrid", reg_time=2.0 ** -5, Nd=8, steps=args.steps, rounds=args.rounds, forms={})
    for name, term, weighted, nbytes in FORMS:
        ms = float(np.median(times[name]))
        bound = 1.03 * rof_ms * nbytes / 116.0
        res["forms"][name] = dict(data_term=term, weight_map=weighted, bytes_per_voxel=nbytes, ms_per_iter=round(ms, 4),
                                  ms_per_iter_all_rounds=[round(t, 4) for t in times[name]],
                                  algorithmic_GB_per_s=round(voxels * nbytes / (ms * 1e-3) / 1e9, 1), ratio_to_rof=round(ms / rof_ms, 4),
                                  within_1p03_of_rof_x_bytes=bool(ms <= bound))
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()

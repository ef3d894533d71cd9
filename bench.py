#!/usr/bin/env python
"""Benchmark of the TV hot path (BASELINE.json `metric`: Chambolle-Pock iteration voxel-updates/s, HBM GB/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C4|C3|C5]      our arm (sm_100a kernels)
    python bench.py --impl reference [--gpus N] [--steps K] ...                    the reference's CPU path on the host cores

Workloads (BASELINE.json `configs`):
  C4 (default, the configuration the metric is quoted on): per-GPU z-slab (128, 4, 1024, 1024) float32 of a
      (128*N, 4, 1024, 1024) dynamic-CT volume, hybrid scheme, reg_time = 2^-5 (Nd = 8), ROF-form Chambolle-Pock
      iteration = dual pass + primal pass, energy tracked every iteration.  Weak scaling: Nz grows with N, one-plane halos
      per pass (pushed into the neighbours' peer memory by the kernels, or NCCL send/recv), two doubles all-reduced per
      iteration.
  C3: 512^3 float32 (M = 1), hybrid, Nd = 6, the same iteration (per-GPU slab (512, 1, 512, 512)).
  C5: discretisation sweep - fused tv_<scheme> (value + sub-gradient, with `mask`), D_<scheme> and D_T_<scheme> for the four
      schemes with mask_static on a per-GPU slab (64, 8, 2048, 2048), sharded with pytv.sharded.ShardedTV.  A step = the 12
      calls; `value` = voxels x 12 / time ("voxel-operator-applications/s"); per-operator rooflines under `per_op`.

Order of a run (our arm): (1) PARITY GATE - a reduced slab of the same workload at the benchmark's plane size is computed on
the GPU and by the reference's CPU code (baseline/_ref when it travels with the repo, else the oracle port; the same CPU run
is the timed `cpu_baseline`), and the line carries no `value` unless they agree (energy / TV 1e-5 relative, x 1e-5
absolute: the north-star tolerances); (2) N > 1: MULTI-GPU CHECK - a small volume computed by every rank alone and by the
group sharded, with the halo transport the timed run uses, must agree bit for bit; (3) device-resident timing (CUDA events,
max over ranks); (4) host-link peak (pinned H2D || D2H, all ranks at once) and the end-to-end timing through the
host-buffer API.

A "step" is one iteration over the whole volume.  `value` = voxels * K / t with the state resident in HBM.  `e2e` = the same
iteration driven through the public host-buffer call `CPSolver.step_host_async`: every step uploads the data term x0 from
pinned host memory, runs the iteration, downloads the current image x and the energy (three steps in flight).  The state
per GPU (23.6 GB for C4) is far larger than the 126 MB L2, so no L2 flush is needed between iterations.

--dump-outputs DIR writes what the timed path computed in its last timed step as DIR/<name>.npy (one file per rank, suffix
_rank<r>, when N > 1): C4 / C3 the image x (float32) and the energy (float64); C5 per scheme the tv value (float64) and
the sub-gradient G, D x and D_T D x (float32).  The float32 arrays of all ranks share 48 MiB; an array larger than its
share is stored as the elements at fixed seeded flat positions.  The inputs are seeded, so two builds run with the same
arguments can be compared file by file.  C5 gathers those elements inside its last timed step (the fields of the four
schemes do not fit in memory together), which adds 12 small gather kernels to the time of a run with --dump-outputs.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the source tree (it may be read-only)

UNIT = "voxel-updates/s"
LAM = 0.1
DUMP_BYTES = 48 << 20               # --dump-outputs: bytes of float32 output samples of all ranks (the files stay below 64 MB)

WORKLOADS = {
    # name: slab per GPU, scheme weights, gate sample, CPU-arm sample per process
    "C4": dict(metric="cp_iter_voxel_updates_per_s", slab=(128, 4, 1024, 1024), kw=dict(reg_time=2.0 ** -5), Nd=8,
               gate=(4, 4, 1024, 1024), cpu_sample=(2, 4, 1024, 1024),
               text="C4 dynamic-CT slab (Nz=128*N_gpus, M=4, N=1024) f32, hybrid scheme, reg_time=2^-5 (Nd=8), CP-ROF iteration"),
    "C3": dict(metric="cp_iter_voxel_updates_per_s", slab=(512, 1, 512, 512), kw=dict(), Nd=6,
               gate=(16, 1, 512, 512), cpu_sample=(8, 1, 512, 512),
               text="C3 volume (Nz=512*N_gpus, M=1, N=512) f32, hybrid scheme (Nd=6), CP-ROF iteration"),
    "C5": dict(metric="tv_scheme_sweep_voxel_ops_per_s", slab=(64, 8, 2048, 2048), kw=dict(reg_time=2.0 ** -5, factor_reg_static=4.0), Nd=8,
               gate=(3, 8, 512, 512), cpu_sample=(2, 8, 256, 256),
               text="C5 discretisation sweep (Nz=64*N_gpus, M=8, N=2048) f32: tv/D/D_T x upwind/downwind/central/hybrid, mask disc 0.48N, "
                    "mask_static disc 0.25N x4, reg_time=2^-5"),
}
SCHEMES = ("upwind", "downwind", "central", "hybrid")


def config_dict(wl, n_gpus, extra=None):
    w = WORKLOADS[wl]
    cfg = {"workload": w["text"], "slab_per_gpu": list(w["slab"]), "scheme": "hybrid" if wl != "C5" else "all four", "Nd": w["Nd"],
           "reg_time": w["kw"].get("reg_time", 0.0), "lam": LAM, "variant": "rof", "parallelism": "z-slabs x%d, 1-plane halos" % n_gpus,
           "l2_policy": "working set per GPU >> 126 MB L2, no flush needed"}
    if extra:
        cfg.update(extra)
    return cfg


# --------------------------------------------------------------------------------------------------------
# CPU arms (oracle / reference): test-infrastructure code, used only as the checker of the parity gate and as the
# reported baseline
def _cpu_modules():
    """(tv_operators_CPU-like module, tv_CPU-like module or None, kind): the unmodified reference numpy modules when a copy
    travels with the repo (baseline/_ref, git-ignored), else None -> the oracle port."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(os.path.join(ref_dir, "pytv")) and os.environ.get("PYTVB_BENCH_FORCE_PORT") != "1":
        try:
            import importlib.util
            import warnings
            warnings.filterwarnings("ignore", category=SyntaxWarning)
            mods = []
            for name in ("tv_operators_CPU",):
                spec = importlib.util.spec_from_file_location("_ref_" + name, os.path.join(ref_dir, "pytv", name + ".py"))
                mod = importlib.util.module_from_spec(spec)
                spec.loader.exec_module(mod)
                mods.append(mod)
            return mods[0], "reference"
        except Exception:
            pass
    return None, "port"


def _cpu_ops(scheme="hybrid"):
    """(D, D_T, l21, kind) for one scheme."""
    mod, kind = _cpu_modules()
    if mod is not None:
        return getattr(mod, "D_" + scheme), getattr(mod, "D_T_" + scheme), mod.compute_L21_norm, kind
    from oracle import tv_oracle as orc
    return (lambda x, **kw: orc.D(x, scheme, **kw)), (lambda p, **kw: orc.D_T(p, scheme, **kw)), orc.l21, "port"


def _cpu_cp_iteration(D, DT, l21, state, x0, lam, sigma, tau, kw):
    """CP-ROF iteration from the CPU operators (the loop of README.md:145-157 in its over-relaxed form)."""
    x, xbar, y = state
    Dxb = D(xbar, **kw).astype(x0.dtype, copy=False)      # the reference upcasts float32 under numpy >= 2 (SURVEY B8)
    pa = y + sigma * Dxb
    y = pa / np.maximum(1.0, np.sqrt(np.sum(pa ** 2, axis=1, keepdims=True)) / lam)
    x_new = (x - tau * DT(y, **kw).astype(x0.dtype, copy=False) + tau * x0) / (1.0 + tau)
    xbar = x_new + (x_new - x)
    # energy in float64 from the float32 state (the checker's summation must not be the error source)
    nrm = np.sqrt(np.sum(np.square(Dxb, dtype=np.float64), axis=1))
    energy = 0.5 * np.sum(np.square(x_new - x0, dtype=np.float64)) + lam * float(np.sum(nrm))
    return (x_new, xbar, y), float(energy)


def tau_for(kw):
    """Default step of CPSolver for the hybrid scheme with z on: 1 / (4 (2 + 1 + reg_time) + 1)."""
    return 1.0 / (4.0 * (3.0 + kw.get("reg_time", 0.0)) + 1.0)


def make_sample(seed, shape, blocks=False):
    rs = np.random.RandomState(seed)
    if blocks:      # C3: piecewise-constant blocks {0, 0.5, 1} of edge 64 + 0.1 randn (SURVEY 8d-3)
        b = rs.randint(0, 3, tuple((s + 63) // 64 for s in shape)).astype(np.float32) * 0.5
        for ax in (0, 2, 3):
            b = np.repeat(b, 64, axis=ax)
        return (b[:shape[0], :, :shape[2], :shape[3]] + 0.1 * rs.randn(*shape)).astype(np.float32)
    return (rs.rand(*shape) + 0.05 * rs.randn(*shape)).astype(np.float32)


def _cpu_worker(args):
    """One process of the CPU arm: `steps` timed iterations on its own sample slab.  Returns (seconds, kind, energies, x)."""
    seed, shape, steps, warmup, kw, keep = args
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    D, DT, l21, kind = _cpu_ops("hybrid")
    x0 = make_sample(seed, shape, blocks=(shape[1] == 1))
    Nd = 4 + 2 * (shape[0] > 1) + 2 * (shape[1] > 1 and kw.get("reg_time", 0) > 0)
    y = np.zeros((shape[0], Nd) + shape[1:], np.float32)
    state = (x0.copy(), x0.copy(), y)
    sigma, tau = np.float32(0.5), np.float32(tau_for(kw))
    for _ in range(warmup):
        state, e = _cpu_cp_iteration(D, DT, l21, state, x0, np.float32(LAM), sigma, tau, kw)
    energies = []
    t0 = time.perf_counter()
    for _ in range(steps):
        state, e = _cpu_cp_iteration(D, DT, l21, state, x0, np.float32(LAM), sigma, tau, kw)
        energies.append(e)
    dt = time.perf_counter() - t0
    return dt, kind, energies, (state[0] if keep else None)


def _cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path on all host cores of the box: one process per core,
    each iterating on its own sample slab (independent z-slabs, which is how the CPU path would be sharded);
    voxel-updates/s is the aggregate."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    wl = args.workload if args.workload != "C5" else "C4"      # the CPU arm times the CP iteration (the metric); C5 has no CP loop
    w = WORKLOADS[wl]
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    procs = max(1, min(cores, 64))
    sample = tuple(w["cpu_sample"])
    # one iteration of this sample takes ~2.5 s on one core
    steps = args.steps
    warmup = min(max(0, args.warmup), 3)
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(procs) as pool:
        res = pool.map(_cpu_worker, [(1000 + p, sample, steps, warmup, w["kw"], False) for p in range(procs)])
    wall = time.perf_counter() - t0
    t_max = max(r[0] for r in res)
    kind = res[0][1]
    vox = int(np.prod(sample)) * procs
    value = vox * steps / t_max
    line = {"impl": "reference", "metric": w["metric"], "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": 1e3 * t_max / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": config_dict(wl, args.gpus, {"note": "CPU arm: bounded sample of the workload at the benchmark's plane size, %d processes x slab %s"
                                                          % (procs, list(sample))}),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": kind, "host_cpu": _cpu_model(), "host_cpu_count": os.cpu_count(),
                             "sample": "%d processes (of %d host cores), each %d CP-ROF iterations on its own %s float32 slab; wall %.1f s"
                                       % (procs, cores, steps, "x".join(map(str, sample)), wall)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi sampling of SM clocks and throttle reasons during the timed region (B200_PROFILING.md)."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(prefix="clocks_", suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        try:
            rows = [r.split(",") for r in open(self.path).read().strip().splitlines() if r.strip()]
            sm = sorted(float(r[1]) for r in rows)
            reasons = set()
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for r in rows:
                for name, v in zip(names, r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(rows[0][2]) if rows else None,
                   "reasons": sorted(reasons), "samples": len(rows), "power_w_max": max(float(r[3]) for r in rows) if rows else None}
            os.unlink(self.path)
        except Exception:
            pass
        return out


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md, 6.65 TB/s)"


def lib_build_id():
    """Identity of the CUDA library the run loaded: pytvb_build_id(), the hash of the sources it was built from (stable across
    rebuilds, unlike the bytes of the binary).  Ties recorded ncu traffic to a build."""
    from pytv_b200 import _lib
    try:
        return _lib.lib().pytvb_build_id().decode()
    except Exception:
        return None


def recorded_traffic():
    """DRAM bytes per launch from the committed `ncu --set full` capture (profiles/traffic.json, written by
    scripts/ncu_traffic.py together with the hash of the library it profiled).  Returned only when that hash equals the
    library this run loaded; otherwise `roofline.traffic` is null rather than a number from another build."""
    try:
        doc = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return {}
    if doc.get("build_id") and doc.get("build_id") == lib_build_id():
        return doc.get("kernels", {})
    return {}


# --------------------------------------------------------------------------------------------------------
# (1) parity gate
def parity_gate_cp(wl, dev, iters=5):
    """A reduced slab of the workload (same plane size, scheme, weights, dtype) through `iters` CP-ROF iterations on the GPU
    and by the CPU checker; returns (gate dict, cpu_baseline dict)."""
    import torch
    import pytv_b200 as pytv
    w = WORKLOADS[wl]
    shape, kw = tuple(w["gate"]), w["kw"]
    x0 = make_sample(4242, shape, blocks=(shape[1] == 1))
    s = pytv.CPSolver(torch.from_numpy(x0).to(dev), lam=LAM, scheme="hybrid", variant="rof", **kw)
    assert abs(s.tau - tau_for(kw)) < 1e-12
    e_gpu = []
    for _ in range(iters):
        s.step()
        e_gpu.append(s.energy())
    x_gpu = s.x.cpu().numpy()
    tv_gpu, _ = pytv.tv_GPU.tv_hybrid(s.x, return_pytorch_tensor=True, **kw)
    del s
    dt, kind, e_cpu, x_cpu = _cpu_worker((4242, shape, iters, 0, kw, True))
    D, _, l21, _ = _cpu_ops("hybrid")
    tv_cpu = float(np.sum(np.sqrt(np.sum(np.square(D(x_cpu, **kw), dtype=np.float64), axis=1))))
    e_rel = max(abs(a - b) / abs(b) for a, b in zip(e_gpu, e_cpu))
    x_abs = float(np.abs(x_gpu - x_cpu).max())
    tv_rel = abs(float(tv_gpu) - tv_cpu) / abs(tv_cpu)
    ok = bool(e_rel <= 1e-5 and x_abs <= 1e-5 and tv_rel <= 1e-5)
    gate = {"passed": ok, "checker": kind, "sample": list(shape), "iterations": iters, "energy_rel_err_max": e_rel, "x_abs_err_max": x_abs,
            "tv_rel_err": tv_rel, "tolerance": {"energy_rel": 1e-5, "x_abs": 1e-5, "tv_rel": 1e-5},
            "what": "GPU float32 CP-ROF iterations vs the %s numpy CPU path (float32 state, float64 sums) on the same seeded slab at the benchmark's plane size"
                    % ("reference's (baseline/_ref, unmodified)" if kind == "reference" else "oracle's")}
    vox = int(np.prod(shape))
    cpu = {"value": vox * iters / dt, "unit": UNIT, "cores": 1, "kind": kind, "host_cpu": _cpu_model(), "host_cpu_count": os.cpu_count(),
           "sample": "%d CP-ROF iterations on a %s float32 slab of the same workload and plane size (the parity-gate run), %.1f s"
                     % (iters, "x".join(map(str, shape)), dt)}
    return gate, cpu


def disc(N, frac, dev=None):
    import torch
    r = torch.arange(N, dtype=torch.float32) - (N - 1) / 2.0
    m = (r[:, None] ** 2 + r[None, :] ** 2) <= (frac * N) ** 2
    return m if dev is None else m.to(dev)


def parity_gate_c5(dev):
    """C5: every scheme's tv (with mask), D and D_T on a reduced slab against the CPU checker."""
    import torch
    import pytv_b200 as pytv
    from oracle import tv_oracle as orc
    w = WORKLOADS["C5"]
    shape = tuple(w["gate"])
    N = shape[-1]
    x = make_sample(777, shape)
    mask = disc(N, 0.48).numpy()
    ms = disc(N, 0.25).numpy().reshape(1, 1, N, N)
    kw = dict(reg_time=w["kw"]["reg_time"], mask_static=ms, factor_reg_static=w["kw"]["factor_reg_static"])
    worst = {"tv_rel": 0.0, "G_abs": 0.0, "D_abs": 0.0, "DT_abs": 0.0}
    t0 = time.perf_counter()
    for scheme in SCHEMES:
        xm = x * mask
        tv_o, G_o = orc.tv(xm.astype(np.float64), scheme, **kw)
        D_o = orc.D(xm.astype(np.float64), scheme, **kw)
        DT_o = orc.D_T(D_o, scheme, **kw)
        xg = torch.from_numpy(x.copy()).to(dev)
        tv_g, G_g = getattr(pytv.tv_GPU, "tv_" + scheme)(xg, mask=torch.from_numpy(mask).to(dev), return_pytorch_tensor=True, **kw)
        D_g = getattr(pytv.tv_operators_GPU, "D_" + scheme)(xg, **kw)       # xg was zeroed outside the mask in place
        DT_g = getattr(pytv.tv_operators_GPU, "D_T_" + scheme)(D_g, **kw)
        worst["tv_rel"] = max(worst["tv_rel"], abs(float(tv_g) - tv_o) / abs(tv_o))
        # sub-gradient tolerance: 1e-5 absolute, or the float32 rounding floor of the formula where D/|D| is ill-conditioned
        _, G_o32 = orc.tv(xm, scheme, **kw)
        floor = float(np.abs(G_o32 - G_o).max())
        worst["G_abs"] = max(worst["G_abs"], float(np.abs(G_g.cpu().numpy() - G_o).max()) / max(1.0, 3.0 * floor / 1e-5))
        worst["D_abs"] = max(worst["D_abs"], float(np.abs(D_g.cpu().numpy() - D_o).max()))
        worst["DT_abs"] = max(worst["DT_abs"], float(np.abs(DT_g.cpu().numpy() - DT_o).max()))
    ok = bool(worst["tv_rel"] <= 1e-5 and worst["G_abs"] <= 1e-5 and worst["D_abs"] <= 1e-5 and worst["DT_abs"] <= 1e-5)
    return {"passed": ok, "checker": "port", "sample": list(shape), "tv_rel_err_max": worst["tv_rel"], "G_abs_err_max_normalised": worst["G_abs"],
            "D_abs_err_max": worst["D_abs"], "DT_abs_err_max": worst["DT_abs"], "seconds": time.perf_counter() - t0,
            "what": "tv (with mask) / D / D_T of the four schemes, float32 on the GPU vs the float64 oracle; G is held to max(1e-5, 3 x the float32 "
                    "rounding floor of the reference formula evaluated in numpy float32)"}


# (2) multi-GPU self-check
def multi_gpu_check(dev, rank, world, comm, kw):
    """Every rank computes a small whole volume alone; the group computes it sharded with the halo transport of the timed
    run; the slabs must equal the whole-volume result bit for bit (x, xbar, y) after 3 iterations."""
    import torch
    import torch.distributed as dist
    import pytv_b200 as pytv
    nz = 3
    shape = (nz * world, 4, 96, 512)
    g = torch.Generator(device="cpu").manual_seed(99)
    x0 = (torch.rand(shape, generator=g) + 0.05 * torch.randn(shape, generator=g)).to(dev)
    whole = pytv.CPSolver(x0, lam=LAM, scheme="hybrid", variant="rof", **kw)
    whole.step(3)
    e_whole = whole.energy()
    a, b = rank * nz, (rank + 1) * nz
    sh = pytv.CPSolver(x0[a:b].clone(), lam=LAM, scheme="hybrid", variant="rof", distributed=True, z_offset=a, Nz_global=shape[0], comm=comm, **kw)
    sh.step(3)
    e_sh = sh.energy()
    ok = torch.equal(sh.x, whole.x[a:b]) and torch.equal(sh.aux, whole.aux[a:b]) and torch.equal(sh.y, whole.y[a:b])
    ok = ok and abs(e_sh - e_whole) <= 1e-9 * abs(e_whole)
    flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    transport = "p2p" if sh._peer is not None else "nccl"
    del sh, whole
    return ("bitwise_equal" if int(flag.item()) == 1 else "MISMATCH"), transport


# (4) host link
def link_peak(dev, h_in, h_out, world, reps=3):
    """Pinned cudaMemcpyAsync H2D and D2H at the same time (the traffic pattern of the pipelined e2e loop), every rank at
    once; GB/s per direction of THIS rank (best of `reps`)."""
    import torch
    import torch.distributed as dist
    d_in = torch.empty_like(h_in, device=dev)
    d_out = torch.empty_like(h_out, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    best = None
    for _ in range(reps + 1):
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        with torch.cuda.stream(s1):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_out, non_blocking=True)
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return h_in.numel() * h_in.element_size() / best / 1e9


def init_dist(dev):
    import torch
    import torch.distributed as dist
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    # NCCL prints its version banner on stdout: keep stdout clean for the one JSON line
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()
        warm = torch.zeros(1, device=dev)
        dist.all_reduce(warm)
        torch.cuda.synchronize()
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)


# --dump-outputs
def sample_positions(numel, n, dev):
    """`n` flat positions in [0, numel) drawn from a fixed seed (the same in every run), or None when all `numel` fit."""
    import torch
    if numel <= n:
        return None
    return torch.from_numpy(np.random.RandomState(0).randint(0, numel, size=n, dtype=np.int64)).to(dev)


def take(t, pos):
    """The elements of `t` at the flat positions `pos` (all of `t` when None), as a new tensor on t's device."""
    return t.detach().clone() if pos is None else t.detach().reshape(-1)[pos]


def write_outputs(out_dir, arrays, rank, world):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.cpu().numpy() if hasattr(a, "cpu") else a
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ("_rank%d" % rank if world > 1 else "") + ".npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist
    import pytv_b200 as pytv
    from pytv_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        init_dist(dev)
    if args.gpus != world and rank == 0:
        print("bench.py: --gpus %d but WORLD_SIZE=%d; running on %d" % (args.gpus, world, world), file=sys.stderr)
    lib = _lib.lib()
    wl = args.workload
    w = WORKLOADS[wl]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- (1) parity gate on rank 0 (the other ranks wait), before any timing counts (BASELINE.md section 3)
    gate, cpu_base = None, None
    if not args.no_parity_gate:
        if rank == 0:
            if wl == "C5":
                gate = parity_gate_c5(dev)
            else:
                gate, cpu_base = parity_gate_cp(wl, dev)
        gate_ok = torch.tensor([1 if (gate is None or gate["passed"]) else 0], dtype=torch.int32, device=dev)
        if world > 1:
            dist.all_reduce(gate_ok, op=dist.ReduceOp.MIN)
        if int(gate_ok.item()) == 0:
            if rank == 0:
                print(json.dumps({"metric": w["metric"], "value": None, "unit": UNIT, "n_gpus": world, "parity_gate": gate,
                                  "error": "parity gate failed: no timing is reported for a path whose results differ from the reference's"}), flush=True)
            if world > 1:
                dist.destroy_process_group()
            raise SystemExit(2)
    # ---- (2) sharded-vs-whole self-check with the transport of the timed run
    comm = args.comm if world > 1 else "nccl"
    mg_check, mg_transport = None, None
    if world > 1 and not args.no_parity_gate:
        mg_check, mg_transport = multi_gpu_check(dev, rank, world, comm, dict(reg_time=2.0 ** -5))
        if mg_check != "bitwise_equal":
            if rank == 0:
                print(json.dumps({"metric": w["metric"], "value": None, "unit": UNIT, "n_gpus": world, "parity_gate": gate, "multi_gpu_check": mg_check,
                                  "error": "sharded result differs from the whole-volume result"}), flush=True)
            dist.destroy_process_group()
            raise SystemExit(3)
    torch.cuda.empty_cache()
    if wl == "C5":
        return run_c5(args, dev, rank, world, gate, mg_check, barrier)

    K, W = args.steps, max(3, args.warmup)
    shape = tuple(args.slab) if args.slab else tuple(w["slab"])
    kw = w["kw"]
    V_local = int(np.prod(shape))
    # ---- synthetic data, seeded per rank (BASELINE.md C4: uniform [0,1) + 0.05 randn, seed 1000+rank; C3: blocks + 0.1 randn)
    g = torch.Generator(device=dev).manual_seed(1000 + rank)
    if wl == "C3":
        bl = (torch.randint(0, 3, tuple((s + 63) // 64 for s in shape), generator=g, device=dev).float() * 0.5)
        for ax in (0, 2, 3):
            bl = bl.repeat_interleave(64, dim=ax)
        x0 = bl[:shape[0], :, :shape[2], :shape[3]].contiguous() + 0.1 * torch.randn(shape, generator=g, device=dev)
        del bl
    else:
        x0 = torch.rand(shape, generator=g, device=dev) + 0.05 * torch.randn(shape, generator=g, device=dev)
    solver = pytv.CPSolver(x0, lam=LAM, scheme="hybrid", variant="rof", distributed=(world > 1), z_offset=rank * shape[0] if world > 1 else None,
                           Nz_global=world * shape[0] if world > 1 else None, comm=comm, **kw)
    del x0
    assert solver.Nd == w["Nd"] or args.slab

    # ---- (3) device-resident timing
    for _ in range(W):
        solver.step()
        solver.energy()
        if world > 1:
            solver.energy_result(solver.energy_async())
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    time.sleep(0.3)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = lib.pytvb_launch_count()
    barrier()
    start.record()
    for k in range(K):
        # the solver's step(), spelled out so that the two passes can be bracketed by events on their stream
        ev[k][0].record()
        solver._pass_A()
        ev[k][1].record()
        solver._pass_B()
        ev[k][2].record()
        solver.iterations += 1
        if world > 1:
            pending_energy = solver.energy_async()     # scalar all-reduce for the energy, every iteration (own communicator)
    if world > 1:
        solver.energy_result(pending_energy)           # the last all-reduce lands inside the timed region
    end.record()
    barrier()
    launches = lib.pytvb_launch_count() - launches0
    t_ms = start.elapsed_time(end)
    clocks = sampler.stop() if sampler else None
    energy = solver.energy()
    if args.dump_outputs:      # before the end-to-end timing below iterates the solver further
        pos = sample_positions(solver.x.numel(), DUMP_BYTES // world // 4, dev)
        write_outputs(args.dump_outputs, {"x": take(solver.x, pos), "energy": np.array([energy], np.float64)}, rank, world)
    dual_ms = sum(e[0].elapsed_time(e[1]) for e in ev) / K
    primal_ms = sum(e[1].elapsed_time(e[2]) for e in ev) / K
    per_rank = None
    if world > 1:
        mine = torch.tensor([t_ms, dual_ms, primal_ms], dtype=torch.float64, device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = {"total_ms": [float(a[0]) for a in allr], "pass_A_ms": [float(a[1]) for a in allr], "pass_B_ms": [float(a[2]) for a in allr]}
        t = mine.clone()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_ms, dual_ms, primal_ms = t.tolist()
    value = V_local * world * K / (t_ms * 1e-3)

    # ---- (4) end to end through the host-buffer API (pinned host memory in and out, every step)
    # step_host_async pipelines the three legs of a step (upload of x0 | the two passes | download of x and the energy)
    # across consecutive steps, three steps in flight; every step still uploads its data and downloads its result inside
    # the timed region, and the region ends only when the last download has landed.
    D = solver.PIPE_DEPTH
    x0_host = torch.empty(shape, dtype=torch.float32).pin_memory()
    x0_host.copy_(solver.x0)
    x_hosts = [torch.empty(shape, dtype=torch.float32).pin_memory() for _ in range(D)]
    link = link_peak(dev, x0_host, x_hosts[0], world)
    for _ in range(D):
        solver.wait(solver.step_host_async(x0_host, x_hosts[0]))
    barrier()
    t0 = time.perf_counter()
    tickets = []
    for k in range(K):
        tickets.append(solver.step_host_async(x0_host, x_hosts[k % D]))
        if len(tickets) >= D:
            solver.wait(tickets.pop(0))
    while tickets:
        e2e_energy = solver.wait(tickets.pop(0))
    barrier()
    e2e_s = time.perf_counter() - t0
    # the unpipelined call, for reference
    t1 = time.perf_counter()
    for _ in range(3):
        solver.step_host(x0_host, x_hosts[0])
    torch.cuda.synchronize()
    e2e_sync_ms = (time.perf_counter() - t1) / 3 * 1e3
    link_all = link
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t[0])
        t = torch.tensor([link], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        link_all = float(t[0])
    e2e_value = V_local * world * K / e2e_s
    img_bytes = V_local * 4

    # ---- informational: the opt-in reduced-precision mode (dual field stored as normalised half; NOT the parity path)
    extras = {}
    if world == 1 and not args.no_extras and wl == "C4":
        hs = pytv.CPSolver(solver.x0, lam=LAM, scheme="hybrid", variant="rof", dual_dtype=torch.float16, **kw)
        for _ in range(W):
            hs.step()
        torch.cuda.synchronize()
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0.record()
        hs.step(K)
        h1.record()
        torch.cuda.synchronize()
        hms = h0.elapsed_time(h1) / K
        hbytes = (6.0 * hs.Nd + 20.0) * V_local
        extras["half_precision_dual_storage"] = {"ms_per_step": hms, "value": V_local / (hms * 1e-3), "unit": UNIT, "bytes_per_voxel": 6 * hs.Nd + 20,
                                                 "achieved_GBps": hbytes / (hms * 1e-3) / 1e9,
                                                 "note": "CPSolver(dual_dtype=torch.float16): opt-in, max error ~3e-4 on [0,1] data; not the headline"}
        del hs

    if rank == 0:
        Nd = solver.Nd
        peak, peak_src = measured_hbm_peak()
        dual_bytes = 4.0 * (2 * Nd + 1) * V_local       # read xbar, read y, write y  (SURVEY 8d: pass A of 4(3Nd+5))
        primal_bytes = 4.0 * (Nd + 4) * V_local         # read y, x, x0; write x, xbar
        achieved = dual_bytes / (dual_ms * 1e-3) / 1e9
        traffic = recorded_traffic() if wl == "C4" and not args.slab else {}
        roofline = {"bound": "hbm", "kernel": "cp_dual_strip_kernel (pass A)", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": dual_bytes, "avg_launch_ms": dual_ms,
                    "traffic": traffic.get("cp_dual_strip_kernel"),
                    "pass_B": {"kernel": "cp_primal_strip_kernel", "achieved": primal_bytes / (primal_ms * 1e-3) / 1e9,
                               "frac": primal_bytes / (primal_ms * 1e-3) / 1e9 / peak, "avg_launch_ms": primal_ms,
                               "traffic": traffic.get("cp_primal_strip_kernel")},
                    "iteration": {"algorithmic_bytes": dual_bytes + primal_bytes, "achieved": (dual_bytes + primal_bytes) * K / (t_ms * 1e-3) / 1e9,
                                  "frac": (dual_bytes + primal_bytes) * K / (t_ms * 1e-3) / 1e9 / peak},
                    "build_id": lib_build_id()}
        e2e_gbps = img_bytes * world / (e2e_s / K) / 1e9
        line = {"metric": w["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": t_ms / K,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config_dict(wl, world, {"slab_per_gpu": list(shape), "energy_last": energy,
                                                  "halo_comm": "none (one GPU)" if world == 1 else
                                                  ("p2p (kernels store boundary planes into the neighbours' halo buffers over NVLink)"
                                                   if solver._peer is not None else "nccl send/recv")}),
                "parity_gate": gate if gate is not None else "skipped (--no-parity-gate)",
                "roofline": roofline,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": img_bytes * world, "d2h_bytes_per_step": (img_bytes + 48) * world,
                        "ms_per_step": 1e3 * e2e_s / K, "ms_per_step_unpipelined": e2e_sync_ms,
                        "link_peak_GBps": link_all, "achieved_GBps_per_direction": e2e_gbps, "frac_of_link": e2e_gbps / link_all,
                        "link_peak_what": "pinned cudaMemcpyAsync H2D and D2H of one image at the same time, all %d rank(s) at once, sum over ranks, "
                                          "GB/s per direction (measured in this run)" % world,
                        "what": "CPSolver.step_host_async/wait: every step uploads x0 from pinned host memory, runs one iteration, "
                                "downloads x and the energy; %d consecutive steps in flight over two copy streams" % D},
                "gpu_launches": int(launches), "clocks": clocks}
        if mg_check is not None:
            line["multi_gpu_check"] = mg_check
            line["multi_gpu_check_what"] = ("3 CP iterations on a (%d, 4, 96, 512) volume: every rank alone vs the group sharded over %s halos; x, xbar, y compared "
                                            "with torch.equal on every rank" % (3 * world, mg_transport))
        if extras:
            line["extras"] = extras
        if per_rank:
            line["per_rank"] = per_rank      # event times of every rank (the headline uses the max)
        if cpu_base is not None and world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_base
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------------------
def run_c5(args, dev, rank, world, gate, mg_check, barrier):
    """BASELINE config 5: the four schemes' fused tv (with mask), D and D_T on this rank's (64, 8, 2048, 2048) slab of the
    sharded volume, through pytv.sharded.ShardedTV (halo planes + one all-reduced double per tv)."""
    import torch
    import torch.distributed as dist
    import pytv_b200 as pytv
    from pytv_b200 import _lib, sharded
    lib = _lib.lib()
    w = WORKLOADS["C5"]
    K, W = args.steps, max(3, args.warmup)
    shape = tuple(args.slab) if args.slab else tuple(w["slab"])
    N = shape[-1]
    V_local = int(np.prod(shape))
    g = torch.Generator(device=dev).manual_seed(1000 + rank)
    x = torch.rand(shape, generator=g, device=dev)
    mask = disc(N, 0.48, dev)
    x *= mask                                   # the mask is applied once here; tv() applies it again in place (idempotent)
    ms = disc(N, 0.25, dev).reshape(1, 1, N, N)
    if world == 1:
        # one GPU: the plain drop-in calls
        class Plain:
            def __init__(self, scheme):
                self.kw = dict(reg_time=w["kw"]["reg_time"], mask_static=ms, factor_reg_static=w["kw"]["factor_reg_static"])
                self.scheme = scheme

            def tv(self, x, mask=None):
                t, G = getattr(pytv.tv_GPU, "tv_" + self.scheme)(x, mask=mask, return_pytorch_tensor=True, **self.kw)
                return t, G

            def D(self, x):
                return getattr(pytv.tv_operators_GPU, "D_" + self.scheme)(x, **self.kw)

            def D_T(self, p):
                return getattr(pytv.tv_operators_GPU, "D_T_" + self.scheme)(p, **self.kw)
        ops = {s: Plain(s) for s in SCHEMES}
    else:
        ops = {s: sharded.ShardedTV(s, reg_time=w["kw"]["reg_time"], mask_static=ms, factor_reg_static=w["kw"]["factor_reg_static"],
                                    comm=args.comm) for s in SCHEMES}
    times = {s: {"tv": 0.0, "D": 0.0, "D_T": 0.0} for s in SCHEMES}
    Nd_of = {}
    tv_vals = {}

    def one_pass(record, dump=None, pos=None):
        for s in SCHEMES:
            e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            e[0].record()
            tvv, G = ops[s].tv(x, mask=mask)
            e[1].record()
            Dx = ops[s].D(x)
            e[2].record()
            out = ops[s].D_T(Dx)
            e[3].record()
            Nd_of[s] = int(Dx.shape[1])
            tv_vals[s] = float(tvv)
            if dump is not None:      # gathered on the device here: the fields of all four schemes do not fit in memory together
                dump.update({"tv_" + s: np.array([tv_vals[s]], np.float64), "G_" + s: take(G, pos[G.numel()]), "D_" + s: take(Dx, pos[Dx.numel()]),
                             "D_T_" + s: take(out, pos[out.numel()])})
            del G, Dx, out
            if record:
                torch.cuda.synchronize()
                for k, name in enumerate(("tv", "D", "D_T")):
                    times[s][name] += e[k].elapsed_time(e[k + 1])

    for _ in range(W):
        one_pass(False)
    barrier()
    sampler = ClockSampler(dev.index) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = lib.pytvb_launch_count()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    dump, pos = None, None
    if args.dump_outputs:      # the positions are drawn before the timed region; the last timed step only gathers
        dump = {}
        pos = {m: sample_positions(m, DUMP_BYTES // world // 4 // (3 * len(SCHEMES)), dev) for m in [V_local] + [Nd_of[s] * V_local for s in SCHEMES]}
    start.record()
    for k in range(K):
        one_pass(True, dump if k == K - 1 else None, pos)
    end.record()
    barrier()
    launches = lib.pytvb_launch_count() - launches0
    clocks = sampler.stop() if sampler else None
    t_ms = start.elapsed_time(end)
    if dump is not None:
        write_outputs(args.dump_outputs, dump, rank, world)
    flat = torch.tensor([times[s][o] / K for s in SCHEMES for o in ("tv", "D", "D_T")] + [t_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.MAX)
    flat = flat.tolist()
    t_ms = flat[-1]
    value = V_local * world * 12 * K / (t_ms * 1e-3)
    # e2e: numpy in / numpy out through the drop-in call (the reference's default convention), one scheme, a reduced slab per step
    e2e_shape = (4,) + shape[1:]
    xh = torch.rand(e2e_shape).pin_memory().numpy()
    for _ in range(2):
        pytv.tv_GPU.tv_hybrid(xh, reg_time=w["kw"]["reg_time"])
    barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        tvh, Gh = pytv.tv_GPU.tv_hybrid(xh, reg_time=w["kw"]["reg_time"])
    e2e_s = (time.perf_counter() - t0) / 3
    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        per_op = {}
        k = 0
        for s in SCHEMES:
            Nd = Nd_of[s]
            per_op[s] = {"Nd": Nd}
            for o, bpv in (("tv", 8 + 1), ("D", 4 * (1 + Nd)), ("D_T", 4 * (Nd + 1))):
                ms_ = flat[k]
                k += 1
                gbps = bpv * V_local / (ms_ * 1e-3) / 1e9
                per_op[s][o] = {"ms": ms_, "bytes_per_voxel": bpv, "achieved_GBps": gbps, "frac": gbps / peak}
        dom = per_op["hybrid"]["D"]
        line = {"metric": w["metric"], "value": value, "unit": "voxel-operator-applications/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": t_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config_dict("C5", world, {"slab_per_gpu": list(shape), "tv_values": tv_vals,
                                                    "halo_comm": "none (one GPU)" if world == 1 else getattr(ops["hybrid"], "transport", "nccl")}),
                "parity_gate": gate if gate is not None else "skipped (--no-parity-gate)",
                "roofline": {"bound": "hbm", "kernel": "D_strip_kernel (hybrid, Nd=8; the largest share of the step)", "achieved": dom["achieved_GBps"],
                             "peak": peak, "unit": "GB/s", "frac": dom["frac"], "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": dom["bytes_per_voxel"] * V_local, "avg_launch_ms": dom["ms"], "traffic": None,
                             "build_id": lib_build_id()},
                "per_op": per_op,
                "e2e": {"value": int(np.prod(e2e_shape)) / e2e_s, "unit": "voxels/s", "h2d_bytes_per_step": int(np.prod(e2e_shape)) * 4,
                        "d2h_bytes_per_step": int(np.prod(e2e_shape)) * 4 + 8, "ms_per_step": e2e_s * 1e3,
                        "what": "pytv.tv_GPU.tv_hybrid(numpy float32 %s) -> (tv, G as numpy): the reference's default numpy-in / numpy-out call, "
                                "pageable host memory, on rank 0" % (list(e2e_shape),)},
                "gpu_launches": int(launches), "clocks": clocks}
        if mg_check is not None:
            line["multi_gpu_check"] = mg_check
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="C4", help="BASELINE config: C4 (default, the headline), C3, C5")
    ap.add_argument("--comm", choices=["auto", "nccl", "p2p"], default=os.environ.get("PYTVB_BENCH_COMM", "auto"),
                    help="N > 1: halo planes by NCCL send/recv between the passes, or pushed by the kernels into peer memory")
    ap.add_argument("--slab", type=int, nargs=4, default=None, help="override the per-GPU slab (Nz M Ni Nj); debugging only")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="leave the cpu_baseline object out of the line")
    ap.add_argument("--no-parity-gate", action="store_true", help="skip the parity gate and the multi-GPU check (profiling runs under ncu only)")
    ap.add_argument("--no-extras", action="store_true", help="skip the informational reduced-precision measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

"""Fused Chambolle-Pock TV denoising: two HBM passes per iteration, state resident on the device.

The reference ships no solver, only the loop in README.md:139-158 (and examples/a_getting_started.ipynb
cell 5) that users build from D_hybrid / D_T_hybrid / compute_L21_norm with all point-wise maths on the
host.  This module is that loop as a library:

  variant="readme"  the README's "simple" iteration, state (x, y_f, y_tv): bit-for-bit the same update order
  variant="rof"     Chambolle & Pock (2011) Alg. 1 for 0.5|x-x0|^2 + lam TV(x), state (x, xbar, y): exact
                    prox of the data term and over-relaxation.  With data_term="l1" and / or a data_weight map w the
                    data term becomes sum_v w_v |x_v - x0_v| (TV-L1: impulse noise, dead / hot pixels) or
                    0.5 sum_v w_v (x_v - x0_v)^2 (confidence weights; w = 0 marks missing voxels that TV fills in)

Each iteration is pass A (dual: D(xbar), projection onto the lam-ball, L21 partial sums) and pass B (primal:
D^T y, data-term update, over-relaxation, fidelity partial sums), i.e. `pytvb_cp_dual` + `pytvb_cp_primal_*`.

Multi-GPU: one process per GPU, each owning a contiguous slab of z planes (the layout is z-major, so a slab
is one contiguous byte range; README.md:235).  Before pass A the boundary planes of xbar go to the two
z-neighbours, before pass B the boundary planes of the z-components of y; the energy needs one all-reduce
of two doubles.  M and N are never split.  With the z axis off the slabs are independent.
"""
import ctypes
import os

import numpy as np
import torch

from . import _dev, _lib


DATA_TERMS = {"l2": 0, "l1": 1}     # pytvb_data_term


def partition_z(Nz_global, world_size):
    """Contiguous, balanced z-slabs: [(offset, count)] for every rank (earlier ranks take the remainder)."""
    if Nz_global < world_size:
        raise ValueError("cannot split %d planes over %d ranks" % (Nz_global, world_size))
    base, rem = divmod(Nz_global, world_size)
    out, off = [], 0
    for r in range(world_size):
        n = base + (1 if r < rem else 0)
        out.append((off, n))
        off += n
    return out


def operator_norm_sq_bound(scheme, z_on, t_on, reg_z_over_reg, reg_time, factor_reg_static, has_mask_static, max_time_weight=1.0):
    """Upper bound of |D|^2: 4 per unit-weight axis for the one-sided schemes and hybrid, 1 for central.  The time axis
    carries reg_time x (factor_reg_static where mask_static) x (the largest entry of a time_weight map)."""
    w = 2.0
    if z_on:
        w += reg_z_over_reg
    if t_on:
        w += reg_time * (max(1.0, factor_reg_static) if has_mask_static else 1.0) * max(1.0, float(max_time_weight))
    return w if scheme == "central" else 4.0 * w


class CudaOps:
    """The product path: every pass is one call into libpytv_b200.so on the current stream."""

    def __init__(self):
        self.lib = _lib.lib()

    def cp_dual(self, pb, xbar, y, lam, sigma, d_l21, lo, hi, ws):
        if y.dtype == torch.float16:
            _lib.check(self.lib.pytvb_cp_dual_f16y(ctypes.byref(pb), _dev.ptr(xbar), _dev.ptr(y), lam, sigma, _dev.ptr(d_l21), _dev.ptr(lo),
                                                   _dev.ptr(hi), _dev.ptr(ws), _dev.stream_ptr()))
            return
        _lib.check(self.lib.pytvb_cp_dual(ctypes.byref(pb), _dev.ptr(xbar), _dev.ptr(y), lam, sigma, _dev.ptr(d_l21), _dev.ptr(lo), _dev.ptr(hi),
                                          _dev.ptr(ws), _dev.stream_ptr()))

    def cp_primal(self, variant, pb, y, x, aux, x0, tau, c2, d_fid, lo, hi, ws, lam=None):
        if y.dtype == torch.float16:
            _lib.check(self.lib.pytvb_cp_primal_rof_f16y(ctypes.byref(pb), _dev.ptr(y), _dev.ptr(x), _dev.ptr(aux), _dev.ptr(x0), lam, tau, c2,
                                                         _dev.ptr(d_fid), _dev.ptr(lo), _dev.ptr(hi), _dev.ptr(ws), _dev.stream_ptr()))
            return
        fn = self.lib.pytvb_cp_primal_rof if variant == "rof" else self.lib.pytvb_cp_primal_readme
        _lib.check(fn(ctypes.byref(pb), _dev.ptr(y), _dev.ptr(x), _dev.ptr(aux), _dev.ptr(x0), tau, c2, _dev.ptr(d_fid), _dev.ptr(lo), _dev.ptr(hi),
                      _dev.ptr(ws), _dev.stream_ptr()))

    def cp_primal_data(self, pb, data_term, w, y, x, xbar, x0, tau, theta, d_fid, lo, hi, mirror_prev, mirror_next, ws):
        _lib.check(self.lib.pytvb_cp_primal_data(ctypes.byref(pb), DATA_TERMS[data_term], _dev.ptr(w), _dev.ptr(y), _dev.ptr(x), _dev.ptr(xbar),
                                                 _dev.ptr(x0), tau, theta, _dev.ptr(d_fid), _dev.ptr(lo), _dev.ptr(hi), mirror_prev, mirror_next,
                                                 _dev.ptr(ws), _dev.stream_ptr()))

    def cp_dual_p2p(self, pb, xbar, y, lam, sigma, d_l21, lo, hi, mirror_prev, mirror_next, ws):
        _lib.check(self.lib.pytvb_cp_dual_p2p(ctypes.byref(pb), _dev.ptr(xbar), _dev.ptr(y), lam, sigma, _dev.ptr(d_l21), _dev.ptr(lo), _dev.ptr(hi),
                                              mirror_prev, mirror_next, _dev.ptr(ws), _dev.stream_ptr()))

    def cp_primal_p2p(self, variant, pb, y, x, aux, x0, tau, c2, d_fid, lo, hi, mirror_prev, mirror_next, ws):
        _lib.check(self.lib.pytvb_cp_primal_p2p(ctypes.byref(pb), 0 if variant == "rof" else 1, _dev.ptr(y), _dev.ptr(x), _dev.ptr(aux), _dev.ptr(x0),
                                                tau, c2, _dev.ptr(d_fid), _dev.ptr(lo), _dev.ptr(hi), mirror_prev, mirror_next, _dev.ptr(ws),
                                                _dev.stream_ptr()))

    def cp_dual_adj(self, pb, xbar, y, q, lam, sigma, d_l21, lo, hi, mirror_prev, mirror_next, ws):
        _lib.check(self.lib.pytvb_cp_dual_adj_p2p(ctypes.byref(pb), _dev.ptr(xbar), _dev.ptr(y), _dev.ptr(q), lam, sigma, _dev.ptr(d_l21), _dev.ptr(lo),
                                                  _dev.ptr(hi), mirror_prev, mirror_next, _dev.ptr(ws), _dev.stream_ptr()))

    def cp_primal_adj(self, pb, data_term, w, y, q, x, xbar, x0, tau, theta, d_fid, lo, hi, mirror_prev, mirror_next, ws):
        _lib.check(self.lib.pytvb_cp_primal_adj_p2p(ctypes.byref(pb), DATA_TERMS[data_term], _dev.ptr(w), _dev.ptr(y), _dev.ptr(q), _dev.ptr(x),
                                                    _dev.ptr(xbar), _dev.ptr(x0), tau, theta, _dev.ptr(d_fid), _dev.ptr(lo), _dev.ptr(hi), mirror_prev,
                                                    mirror_next, _dev.ptr(ws), _dev.stream_ptr()))

    def workspace(self, pb, device):
        return _dev.reduce_workspace(pb, device)

    def tv_value(self, pb, x, d_tv, lo, hi, ws):
        _lib.check(self.lib.pytvb_tv_value(ctypes.byref(pb), _dev.ptr(x), _dev.ptr(d_tv), _dev.ptr(lo), _dev.ptr(hi), _dev.ptr(ws), _dev.stream_ptr()))

    def adjoint(self, pb, y, out, lo, hi):
        _lib.check(self.lib.pytvb_DT(ctypes.byref(pb), _dev.ptr(y), _dev.ptr(out), _dev.ptr(lo), _dev.ptr(hi), _dev.stream_ptr()))


class HaloExchange:
    """Nearest-neighbour plane exchange between z-slabs over torch.distributed (NCCL send/recv on NVLink;
    gloo in the CPU tests)."""

    def __init__(self, group=None, reduce_group=None):
        import torch.distributed as dist
        self.dist = dist
        self.group = group
        self._reduce_group = reduce_group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        self.prev = self.rank - 1 if self.rank > 0 else None
        self.next = self.rank + 1 if self.rank < self.world - 1 else None

    def _global(self, r):
        return r if self.group is None else self.dist.get_global_rank(self.group, r)

    def exchange(self, to_prev, to_next, from_prev, from_next):
        """Blocking form of start_exchange + finish."""
        self.finish(self.start_exchange(to_prev, to_next, from_prev, from_next))

    def finish(self, reqs):
        """Make the current stream (NCCL) / the host (gloo) wait for an exchange started earlier."""
        for req in reqs or ():
            req.wait()

    def start_exchange(self, to_prev, to_next, from_prev, from_next):
        """Send plane `to_prev` to rank-1 and `to_next` to rank+1; receive into `from_prev` / `from_next`.
        Any of the four may be None (direction not needed by the scheme).  Returns the outstanding requests: with
        NCCL the transfers run on NCCL's stream, ordered after everything enqueued so far on the current stream,
        and overlap whatever is launched next."""
        ops = []
        P2P = self.dist.P2POp
        if self.prev is not None:
            if to_prev is not None:
                ops.append(P2P(self.dist.isend, to_prev, self._global(self.prev), self.group))
            if from_prev is not None:
                ops.append(P2P(self.dist.irecv, from_prev, self._global(self.prev), self.group))
        if self.next is not None:
            if to_next is not None:
                ops.append(P2P(self.dist.isend, to_next, self._global(self.next), self.group))
            if from_next is not None:
                ops.append(P2P(self.dist.irecv, from_next, self._global(self.next), self.group))
        return self.dist.batch_isend_irecv(ops) if ops else []

    def allreduce_sum(self, t):
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.group)
        return t

    def allreduce_sum_async(self, t):
        """Scalar all-reduce, asynchronously; returns the work handle.  With a communicator of its own (`reduce_group`,
        see make_reduce_group) it never queues in front of the halo send/recv of the next pass (one NCCL communicator
        executes its operations in order); without one it runs on the solver's group."""
        g = self._reduce_group if self._reduce_group is not None else self.group
        return self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=g, async_op=True)

    def make_reduce_group(self):
        """Create the second communicator for the scalar all-reduces.  `new_group` is collective over the DEFAULT process
        group, so this is only done when the solver spans the default group (every rank then gets here, in the solver's
        constructor); a solver on a sub-group takes a caller-made `reduce_group` or shares its group."""
        if self._reduce_group is None and self.group is None:
            self._reduce_group = self.dist.new_group(ranks=list(range(self.dist.get_world_size())))


def neighbour_handshake(hdl, prev, nxt, timeout_ms, sync="auto"):
    """Device-side fence between z-NEIGHBOURS on the current stream (no data): "everything I stored into your halo buffers
    so far is visible" to both neighbours, then wait for the same from them.  Signals travel through the signal pads of the
    symmetric-memory allocation `hdl` (put_signal / wait_signal: one flag per (channel, source rank), set by the sender
    once the receiver has consumed the previous one).  A rank is therefore at most one pass ahead of its neighbours - which
    is also what makes it safe for them to overwrite its halo planes in their next pass - and a slow rank delays only its
    neighbours by one pass instead of stalling the whole group at a barrier.  All puts precede all waits on every rank, so
    the pattern cannot deadlock.  sync="barrier" (or a torch without put_signal) uses the group-wide barrier instead."""
    if sync == "barrier" or not hasattr(hdl, "put_signal"):
        hdl.barrier(channel=0, timeout_ms=timeout_ms)
        return
    if nxt is not None:
        hdl.put_signal(nxt, channel=1, timeout_ms=timeout_ms)
    if prev is not None:
        hdl.put_signal(prev, channel=2, timeout_ms=timeout_ms)
    if prev is not None:
        hdl.wait_signal(prev, channel=1, timeout_ms=timeout_ms)
    if nxt is not None:
        hdl.wait_signal(nxt, channel=2, timeout_ms=timeout_ms)


class PeerHalos:
    """The four halo planes of a rank, [img_lo, img_hi, fld_lo, fld_hi], in symmetric memory (torch.distributed.
    _symmetric_memory: cuMem allocations mapped into every rank of the node over NVLink).  The passes of the
    neighbouring ranks store into these planes directly (`peer`), the local passes read them (`local`); `barrier` is
    the fence between passes: a device-side handshake with the two z-neighbours only (neighbour_handshake)."""
    IMG_LO, IMG_HI, FLD_LO, FLD_HI = 0, 1, 2, 3

    def __init__(self, halo, plane, dtype, device):
        import torch.distributed._symmetric_memory as symm
        group = halo.group if halo.group is not None else halo.dist.group.WORLD
        self.buf = symm.empty((4,) + tuple(plane), dtype=dtype, device=device)
        self.hdl = symm.rendezvous(self.buf, group)
        self.buf.zero_()
        self.plane_bytes = self.buf[0].numel() * self.buf.element_size()
        self.timeout_ms = int(os.environ.get("PYTVB_P2P_TIMEOUT_MS", "60000"))   # a lost rank traps instead of hanging the GPU
        self.sync = os.environ.get("PYTVB_P2P_SYNC", "auto")                      # "barrier": the group-wide fence of round 1 (A/B runs)
        self.prev, self.next = halo.prev, halo.next
        self.hdl.barrier(channel=0, timeout_ms=self.timeout_ms)                  # everyone has zeroed its planes and signal pads are idle

    def local(self, slot):
        return self.buf[slot]

    def peer(self, rank, slot):
        """Address of plane `slot` of rank `rank` (rank within the solver's group) as mapped into this process."""
        return None if rank is None else int(self.hdl.buffer_ptrs[rank]) + slot * self.plane_bytes

    def barrier(self):
        neighbour_handshake(self.hdl, self.prev, self.next, self.timeout_ms, self.sync)


class CPSolver:
    """Device-resident Chambolle-Pock state for one volume, or for this rank's z-slab of a sharded volume.

    x0 : (Nz_local, M, Ni, Nj) numpy array or tensor - the noisy data of this rank's slab.
    distributed : True to shard over torch.distributed's default group (or pass `group`); the slab position is
                  derived from the rank with `partition_z` unless z_offset / Nz_global are given.
    comm : how the one-plane halos travel between z-neighbours.  "p2p": the pass kernels store their boundary planes
           straight into the neighbour's halo buffers (symmetric memory over NVLink, one node), a device-side barrier
           separates the passes; "nccl": batched isend/irecv before each pass; "auto" (default, or the environment
           variable PYTVB_COMM): p2p where every rank can set it up, else nccl.  Half-precision duals and injected
           executors always use nccl.
    data_term : "l2" (default) or "l1": the data term sum_v w_v phi(x_v - x0_v) with phi = 0.5 r^2 or |r|.
    data_weight : w, broadcast to the slab shape like time_weight (a sharded solver passes its own slab's part), finite and
                  >= 0; None means w = 1.  w = 0 marks missing data.  With "l2" and no weight the solver is exactly the ROF
                  solver.  The other data terms need variant="rof" and full-precision duals.
    """

    def __init__(self, x0, lam, scheme="hybrid", variant="rof", sigma=0.5, tau=None, theta=1.0, sigma_A=1.0, reg_z_over_reg=1.0,
                 reg_time=0.0, mask_static=False, factor_reg_static=0, distributed=False, group=None, z_offset=None, Nz_global=None,
                 ops=None, track_energy=True, dual_dtype=None, time_weight=None, comm=None, reduce_group=None, data_term="l2", data_weight=None):
        if scheme not in _dev.SCHEMES:
            raise ValueError("unknown scheme %r" % (scheme,))
        if variant not in ("rof", "readme"):
            raise ValueError("variant must be 'rof' or 'readme'")
        if data_term not in DATA_TERMS:
            raise ValueError("data_term must be 'l2' or 'l1'")
        self.ops = ops if ops is not None else CudaOps()
        self.scheme, self.variant = scheme, variant
        self.lam, self.sigma, self.theta, self.sigma_A = float(lam), float(sigma), float(theta), float(sigma_A)
        self.track_energy = track_energy
        shape = _dev.image_shape(x0)
        if ops is None:
            self.x0, _ = _dev.to_device(x0)
            if self.x0.data_ptr() == (x0.data_ptr() if isinstance(x0, torch.Tensor) else 0):
                self.x0 = self.x0.clone()
        else:   # injected executor (CPU tests): keep the array where it is
            self.x0 = torch.as_tensor(np.ascontiguousarray(x0)).clone() if not isinstance(x0, torch.Tensor) else x0.clone().contiguous()
        dev, dt = self.x0.device, self.x0.dtype
        self.halo = HaloExchange(group, reduce_group) if (distributed or group is not None) else None
        if self.halo is not None and self.halo.world > 1:
            if track_energy:
                self.halo.make_reduce_group()
            if (Nz_global is None) != (z_offset is None):
                raise ValueError("sharded solver: give both z_offset and Nz_global, or neither (they are then derived from the ranks' plane counts)")
            if Nz_global is None:
                counts = torch.zeros(self.halo.world, dtype=torch.int64, device=dev)
                counts[self.halo.rank] = shape[0]
                self.halo.allreduce_sum(counts)
                Nz_global = int(counts.sum().item())
                z_offset = int(counts[: self.halo.rank].sum().item())
        else:
            self.halo = None
        self.z_offset = int(z_offset or 0)
        self.Nz_global = int(Nz_global if Nz_global is not None else shape[0])
        self.shape = shape
        self._ms = None
        if not isinstance(mask_static, bool):
            if ops is None:
                self._ms = _dev.mask_static_to_device(mask_static, shape[2], shape[3])
            else:
                m = mask_static if isinstance(mask_static, torch.Tensor) else torch.as_tensor(np.asarray(mask_static))
                self._ms = (m.reshape(shape[2], shape[3]) != 0).to(torch.uint8).contiguous()
        # extension (reference TODO, README.md:258): per-voxel weight map of the time regularisation for this slab
        self._ts = None
        max_tw = 1.0
        if time_weight is not None:
            w = time_weight if isinstance(time_weight, torch.Tensor) else torch.as_tensor(np.asarray(time_weight))
            w = torch.broadcast_to(w.to(dev).to(torch.float64), shape)
            if bool((w < 0).any()):
                raise ValueError("time_weight must be >= 0")
            self._ts = torch.sqrt(w).to(dt).contiguous()
            # the default step size needs |D|^2, which grows with the largest weight (of the WHOLE volume when sharded)
            mx = w.max().reshape(1).clone()
            if self.halo is not None:
                self.halo.dist.all_reduce(mx, op=self.halo.dist.ReduceOp.MAX, group=self.halo.group)
            max_tw = float(mx.item())
        # data term: the weight map of this slab, in the image dtype; _w_min = its smallest entry over the whole volume, as stored
        # (a tiny positive weight may round to 0 in float32, and the dual energy must then be refused)
        self.data_term = data_term
        self._dw = None
        self._w_min = 1.0
        if data_weight is not None:
            w = data_weight if isinstance(data_weight, torch.Tensor) else torch.as_tensor(np.asarray(data_weight))
            w = torch.broadcast_to(w.to(dev).to(torch.float64), shape)
            if not bool(torch.isfinite(w).all()) or bool((w < 0).any()):
                raise ValueError("data_weight must be finite and >= 0")
            self._dw = w.to(dt).contiguous()
            mn = self._dw.min().double().reshape(1).clone()
            if self.halo is not None:
                self.halo.dist.all_reduce(mn, op=self.halo.dist.ReduceOp.MIN, group=self.halo.group)
            self._w_min = float(mn.item())
        self._data = data_term != "l2" or self._dw is not None    # pass B through pytvb_cp_primal_data
        self.pb = _lib.make_problem(scheme, _lib.F32 if dt == torch.float32 else _lib.F64, shape, float(reg_z_over_reg), float(reg_time),
                                    float(factor_reg_static), self._ms.data_ptr() if self._ms is not None else None, self.z_offset,
                                    self.Nz_global, self._ts.data_ptr() if self._ts is not None else None)
        self.z_on = self.Nz_global > 1 and float(reg_z_over_reg) > 0
        self.t_on = shape[1] > 1 and float(reg_time) > 0
        self.Nd = (4 + 2 * self.z_on + 2 * self.t_on) if scheme == "hybrid" else (2 + self.z_on + self.t_on)
        if tau is None:
            L2 = operator_norm_sq_bound(scheme, self.z_on, self.t_on, float(reg_z_over_reg), float(reg_time), float(factor_reg_static),
                                        self._ms is not None, max_tw)
            tau = 1.0 / (L2 + 1.0)
        self.tau = float(tau)
        # state
        self.x = self.x0.clone()
        self.aux = self.x0.clone() if variant == "rof" else torch.zeros_like(self.x0)   # xbar | y_f
        # dual_dtype=torch.float16: the dual field is STORED in half precision, normalised to the unit ball (the array
        # holds y / lam); arithmetic stays float32.  68 instead of 116 B/voxel for Nd = 8, max error ~3e-4 on [0,1]
        # images: an opt-in, not the parity path.  ROF form, float32 images.
        self.dual_dtype = dt if dual_dtype is None else dual_dtype
        if self.dual_dtype != dt:
            if self.dual_dtype != torch.float16 or dt != torch.float32 or variant != "rof":
                raise ValueError("dual_dtype=torch.float16 needs float32 images and variant='rof'")
            if not self.lam > 0:
                raise ValueError("half-precision dual storage needs lam > 0")
        if self._data and (variant != "rof" or self.dual_dtype != dt):
            raise ValueError("data_term='l1' and data_weight need variant='rof' and full-precision duals")
        self.y = torch.zeros((shape[0], self.Nd) + shape[1:], dtype=self.dual_dtype, device=dev)
        # ROF form with full-precision duals and M <= 8 frames: the dual pass also finishes the row, column and time terms of
        # D^T y into q (one image), and the primal pass adds the z term (pytvb_cp_dual_adj): 100 instead of 116 B/voxel at
        # Nd = 8, bitwise the same iterates
        self._adj = isinstance(self.ops, CudaOps) and variant == "rof" and self.dual_dtype == dt and shape[1] <= 8
        self.q = torch.empty_like(self.x0) if self._adj else None
        # partial sums of this slab: [0:3] L21(D u) and [3:6] |x - x0|^2, one slot per sub-slab call of a pass
        self.scal = torch.zeros(6, dtype=torch.float64, device=dev)
        # sharded runs: optionally run the boundary planes of each pass first and hide the halo send/recv behind the
        # interior planes (PYTVB_OVERLAP=1).  Measured on 8 x B200 (profiles/r01j_*): the exchange is ~1 % of an
        # iteration and the six extra launches of the split cost as much as it hides (10.23 vs 10.20 ms), so the
        # default is the plain exchange-then-pass schedule.
        self.overlap = os.environ.get("PYTVB_OVERLAP", "0") == "1"
        self._pending = None       # outstanding exchange of the image halos for the next dual pass
        self._field_req = None     # outstanding exchange of the field halos for the primal pass
        self._pb_cache = {}
        self.ws = self.ops.workspace(self.pb, dev)
        self.iterations = 0
        # halo planes.  comm="p2p": no exchange step at all - the planes live in symmetric memory and the passes of the
        # neighbouring ranks store into them (PeerHalos); comm="nccl": send/recv between the passes; "auto" (default,
        # or PYTVB_COMM): p2p where it can be set up on every rank, else nccl.
        self._img_lo = self._img_hi = self._fld_lo = self._fld_hi = None
        self._peer = None
        if comm is None:
            comm = os.environ.get("PYTVB_COMM", "auto")
        if comm not in ("auto", "nccl", "p2p"):
            raise ValueError("comm must be 'auto', 'nccl' or 'p2p'")
        if self.halo is not None and self.z_on:
            plane = (shape[1], shape[2], shape[3])
            interior_lo, interior_hi = self.halo.prev is not None, self.halo.next is not None
            need_img_lo, need_img_hi = scheme != "upwind", scheme != "downwind"
            need_fld_lo, need_fld_hi = scheme != "downwind", scheme != "upwind"
            p2p_ok = (ops is None and self.dual_dtype == dt and not self.overlap
                      and str(self.halo.dist.get_backend(self.halo.group)).lower() == "nccl")
            if comm == "p2p" and not p2p_ok:
                raise ValueError("comm='p2p' needs the CUDA executor over an NCCL group, the blocking schedule and full-precision duals")
            if comm != "nccl" and p2p_ok:
                # measured on 8 x B200 (profiles/r01zb_*): 9.86 ms per iteration against 10.18 ms with send/recv (one GPU: 9.60)
                try:
                    self._peer = PeerHalos(self.halo, plane, dt, dev)
                except Exception as exc:              # no symmetric memory here (multi-node group, no P2P, old driver)
                    if comm == "p2p":
                        raise
                    self._peer_error = repr(exc)
                if comm == "auto":                    # every rank must take the same path
                    ok = torch.tensor([1 if self._peer is not None else 0], dtype=torch.int32, device=dev)
                    self.halo.dist.all_reduce(ok, op=self.halo.dist.ReduceOp.MIN, group=self.halo.group)
                    if int(ok.item()) == 0:
                        self._peer = None
            if self._peer is not None:
                mk = lambda d=dt, slot=0: self._peer.local(slot)
            else:
                mk = lambda d=dt, slot=0: torch.empty(plane, dtype=d, device=dev)
            self._img_lo = mk(slot=0) if (interior_lo and need_img_lo) else None
            self._img_hi = mk(slot=1) if (interior_hi and need_img_hi) else None
            self._fld_lo = mk(self.dual_dtype, 2) if (interior_lo and need_fld_lo) else None
            self._fld_hi = mk(self.dual_dtype, 3) if (interior_hi and need_fld_hi) else None
            if self._peer is not None:
                P, h = self._peer, self.halo
                # pass A pushes: my backward-type z slot of plane 0 is the previous rank's fld_hi, my forward-type slot of
                # the last plane the next rank's fld_lo.  Pass B pushes: my first plane is the previous rank's img_hi, my
                # last plane the next rank's img_lo.
                self._mir_A = (P.peer(h.prev, P.FLD_HI) if need_fld_hi else None, P.peer(h.next, P.FLD_LO) if need_fld_lo else None)
                self._mir_B = (P.peer(h.prev, P.IMG_HI) if need_img_hi else None, P.peer(h.next, P.IMG_LO) if need_img_lo else None)
        self._zf = 4 if scheme == "hybrid" else 2   # forward-type z slot of y
        self._zb = 5 if scheme == "hybrid" else 2   # backward-type z slot

    # -- the image the dual pass differentiates: xbar (rof) or x (readme, README.md:149)
    def _dual_input(self):
        return self.aux if self.variant == "rof" else self.x

    # -- halo traffic.  Image halos: my first plane is the previous rank's halo_hi (needed unless downwind), my last
    # plane the next rank's halo_lo (unless upwind).  Field halos: the neighbour's adjoint reads my backward-type z
    # slot at its z = Nz (unless upwind) and my forward-type z slot at its z = -1 (unless downwind).
    def _image_planes(self):
        src = self._dual_input()
        return (src[0] if self.scheme != "downwind" else None, src[-1] if self.scheme != "upwind" else None)

    def _start_image_exchange(self):
        return self.halo.start_exchange(*self._image_planes(), self._img_lo, self._img_hi)

    def _start_field_exchange(self):
        to_prev = self.y[0, self._zb] if self.scheme != "upwind" else None
        to_next = self.y[-1, self._zf] if self.scheme != "downwind" else None
        return self.halo.start_exchange(to_prev, to_next, self._fld_lo, self._fld_hi)

    def _sub_problem(self, a, b):
        """Problem descriptor of local planes [a, b) (the whole slab, or a boundary / interior part of it)."""
        key = (a, b)
        pb = self._pb_cache.get(key)
        if pb is None:
            pb = _lib.Problem.from_buffer_copy(self.pb)
            pb.Nz = b - a
            pb.z_offset = self.z_offset + a
            if self._ts is not None:
                pb.time_scale = self._ts[a].data_ptr()
            self._pb_cache[key] = pb
        return pb

    def _dual_range(self, a, b, slot):
        """Pass A on local planes [a, b); planes just outside come from the slab itself or from the halo buffers."""
        if b <= a:
            return
        u = self._dual_input()
        Nz = self.shape[0]
        lo = u[a - 1] if a > 0 else self._img_lo
        hi = u[b] if b < Nz else self._img_hi
        d = self.scal[slot:slot + 1] if self.track_energy else None
        if self._adj:
            self.ops.cp_dual_adj(self._sub_problem(a, b), u[a:b], self.y[a:b], self.q[a:b], self.lam, self.sigma, d, lo, hi, None, None, self.ws)
            return
        self.ops.cp_dual(self._sub_problem(a, b), u[a:b], self.y[a:b], self.lam, self.sigma, d, lo, hi, self.ws)

    def _primal_range(self, a, b, slot):
        if b <= a:
            return
        Nz = self.shape[0]
        lo = self.y[a - 1, self._zf] if a > 0 else self._fld_lo
        hi = self.y[b, self._zb] if b < Nz else self._fld_hi
        d = self.scal[3 + slot:4 + slot] if self.track_energy else None
        if self._adj:
            self.ops.cp_primal_adj(self._sub_problem(a, b), self.data_term, self._dw[a:b] if self._dw is not None else None, self.y[a:b], self.q[a:b],
                                   self.x[a:b], self.aux[a:b], self.x0[a:b], self.tau, self.theta, d, lo, hi, None, None, self.ws)
            return
        if self._data:
            self.ops.cp_primal_data(self._sub_problem(a, b), self.data_term, self._dw[a:b] if self._dw is not None else None, self.y[a:b], self.x[a:b],
                                    self.aux[a:b], self.x0[a:b], self.tau, self.theta, d, lo, hi, None, None, self.ws)
            return
        c2 = self.theta if self.variant == "rof" else self.sigma_A
        if self.y.dtype == torch.float16:
            self.ops.cp_primal(self.variant, self._sub_problem(a, b), self.y[a:b], self.x[a:b], self.aux[a:b], self.x0[a:b], self.tau, c2, d, lo, hi,
                               self.ws, lam=self.lam)
        else:
            self.ops.cp_primal(self.variant, self._sub_problem(a, b), self.y[a:b], self.x[a:b], self.aux[a:b], self.x0[a:b], self.tau, c2, d, lo,
                               hi, self.ws)

    def _split(self):
        return self.halo is not None and self.z_on and self.overlap and self.shape[0] >= 2

    def _pass_A(self):
        """Dual pass.  Sharded: boundary planes first, their z-components go to the neighbours while the interior
        planes are computed."""
        Nz = self.shape[0]
        if self.halo is None or not self.z_on:
            self._dual_range(0, Nz, 0)
            return
        if self._peer is None:
            if self._pending is None:                  # first iteration (or after a reset): blocking exchange
                self._pending = self._start_image_exchange()
            self.halo.finish(self._pending)
            self._pending = None
        if self.track_energy:
            self.scal[0:3].zero_()
        if self._peer is not None:
            # no exchange: the image halos were stored here by the neighbours' pass B (by one NCCL exchange at start-up),
            # this pass stores the field halos of the neighbours' pass B; the barrier orders the two across ranks
            if self._pending is None:
                self.halo.exchange(*self._image_planes(), self._img_lo, self._img_hi)
                self._peer.barrier()
            self._pending = ()
            d = self.scal[0:1] if self.track_energy else None
            if self._adj:
                self.ops.cp_dual_adj(self.pb, self._dual_input(), self.y, self.q, self.lam, self.sigma, d, self._img_lo, self._img_hi, self._mir_A[0],
                                     self._mir_A[1], self.ws)
            else:
                self.ops.cp_dual_p2p(self.pb, self._dual_input(), self.y, self.lam, self.sigma, d, self._img_lo, self._img_hi, self._mir_A[0],
                                     self._mir_A[1], self.ws)
            self._peer.barrier()
            self._field_req = ()
            return
        if not self._split():
            self._dual_range(0, Nz, 0)
            self._field_req = self._start_field_exchange()
            return
        self._dual_range(0, 1, 0)
        self._dual_range(Nz - 1, Nz, 1)
        self._field_req = self._start_field_exchange()
        self._dual_range(1, Nz - 1, 2)

    def _pass_B(self):
        """Primal pass.  Sharded: boundary planes first, then the new xbar boundary planes travel while the interior is
        updated; they are the halos of the next dual pass."""
        Nz = self.shape[0]
        if self.halo is None or not self.z_on:
            self._primal_range(0, Nz, 0)
            return
        self.halo.finish(self._field_req)
        self._field_req = None
        if self.track_energy:
            self.scal[3:6].zero_()
        if self._peer is not None:
            d = self.scal[3:4] if self.track_energy else None
            if self._adj:
                self.ops.cp_primal_adj(self.pb, self.data_term, self._dw, self.y, self.q, self.x, self.aux, self.x0, self.tau, self.theta, d,
                                       self._fld_lo, self._fld_hi, self._mir_B[0], self._mir_B[1], self.ws)
            elif self._data:
                self.ops.cp_primal_data(self.pb, self.data_term, self._dw, self.y, self.x, self.aux, self.x0, self.tau, self.theta, d, self._fld_lo,
                                        self._fld_hi, self._mir_B[0], self._mir_B[1], self.ws)
            else:
                c2 = self.theta if self.variant == "rof" else self.sigma_A
                self.ops.cp_primal_p2p(self.variant, self.pb, self.y, self.x, self.aux, self.x0, self.tau, c2, d, self._fld_lo, self._fld_hi,
                                       self._mir_B[0], self._mir_B[1], self.ws)
            self._peer.barrier()
            self._pending = ()
            return
        if not self._split():
            self._primal_range(0, Nz, 0)
            self._pending = self._start_image_exchange()
            return
        self._primal_range(0, 1, 0)
        self._primal_range(Nz - 1, Nz, 1)
        self._pending = self._start_image_exchange()
        self._primal_range(1, Nz - 1, 2)

    def capture_graph(self, iterations=1):
        """Capture `iterations` iterations into a CUDA graph; `step(n)` then replays it for every full multiple.
        For small volumes (a 256x256 image is 6 kernels of a few microseconds each) the iteration is launch-bound
        and a graph replay removes the per-launch host cost.  Not available for sharded solvers (the halo exchange
        is issued by NCCL)."""
        if self.halo is not None:
            raise RuntimeError("capture_graph is not supported for distributed solvers")
        self._graph = None
        torch.cuda.synchronize()
        state = (self.x.clone(), self.aux.clone(), self.y.clone(), self.scal.clone(), self.iterations)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            self.step(1)                      # warm-up outside the capture (lazy module loading)
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.step(iterations)             # recorded, not executed
        # undo the warm-up iteration
        self.x.copy_(state[0]); self.aux.copy_(state[1]); self.y.copy_(state[2]); self.scal.copy_(state[3])
        self.iterations = state[4]
        self._graph, self._graph_iters = g, int(iterations)
        self._graph_key = self._graph_state_key()
        return self

    def _graph_state_key(self):
        """What a captured graph has baked in: buffer addresses and the scalar parameters of the passes."""
        return (self.x0.data_ptr(), self.x.data_ptr(), self.aux.data_ptr(), self.y.data_ptr(), self.lam, self.sigma, self.tau, self.theta, self.sigma_A,
                self._dw.data_ptr() if self._dw is not None else 0, self.q.data_ptr() if self.q is not None else 0)

    def step(self, n=1):
        """Run n iterations; returns self."""
        g = getattr(self, "_graph", None)
        if g is not None and self._graph_key != self._graph_state_key():
            # x0 was rebound (step_host_async) or lam / tau / sigma changed (TVProx): the recorded launches are stale
            g = self._graph = None
        if g is not None and not torch.cuda.is_current_stream_capturing():
            while n >= self._graph_iters:
                g.replay()
                self.iterations += self._graph_iters
                n -= self._graph_iters
        for _ in range(n):
            self._pass_A()
            self._pass_B()
            self.iterations += 1
        return self

    def step_host(self, x0_host, x_out_host=None):
        """One iteration against HOST-resident data: upload `x0_host` (numpy array or CPU tensor; pinned memory
        gives full PCIe speed) as the data term, iterate once, download the current x into `x_out_host`, return
        the energy.  State (x, xbar | y_f, y) stays on the device.  Synchronises."""
        src = x0_host if isinstance(x0_host, torch.Tensor) else torch.from_numpy(x0_host)
        self.x0.copy_(src, non_blocking=True)
        self.step(1)
        if x_out_host is not None:
            dst = x_out_host if isinstance(x_out_host, torch.Tensor) else torch.from_numpy(x_out_host)
            dst.copy_(self.x, non_blocking=True)
        return self.energy()

    # ---- pipelined host streaming: PCIe in both directions overlaps the two passes ------------------------
    PIPE_DEPTH = 3      # tickets that may be outstanding: upload of step k+1 | passes of step k | download of step k-1

    def _pipe_init(self):
        if getattr(self, "_pipe", None) is None:
            dev = self.x0.device
            D = self.PIPE_DEPTH
            self._pipe = dict(
                h2d=torch.cuda.Stream(device=dev), d2h=torch.cuda.Stream(device=dev),
                x0=[self.x0] + [torch.empty_like(self.x0) for _ in range(D - 1)],   # data term, one buffer per ticket in flight
                snap=[torch.empty_like(self.x) for _ in range(D)],                  # x snapshots being downloaded
                scal=[torch.zeros(6, dtype=torch.float64, device=dev) for _ in range(D)],
                scal_host=[torch.zeros(6, dtype=torch.float64).pin_memory() for _ in range(D)],
                d2h_done=[None] * D, comp_done=[None] * D, k=0)
        return self._pipe

    def step_host_async(self, x0_host, x_out_host=None):
        """Pipelined form of `step_host`: enqueue upload (copy stream), iteration (current stream) and download
        (second copy stream) and return a ticket at once; `wait(ticket)` returns the energy of that step once its
        download has finished.  Successive calls overlap: while step k computes, the data of step k+1 is being
        uploaded and the image of step k-1 downloaded (PCIe is full duplex), so the steady-state cost per step is
        max(upload, download, compute) instead of their sum.  At most PIPE_DEPTH (3) tickets may be outstanding (wait
        for ticket k-2 before issuing step k+1: with only two in flight the link idles while the passes run); host
        buffers must stay untouched until their ticket has been waited for."""
        p = self._pipe_init()
        k = p["k"]
        slot = k % self.PIPE_DEPTH
        cur = torch.cuda.current_stream()
        src = x0_host if isinstance(x0_host, torch.Tensor) else torch.from_numpy(x0_host)
        # upload into the data buffer last read by step k-DEPTH; a buffer used for the first time may still be read (or be
        # initialised) by work enqueued on the current stream, e.g. the constructor's copies or earlier step() calls
        if p["comp_done"][slot] is not None:
            p["h2d"].wait_event(p["comp_done"][slot])
        else:
            first = torch.cuda.Event()
            first.record(cur)
            p["h2d"].wait_event(first)
        with torch.cuda.stream(p["h2d"]):
            p["x0"][slot].copy_(src, non_blocking=True)
            up = torch.cuda.Event()
            up.record()
        cur.wait_event(up)
        self.x0 = p["x0"][slot]
        self.step(1)
        if p["d2h_done"][slot] is not None:
            cur.wait_event(p["d2h_done"][slot])        # snapshot slot: the download of step k-DEPTH has finished
        p["snap"][slot].copy_(self.x)
        p["scal"][slot].copy_(self.scal)
        done = torch.cuda.Event()
        done.record()
        p["comp_done"][slot] = done
        p["d2h"].wait_event(done)
        with torch.cuda.stream(p["d2h"]):
            if x_out_host is not None:
                dst = x_out_host if isinstance(x_out_host, torch.Tensor) else torch.from_numpy(x_out_host)
                dst.copy_(p["snap"][slot], non_blocking=True)
            p["scal_host"][slot].copy_(p["scal"][slot], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
        p["d2h_done"][slot] = ev
        p["k"] = k + 1
        return (k, slot, ev)

    def wait(self, ticket):
        """Block until the step behind `ticket` has been downloaded; returns its energy (all-reduced when sharded)."""
        k, slot, ev = ticket
        ev.synchronize()
        h = self._pipe["scal_host"][slot]
        s = torch.stack((h[0:3].sum(), h[3:6].sum()))
        if self.halo is not None:
            s = s.to(self.x0.device)
            self.halo.allreduce_sum(s)
        return self._energy_of(*s.tolist())

    def _energy_of(self, l21, fid):
        """Energy from the partial sums of the passes: fid = sum w r^2 (l2) or sum w |r| (l1), r = x - x0."""
        return (0.5 * fid if self.data_term == "l2" else fid) + self.lam * l21

    def energy_async(self):
        """Start the all-reduce of this iteration's energy terms without putting it on the critical path; returns a
        handle for `energy_result`.  Single-GPU solvers just snapshot the scalars."""
        if not self.track_energy:
            raise RuntimeError("energy tracking was disabled")
        s = torch.stack((self.scal[0:3].sum(), self.scal[3:6].sum()))
        work = self.halo.allreduce_sum_async(s) if self.halo is not None else None
        return (s, work)

    def energy_result(self, handle):
        s, work = handle
        if work is not None:
            work.wait()
        return self._energy_of(*s.tolist())

    def energy(self):
        """0.5 |x - x0|^2 + lam L21(D u) of the last iteration over the WHOLE volume (u = the image the dual pass
        differentiated: README.md:157), with the chosen data term in place of 0.5 |x - x0|^2.  One all-reduce of two doubles
        when sharded; synchronises."""
        if not self.track_energy:
            raise RuntimeError("energy tracking was disabled")
        s = torch.stack((self.scal[0:3].sum(), self.scal[3:6].sum()))
        if self.halo is not None:
            self.halo.allreduce_sum(s)
        return self._energy_of(*s.tolist())

    # ---- primal-dual gap, stopping rule, data-term hook (SURVEY 8f items 1-2) ----------------------------
    def _sync_halos_for_diagnostics(self):
        """The halo buffers are about to be reused: retire the exchange that was prefetched for the next pass A."""
        if self.halo is not None and self._pending is not None:
            self.halo.finish(self._pending)
            self._pending = None

    def primal_energy(self):
        """P(x) = 0.5 |x - x0|^2 + lam TV(x) (or the chosen data term + lam TV(x)) at the current iterate, over the whole volume
        (synchronises)."""
        lo = hi = None
        if self.halo is not None and self.z_on:
            self._sync_halos_for_diagnostics()
            to_prev = self.x[0] if self.scheme != "downwind" else None
            to_next = self.x[-1] if self.scheme != "upwind" else None
            self.halo.exchange(to_prev, to_next, self._img_lo, self._img_hi)
            lo, hi = self._img_lo, self._img_hi
        d = torch.zeros(2, dtype=torch.float64, device=self.x.device)
        self.ops.tv_value(self.pb, self.x, d[0:1], lo, hi, self.ws)
        if not self._data:
            d[1] = torch.sum((self.x - self.x0).double() ** 2) if self.x.numel() < (1 << 28) else sum(
                torch.sum((self.x[k] - self.x0[k]).double() ** 2) for k in range(self.shape[0]))
        else:
            for k in range(self.shape[0]):      # plane by plane: no volume-sized float64 temporaries
                r = (self.x[k] - self.x0[k]).double()
                r = r * r if self.data_term == "l2" else r.abs()
                d[1] += torch.sum(r * self._dw[k].double() if self._dw is not None else r)
        if self.halo is not None:
            self.halo.allreduce_sum(d)
        tv, fid = d.tolist()
        return self._energy_of(tv, fid)

    def dual_energy(self):
        """D(y) = 0.5 |x0|^2 - 0.5 |x0 - D^T y|^2 for the feasible dual iterate y (|y_v|_2 <= lam after the projection).
        Other data terms, with s = D^T y:  weighted l2: sum_v (s x0 - s^2 / (2 w));  l1: c <s, x0> with c = min(1, min_v w_v / |s_v|),
        the dual scaled into the feasible set |s_v| <= w_v of the conjugate of the data term (a lower bound of the optimum that
        tends to it).  Where some w_v = 0 the dual objective is unbounded: raises ValueError (solve() then stops on the energy)."""
        if self._data and not self._w_min > 0:
            raise ValueError("the dual energy is unbounded where data_weight = 0: no duality gap (solve() uses the energy change)")
        lo = hi = None
        if self.halo is not None and self.z_on:
            to_prev = self.y[0, self._zb] if self.scheme != "upwind" else None
            to_next = self.y[-1, self._zf] if self.scheme != "downwind" else None
            self.halo.exchange(to_prev, to_next, self._fld_lo, self._fld_hi)
            lo, hi = self._fld_lo, self._fld_hi
        dty = torch.empty_like(self.x)
        if self.y.dtype != self.x.dtype:
            raise NotImplementedError("the duality gap is not available with half-precision dual storage")
        self.ops.adjoint(self.pb, self.y, dty, lo, hi)
        if self._data:
            return self._dual_energy_data(dty)
        d = torch.zeros(2, dtype=torch.float64, device=self.x.device)
        for k in range(self.shape[0]):          # plane by plane: no volume-sized float64 temporaries
            x0k = self.x0[k].double()
            d[0] += torch.sum(x0k * x0k)
            d[1] += torch.sum((x0k - dty[k].double()) ** 2)
        if self.halo is not None:
            self.halo.allreduce_sum(d)
        a, b = d.tolist()
        return 0.5 * a - 0.5 * b

    def _dual_energy_data(self, dty):
        d = torch.zeros(2, dtype=torch.float64, device=self.x.device)    # l2: [sum, -]; l1: [<s, x0>, max |s| / w]
        for k in range(self.shape[0]):
            s, x0k = dty[k].double(), self.x0[k].double()
            w = self._dw[k].double() if self._dw is not None else None
            if self.data_term == "l2":
                d[0] += torch.sum(s * x0k - s * s / (2.0 * w))
            else:
                d[0] += torch.sum(s * x0k)
                d[1] = torch.maximum(d[1], (s.abs() / w if w is not None else s.abs()).max())
        if self.halo is not None:
            self.halo.allreduce_sum(d[0:1])
            self.halo.dist.all_reduce(d[1:2], op=self.halo.dist.ReduceOp.MAX, group=self.halo.group)
        a, m = d.tolist()
        if self.data_term == "l2":
            return a
        return a * (1.0 / m if m > 1.0 else 1.0)

    def gap(self):
        """(primal, dual, primal - dual); the gap is >= 0 and vanishes at the solution.  Raises ValueError when the data weight
        has zeros (see dual_energy)."""
        p, d = self.primal_energy(), self.dual_energy()
        return p, d, p - d

    def solve(self, max_iter=1000, tol=1e-4, check_every=25, callback=None):
        """Iterate until the relative primal-dual gap (P - D) / max(|P|, tiny) <= tol or max_iter is reached.
        Where the data weight has zeros there is no gap (see dual_energy): the run then stops when the primal energy changes by
        at most tol relative to its value between two checks, and `D` is None.  info["criterion"] says which rule was used.
        Returns a dict with the number of iterations and the final energies.  `callback(solver, it, P, D)` is called
        at every check (e.g. to record a convergence curve)."""
        if self._data and not self._w_min > 0:
            return self._solve_by_energy(max_iter, tol, check_every, callback)
        info = dict(iterations=0, converged=False, criterion="gap")
        it = 0
        while it < max_iter:
            n = min(check_every, max_iter - it)
            self.step(n)
            it += n
            p, d, g = self.gap()
            if callback is not None:
                callback(self, it, p, d)
            info.update(iterations=it, primal=p, dual=d, gap=g, relative_gap=g / max(abs(p), 1e-300))
            if g <= tol * max(abs(p), 1e-300):
                info["converged"] = True
                break
        return info

    def _solve_by_energy(self, max_iter, tol, check_every, callback):
        info = dict(iterations=0, converged=False, criterion="energy")
        it, p_prev = 0, None
        while it < max_iter:
            n = min(check_every, max_iter - it)
            self.step(n)
            it += n
            p = self.primal_energy()
            if callback is not None:
                callback(self, it, p, None)
            info.update(iterations=it, primal=p)
            if p_prev is not None:
                info["relative_change"] = abs(p - p_prev) / max(abs(p), 1e-300)
                if info["relative_change"] <= tol:
                    info["converged"] = True
                    break
            p_prev = p
        return info

    def set_data(self, x0, reset_primal=False, reset_dual=False):
        """Data-term hook: replace the data x0 of 0.5|x - x0|^2 (e.g. the gradient step of an outer reconstruction loop,
        x0 = x - t A^T(Ax - b)); the dual variable is kept as a warm start unless reset_dual."""
        src = x0 if isinstance(x0, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(x0))
        self.x0.copy_(src.to(self.x0.dtype), non_blocking=True)
        if reset_primal:
            self.x.copy_(self.x0)
            if self.variant == "rof":
                self.aux.copy_(self.x0)
            self._pending = None
        if reset_dual:
            self.y.zero_()
        return self

    def result(self, return_pytorch_tensor=False):
        return self.x if return_pytorch_tensor else self.x.detach().cpu().numpy()


class TVProx:
    """prox_{lam TV}(v) = argmin_x 0.5|x - v|^2 + lam TV(x) as a reusable operator for outer algorithms (proximal
    gradient / ADMM reconstructions, README.md:3): the dual variable is warm-started from the previous call."""

    def __init__(self, example, lam, scheme="hybrid", n_iter=20, **weights):
        self.solver = CPSolver(example, lam, scheme=scheme, variant="rof", track_energy=False, **weights)
        self.n_iter = int(n_iter)

    def __call__(self, v, lam=None, n_iter=None):
        if lam is not None:
            self.solver.lam = float(lam)
        self.solver.set_data(v, reset_primal=True)
        self.solver.step(self.n_iter if n_iter is None else int(n_iter))
        return self.solver.x


def denoise_tv_chambolle(image, weight=0.1, eps=2e-4, max_num_iter=200, channel_axis=None):
    """Same call as skimage.restoration.denoise_tv_chambolle (the reference's TODO, README.md:260): isotropic TV with
    forward differences (the upwind scheme), objective 0.5|x - image|^2 + weight TV(x), stopped when the energy changes
    by less than eps times its initial value.  2-D or 3-D images; channels (channel_axis) are denoised independently."""
    img = np.asarray(image) if not isinstance(image, torch.Tensor) else image
    was_tensor = isinstance(img, torch.Tensor)
    arr = img if was_tensor else torch.as_tensor(np.ascontiguousarray(img))
    if channel_axis is not None:
        arr = arr.movedim(channel_axis, 0)
        spatial = arr.shape[1:]
        vol = arr.reshape((arr.shape[0],) + tuple(spatial))
        vol = vol[None] if len(spatial) == 2 else vol.movedim(0, 1)        # (1, C, H, W) or (D, C, H, W): channels on the M axis
    else:
        spatial = arr.shape
        vol = arr.reshape((1, 1) + tuple(spatial)) if len(spatial) == 2 else arr.reshape((spatial[0], 1) + tuple(spatial[1:]))
    if len(spatial) not in (2, 3):
        raise ValueError("denoise_tv_chambolle handles 2-D and 3-D images")
    vol = vol.contiguous()
    if vol.dtype not in (torch.float32, torch.float64):
        vol = vol.to(torch.float64)
    solver = CPSolver(vol, weight, scheme="upwind", variant="rof", reg_z_over_reg=1.0, reg_time=0.0)
    e_prev = e_init = None
    for it in range(int(max_num_iter)):
        solver.step(1)
        e = solver.energy()
        if it == 0:
            e_init = e
        elif abs(e_prev - e) < eps * e_init:
            break
        e_prev = e
    out = solver.x
    if channel_axis is not None:
        out = out[0] if len(spatial) == 2 else out.movedim(1, 0)
        out = out.movedim(0, channel_axis)
    else:
        out = out.reshape(tuple(spatial))
    return out if was_tensor else out.cpu().numpy()


def gd_denoise(x0, lam, n_iter, step, scheme="hybrid", return_pytorch_tensor=False, return_losses=False, graph=None, reg_z_over_reg=1.0,
               reg_time=0.0, mask_static=False, factor_reg_static=0, time_weight=None):
    """The README's sub-gradient descent loop (README.md:107-124) with the state resident on the device:
        tv, G = tv_<scheme>(x);  x <- x - step ((x - x0) + lam G);  loss = 0.5 |x - x0|^2 + lam tv
    Two launches per iteration: the single-sweep tv kernel, and one fused kernel for the update and the data term of the
    loss (`pytvb_gd_update`); the partial-sum reductions ride along.  The whole loop is captured into one CUDA graph and
    replayed (graph=None: when the volume is small enough for launch overhead to matter, < 2^22 voxels), so a small image
    costs a few microseconds per iteration instead of a host round trip per launch.  Returns x (and the loss history,
    one entry per iteration, read back once at the end)."""
    x0d, was_tensor = _dev.to_device(x0)
    if x0d.data_ptr() == (x0.data_ptr() if isinstance(x0, torch.Tensor) else 0):
        x0d = x0d.clone()
    shape = _dev.image_shape(x0d)
    lib = _lib.lib()
    n_iter = int(n_iter)
    ms = _dev.mask_static_to_device(mask_static, shape[2], shape[3])
    ts = _dev.time_scale_to_device(time_weight, shape, x0d)
    pb = _dev.problem(scheme, x0d, shape, reg_z_over_reg, reg_time, factor_reg_static, ms, ts=ts)
    x = x0d.clone()
    G = torch.empty_like(x)
    ws_r = _dev.reduce_workspace(pb, x.device)
    ws_t = torch.empty(lib.pytvb_tv_workspace_bytes(ctypes.byref(pb)), dtype=torch.uint8, device=x.device)
    tvs = torch.zeros(max(n_iter, 1), dtype=torch.float64, device=x.device)
    fids = torch.zeros(max(n_iter, 1), dtype=torch.float64, device=x.device)

    def iteration(it):
        st = _dev.stream_ptr()
        _lib.check(lib.pytvb_tv(ctypes.byref(pb), _dev.ptr(x), _dev.ptr(G), None, _dev.ptr(tvs[it:it + 1]), None, None, _dev.ptr(ws_r), _dev.ptr(ws_t), st))
        _lib.check(lib.pytvb_gd_update(ctypes.byref(pb), _dev.ptr(x), _dev.ptr(x0d), _dev.ptr(G), float(step), float(lam),
                                       _dev.ptr(fids[it:it + 1]) if return_losses else None, _dev.ptr(ws_r), st))

    if graph is None:
        graph = x.numel() < (1 << 22) and n_iter >= 8
    if graph and n_iter > 0:
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            iteration(0)                      # warm-up outside the capture (lazy module loading, function attributes)
        torch.cuda.current_stream().wait_stream(side)
        x.copy_(x0d)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for it in range(n_iter):
                iteration(it)
        g.replay()
    else:
        for it in range(n_iter):
            iteration(it)
    out = x if (return_pytorch_tensor or was_tensor) else x.cpu().numpy()
    if return_losses:
        return out, (0.5 * fids[:n_iter] + float(lam) * tvs[:n_iter]).cpu().numpy()
    return out


def cp_denoise(x0, lam, n_iter, scheme="hybrid", variant="rof", return_pytorch_tensor=False, return_energy=False, **kw):
    """Denoise `x0` with n_iter fused Chambolle-Pock iterations; see CPSolver for the keyword arguments (e.g. data_term="l1" for
    impulse noise, data_weight for per-voxel confidence or missing data)."""
    solver = CPSolver(x0, lam, scheme=scheme, variant=variant, track_energy=return_energy, **kw)
    solver.step(int(n_iter))
    if isinstance(x0, torch.Tensor):
        return_pytorch_tensor = True
    out = solver.result(return_pytorch_tensor)
    return (out, solver.energy()) if return_energy else out

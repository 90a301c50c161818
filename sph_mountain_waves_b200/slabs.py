"""x-slab domain decomposition of one particle set over the GPUs of a box
(one process per GPU; SURVEY.md §8e — the reference has no distributed path).

Rank g owns the cell columns [X_g, X_{g+1}) of the global neighbour grid and keeps
two ghost columns on each side.  Every step ONE halo exchange (torch.distributed
send/recv: NCCL over NVLink on the GPUs, gloo in the CPU tests) moves, between
x-adjacent ranks only,
  * migrants — particles whose cell column left the slab (the carried state), and
  * ghosts   — copies of the particles in the two outermost owned columns.
Ghost density is recomputed locally (the second ghost column makes the first one's
sums complete), so there is no second exchange before the force pass, and because
neighbours are visited in (cell, GLOBAL particle index) order the FP64 sums are
bit-identical for any number of ranks.

The transport (`exchange`) and the partition planning (`split_columns`, `plan_slab`,
`global_indices`) are backend-neutral host logic; what packs, unpacks and computes is a
backend: `LibSlabBackend` (libsphmw, CUDA) in production, an oracle-driven one in
tests/test_slabs_gloo.py.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import Callable, List, Optional, Tuple

import numpy as np

from . import _capi, cases
from ._capi import check
from .schemes import wcsph_perturbed_witch as wpw

GHOST_COLS = 2
GHOST3_FLAG = 256  # SPHMW_FLAG_GHOST3: three ghost columns per side (the Hopkins schemes)
RECORD = 13  # the base record: x0 x1 x2 v0 v1 v2 m h rho rho_p type idx kind (csrc/halo_record.cuh)
KIND_MIGRANT, KIND_GHOST = 0.0, 1.0


# ----------------------------------------------------------------------------- planning
def split_columns(ncols: int, world: int, weights: Optional[np.ndarray] = None,
                  ghost: int = GHOST_COLS) -> List[Tuple[int, int]]:
    """Column ranges [lo, hi) per rank; equal widths for a uniform lattice, or
    balanced by per-column particle counts when `weights` is given."""
    if weights is None:
        edges = [round(ncols * r / world) for r in range(world + 1)]
    else:
        c = np.concatenate([[0], np.cumsum(weights)])
        target = c[-1] * np.arange(world + 1) / world
        edges = [int(np.searchsorted(c, t, side="left")) for t in target]
        edges[0], edges[-1] = 0, ncols
    for r in range(world):
        if edges[r + 1] - edges[r] < 2 * ghost:
            raise ValueError(f"a slab must own at least {2 * ghost} cell columns")
    return [(edges[r], edges[r + 1]) for r in range(world)]


def key_tables(box_min, box_max, h: float):
    """structs.jl:66-68"""
    phase = [int(math.floor(box_min[a] / h)) for a in range(3)]
    lim = [int(math.floor(box_max[a] / h)) - phase[a] + 1 for a in range(3)]
    return phase, lim


def column_of(x0: np.ndarray, h: float, phase0: int) -> np.ndarray:
    """global cell column, with the reference's arithmetic (structs.jl:99)"""
    return np.floor(x0 / h).astype(np.int64) - phase0


@dataclass
class SlabPlan:
    rank: int
    world: int
    lo: int
    hi: int
    phase0: int
    ncols: int
    h: float

    @property
    def has_left(self):
        return self.rank > 0

    @property
    def has_right(self):
        return self.rank < self.world - 1

    def x_clip(self, margin: float):
        """a slightly generous x-interval containing every owned lattice site"""
        xa = -1e300 if not self.has_left else (self.phase0 + self.lo) * self.h - margin
        xb = 1e300 if not self.has_right else (self.phase0 + self.hi) * self.h + margin
        return xa, xb

    def owns(self, x0: np.ndarray) -> np.ndarray:
        # a particle beyond the box along x still belongs to somebody — the outermost rank — until the
        # first create_cell_list! removes it (core.jl:60-81: its slot is refilled from the end of
        # sys.particles, which renumbers survivors)
        c = np.clip(column_of(x0, self.h, self.phase0), 0, self.ncols - 1)
        return (c >= self.lo) & (c < self.hi)


def plan_slab(box_min, box_max, h: float, rank: int, world: int, ghost: int = GHOST_COLS) -> SlabPlan:
    phase, lim = key_tables(box_min, box_max, h)
    lo, hi = split_columns(lim[0], world, ghost=ghost)[rank]
    return SlabPlan(rank, world, lo, hi, phase[0], lim[0], h)


def global_indices(group_counts_all: np.ndarray, rank: int) -> np.ndarray:
    """Reference particle index (0-based) of this rank's particles.  The reference fills
    sys.particles group by group (fluid, walls, mountain — wcsph_perturbed_witch.jl:162-164)
    and plane by plane along x within a group; ranks own increasing x-ranges, so the index
    of a local particle = all earlier groups + the same group on lower ranks + local order.
    `group_counts_all[r, g]` = number of particles of group g owned by rank r."""
    gc = np.asarray(group_counts_all, dtype=np.int64)
    group_start = np.concatenate([[0], np.cumsum(gc.sum(axis=0))])
    out = []
    for g in range(gc.shape[1]):
        first = group_start[g] + gc[:rank, g].sum()
        out.append(first + np.arange(gc[rank, g], dtype=np.int64))
    return np.concatenate(out) if out else np.zeros(0, dtype=np.int64)


# ----------------------------------------------------------------------------- transport
def exchange(plan: SlabPlan, send_left, send_right, migr_left: int, migr_right: int, empty: Callable):
    """Move halo records to the x-adjacent ranks.  `send_*` are (count, width) float64
    tensors (or None when there is no neighbour); `empty(n)` allocates a receive tensor on
    the right device.  Returns ((recv_from_left, n_migrants), (recv_from_right, n_migrants))."""
    import torch
    import torch.distributed as dist

    if plan.world == 1:
        return (None, 0), (None, 0)
    dev = send_left.device if send_left is not None else send_right.device
    peers = []
    if plan.has_left:
        peers.append((plan.rank - 1, send_left, migr_left))
    if plan.has_right:
        peers.append((plan.rank + 1, send_right, migr_right))
    # 1. how many records / migrants are coming
    heads_out = [torch.tensor([len(s), m], dtype=torch.int64, device=dev) for _, s, m in peers]
    heads_in = [torch.zeros(2, dtype=torch.int64, device=dev) for _ in peers]
    ops = []
    for (peer, _, _), ho, hi_ in zip(peers, heads_out, heads_in):
        ops.append(dist.P2POp(dist.isend, ho, peer))
        ops.append(dist.P2POp(dist.irecv, hi_, peer))
    for w in dist.batch_isend_irecv(ops):
        w.wait()
    heads = [h.tolist() for h in heads_in]
    # 2. the records
    recv = [empty(int(h[0])) for h in heads]
    ops = []
    for (peer, s, _), r in zip(peers, recv):
        if len(s):
            ops.append(dist.P2POp(dist.isend, s, peer))
        if len(r):
            ops.append(dist.P2POp(dist.irecv, r, peer))
    if ops:
        for w in dist.batch_isend_irecv(ops):
            w.wait()
    out = {peer: (r, int(h[1])) for (peer, _, _), r, h in zip(peers, recv, heads)}
    return out.get(plan.rank - 1, (None, 0)), out.get(plan.rank + 1, (None, 0))


# ----------------------------------------------------------------------------- CUDA backend
class LibSlabBackend:
    """pack / unpack / compute through libsphmw on this rank's GPU"""

    def __init__(self, sys, plan: SlabPlan, cap_records: int):
        import torch
        self.sys, self.plan = sys, plan
        self.cap = int(cap_records)
        self.dev = torch.device("cuda", sys.device)
        self._width = None
        self.buf_l = self.buf_r = None
        self.lost = 0

    @property
    def width(self) -> int:
        """doubles per record: RECORD, or more for a context that carries extra state (the adiabatic flow
        driver's S, P, T, theta).  Asked when first needed — after the particles are on the device — and
        fixed by the library from then on."""
        if self._width is None:
            self.sys._flush()
            w = C.c_int32()
            check(_capi.lib().sphmw_halo_record_width(self.sys.ctx, C.byref(w)))
            self._width = w.value
        return self._width

    def _buffers(self):
        import torch
        if self.buf_l is None and self.buf_r is None:
            shape = (self.cap, self.width)
            self.buf_l = torch.empty(shape, dtype=torch.float64, device=self.dev) if self.plan.has_left else None
            self.buf_r = torch.empty(shape, dtype=torch.float64, device=self.dev) if self.plan.has_right else None

    def empty(self, n: int):
        import torch
        return torch.empty((n, self.width), dtype=torch.float64, device=self.dev)

    @property
    def scheme(self) -> bytes:
        """the scheme this context steps: "wcsph", "hopkins"/"hopkins_full"/"hopkins_total" (three ghost
        columns) or "aflow" (the adiabatic flow driver; a step in which an INFLOW particle converts needs the
        library transport with the open box)"""
        s = getattr(self.sys.T, "scheme", "wcsph")
        return s.encode() if s in ("hopkins", "hopkins_full", "hopkins_total", "aflow") else b"wcsph"

    def pre(self):
        check(_capi.lib().sphmw_step_phase(self.sys.ctx, self.scheme, 0))

    def post(self):
        check(_capi.lib().sphmw_step_phase(self.sys.ctx, self.scheme, 1))

    def build(self):
        self.sys.create_cell_list(want_count=False)

    def pack(self):
        self._buffers()
        counts = (C.c_int64 * 5)()
        pl = C.c_void_p(self.buf_l.data_ptr()) if self.buf_l is not None else None
        pr = C.c_void_p(self.buf_r.data_ptr()) if self.buf_r is not None else None
        check(_capi.lib().sphmw_halo_pack(self.sys.ctx, pl, pr, self.cap, counts))
        self.lost += counts[4]
        sl = self.buf_l[:counts[0]] if self.buf_l is not None else None
        sr = self.buf_r[:counts[1]] if self.buf_r is not None else None
        return sl, sr, int(counts[2]), int(counts[3])

    def unpack(self, recv, n_migrants: int):
        if recv is None or len(recv) == 0:
            return
        check(_capi.lib().sphmw_halo_unpack(self.sys.ctx, C.c_void_p(recv.data_ptr()), len(recv), n_migrants))

    # ---- overlapped step (include/sphmw.h: step_phase 2/3, halo_pack_begin/finish) ----------
    @property
    def can_overlap(self) -> bool:
        # CELL_PAIRS kernels take one column range only; the overlapped schedule is the fused WCSPH
        # step's, laid out for two ghost columns
        return not (self.sys._flags & (2 | GHOST3_FLAG)) and self.scheme == b"wcsph"

    def overlap_enqueue(self):
        """finish the current step and start the next one: edge columns first (force, kick,
        drift, pack), then the interior — everything is only enqueued"""
        lib = _capi.lib()
        self._buffers()
        check(lib.sphmw_step_phase(self.sys.ctx, b"wcsph", 2))
        pl = C.c_void_p(self.buf_l.data_ptr()) if self.buf_l is not None else None
        pr = C.c_void_p(self.buf_r.data_ptr()) if self.buf_r is not None else None
        check(lib.sphmw_halo_pack_begin(self.sys.ctx, pl, pr, self.cap))
        check(lib.sphmw_step_phase(self.sys.ctx, b"wcsph", 3))

    def pack_finish(self):
        counts = (C.c_int64 * 5)()
        check(_capi.lib().sphmw_halo_pack_finish(self.sys.ctx, self.cap, counts))
        self.lost += counts[4]
        sl = self.buf_l[:counts[0]] if self.buf_l is not None else None
        sr = self.buf_r[:counts[1]] if self.buf_r is not None else None
        return sl, sr, int(counts[2]), int(counts[3])

    def pack_wait(self, cuda_stream: int):
        check(_capi.lib().sphmw_halo_pack_wait(self.sys.ctx, C.c_void_p(cuda_stream)))

    def counts(self):
        a, b = C.c_int64(), C.c_int64()
        check(_capi.lib().sphmw_slab_counts(self.sys.ctx, C.byref(a), C.byref(b)))
        return a.value, b.value


# ----------------------------------------------------------------------------- the run
class SlabRun:
    """One rank's share of a mountain-wave run (world == 1: the whole domain, no halo)."""

    def __init__(self, sys, plan: Optional[SlabPlan], n_global: int, backend=None,
                 export=("v", "ρ", "P", "θ", "T", "type")):
        self.sys = sys
        self.plan = plan
        self.backend = backend
        self.n_global = n_global
        self.export = export
        self.case_info = {}
        self._pinned = None
        self._owned_host = None
        self._lib_comm = False
        self._in_flight = None

    @property
    def world(self):
        return 1 if self.plan is None else self.plan.world

    # ------------------------------------------------------------------ construction
    @classmethod
    def bell_hill_3d(cls, nx, ny, nz, rank=0, world=1, device=0, stream=None, flags: int = 0,
                     device_gen: bool = False, **kw):
        """BASELINE config 4/5 split into x-slabs; every rank generates only its own lattice
        planes (on the host, or on the GPU with `device_gen`), global particle indices are agreed
        on by an all-gather of group sizes."""
        if device_gen:
            return cls._bell_hill_3d_device(nx, ny, nz, rank, world, device, stream, flags, **kw)
        if world == 1:
            case = cases.bell_hill_3d(nx, ny, nz, lean=True, **kw)
            sys = cases.to_system(case, device=device, stream=stream, flags=flags)
            sys._flush()
            run = cls(sys, None, case.n)
            run.case_info = case.info
            return run
        import torch
        import torch.distributed as dist
        # the global bounding box is a function of the constants alone
        k = wpw.Constants(n_y=float(ny), dim=3, grid="cubic")
        k.dom_length, k.dom_width = nx * k.dr, nz * k.dr
        w = k.bc_width
        box_min = (-k.dom_length / 2.0 - w, 0.0 - w, -k.dom_width / 2.0 - w)
        box_max = (k.dom_length / 2.0 + w, k.dom_height + w, k.dom_width / 2.0 + w)
        plan = plan_slab(box_min, box_max, k.h0, rank, world)
        case = cases.bell_hill_3d(nx, ny, nz, lean=True, clip=plan.x_clip(2 * k.dr), **kw)
        assert tuple(case.box_min) == box_min and tuple(case.box_max) == box_max
        keep = plan.owns(case.fields["x"][:, 0])
        gc = np.asarray(case.info["group_counts"], dtype=np.int64)
        edges = np.concatenate([[0], np.cumsum(gc)])
        kept = np.array([int(keep[edges[g]:edges[g + 1]].sum()) for g in range(len(gc))], dtype=np.int64)
        case.fields = {f: a[keep] for f, a in case.fields.items()}
        t = torch.tensor(kept, dtype=torch.int64, device=torch.device("cuda", device))
        allc = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allc, t)
        allc = np.stack([a.cpu().numpy() for a in allc])
        gidx = global_indices(allc, rank)
        n_global = int(allc.sum())
        n_own = case.n
        ghost_est = int(n_own * 2 * GHOST_COLS / max(1, plan.hi - plan.lo) * 1.5) + 4096
        sys = cases.to_system(case, device=device, stream=stream, slab=(plan.lo, plan.hi),
                              capacity=int(n_own * 1.1) + 2 * ghost_est, flags=flags)
        sys._flush()
        check(_capi.lib().sphmw_set_index(sys.ctx, _capi.ptr(np.ascontiguousarray(gidx)), n_own))
        run = cls(sys, plan, n_global, LibSlabBackend(sys, plan, ghost_est))
        run.case_info = case.info
        run._owned_host = (case.fields, gidx)
        return run

    @classmethod
    def _bell_hill_3d_device(cls, nx, ny, nz, rank, world, device, stream, flags, h_m=100.0, a=10e3, U=20.0):
        """the same particle set, generated by sphmw_generate_mountain_wave on each rank's GPU"""
        k = wpw.Constants(n_y=float(ny), h_m=h_m, a=a, U=U, dim=3, grid="cubic",
                          mountain_type=wpw.MOUNTAIN if h_m else wpw.FLUID)
        k.dom_length, k.dom_width = nx * k.dr, nz * k.dr
        info = dict(dr=k.dr, dt=k.dt, frame_every=int(round(k.dt_frame / k.dt)))
        if world == 1:
            sys = wpw.make_system_on_device(k, device=device, stream=stream, flags=flags)
            run = cls(sys, None, sys.n_device)
            run.case_info = info
            return run
        import torch
        import torch.distributed as dist
        w = k.bc_width
        box_min = (-k.dom_length / 2.0 - w, 0.0 - w, -k.dom_width / 2.0 - w)
        box_max = (k.dom_length / 2.0 + w, k.dom_height + w, k.dom_width / 2.0 + w)
        plan = plan_slab(box_min, box_max, k.h0, rank, world)
        sites = (nx + 14) * (ny + 14) * (nz + 14)
        own_est = int(sites * (plan.hi - plan.lo + 1) / plan.ncols) + 65536
        ghost_est = int(own_est * 2 * GHOST_COLS / max(1, plan.hi - plan.lo) * 1.5) + 4096
        sys = wpw.make_system_on_device(k, capacity=int(own_est * 1.1) + 2 * ghost_est, device=device,
                                        stream=stream, flags=flags, slab=(plan.lo, plan.hi))
        n_own = sys.n_device
        t = torch.tensor(list(sys.group_counts), dtype=torch.int64, device=torch.device("cuda", device))
        allc = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allc, t)
        allc = np.stack([a_.cpu().numpy() for a_ in allc])
        gidx = global_indices(allc, rank)
        check(_capi.lib().sphmw_set_index(sys.ctx, _capi.ptr(np.ascontiguousarray(gidx)), n_own))
        run = cls(sys, plan, int(allc.sum()), LibSlabBackend(sys, plan, ghost_est))
        run.case_info = info
        # host copies of the carried state for the end-to-end cycle (read back once)
        from .system import FIELD_NCOMP, canonical
        host = {}
        for f in wpw.CORE_FIELDS:
            nc = FIELD_NCOMP[canonical(f)]
            buf = np.empty((nc, n_own) if nc == 3 else n_own, dtype=np.float64)
            check(_capi.lib().sphmw_download_raw(sys.ctx, canonical(f).encode(), _capi.ptr(buf), n_own, nc))
            host[canonical(f)] = np.ascontiguousarray(buf.T) if nc == 3 else buf
        run._owned_host = (host, gidx)
        return run

    @classmethod
    def whole(cls, case, device=0, stream=None, flags: int = 0):
        """any case on one GPU (no slabs)"""
        sys = cases.to_system(case, device=device, stream=stream, flags=flags)
        sys._flush()
        run = cls(sys, None, case.n)
        run.case_info = dict(case.info)
        return run

    @classmethod
    def from_global_case(cls, case, rank: int, world: int, device: int = 0, stream=None, flags: int = 0):
        """Slice a whole (small) case held on the host: reference indices are the positions in
        `case.fields`.  Used by tests and by single-process multi-context runs.  A Hopkins case gets
        three ghost columns per side (SPHMW_FLAG_GHOST3)."""
        ghost = 3 if case.scheme in ("hopkins", "hopkins_full", "hopkins_total") else GHOST_COLS
        if ghost == 3:
            flags |= GHOST3_FLAG
        plan = plan_slab(case.box_min, case.box_max, case.h, rank, world, ghost=ghost)
        own = plan.owns(case.fields["x"][:, 0])
        gidx = np.nonzero(own)[0].astype(np.int64)
        sub = cases.Case(case.name, case.scheme, case.dim, case.box_min, case.box_max, case.h,
                         case.params, {f: a[own] for f, a in case.fields.items()}, dict(case.info))
        n_own = sub.n
        ghost_est = int(n_own * 2 * ghost / max(1, plan.hi - plan.lo) * 2.0) + 4096
        sys = cases.to_system(sub, device=device, stream=stream, slab=(plan.lo, plan.hi),
                              capacity=int(n_own * 1.2) + 2 * ghost_est, flags=flags)
        sys._flush()
        if n_own:
            check(_capi.lib().sphmw_set_index(sys.ctx, _capi.ptr(np.ascontiguousarray(gidx)), n_own))
        run = cls(sys, plan, case.n, LibSlabBackend(sys, plan, ghost_est))
        run.case_info = dict(case.info)
        run._owned_host = (sub.fields, gidx)
        return run

    # ------------------------------------------------------------------ stepping
    @property
    def n_owned(self) -> int:
        return self.sys.n_device if self.backend is None else self.backend.counts()[1]

    @property
    def n_resident(self) -> int:
        return self.sys.n_device

    def _halo(self):
        b = self.backend
        sl, sr, ml, mr = b.pack()
        (rl, nml), (rr, nmr) = exchange(self.plan, sl, sr, ml, mr, b.empty)
        self._wait_for_records(b)
        b.unpack(rl, nml)
        b.unpack(rr, nmr)
        self._in_flight = (rl, rr)   # keep the receive tensors until the next exchange: unpack is asynchronous

    @staticmethod
    def _wait_for_records(b):
        """The receives complete on torch's current stream, the unpack kernel runs on the context's
        own stream: the host waits for the former before it queues the latter."""
        import torch
        if getattr(b, "dev", None) is not None:
            torch.cuda.current_stream(b.dev).synchronize()

    # ------------------------------------------------------------------ transport inside the library
    def use_library_transport(self, halo_capacity: Optional[int] = None, open_box: bool = False):
        """Hand the halo exchange to libsphmw (csrc/slab_comm.cu: ncclSend/ncclRecv on its own
        stream, driven by sphmw_step / sphmw_create_cell_list).  Collective over torch.distributed:
        rank 0 creates the NCCL id, everybody joins."""
        import torch
        import torch.distributed as dist
        if self.backend is None or self.plan.world == 1 or self._lib_comm:
            return self
        lib = _capi.lib()
        dev = torch.device("cuda", self.sys.device)
        ident = torch.zeros(128, dtype=torch.uint8, device=dev)
        if self.plan.rank == 0:
            buf = (C.c_ubyte * 128)()
            check(lib.sphmw_comm_unique_id(buf))
            ident = torch.tensor(list(buf), dtype=torch.uint8, device=dev)
        dist.broadcast(ident, 0)
        cap = torch.tensor([int(halo_capacity or self.backend.cap)], dtype=torch.int64, device=dev)
        dist.all_reduce(cap, op=dist.ReduceOp.MAX)   # the same capacity on every rank
        raw = bytes(ident.cpu().tolist())
        check(lib.sphmw_comm_init(self.sys.ctx, self.plan.rank, self.plan.world, raw, int(cap.item())))
        if open_box:
            # particles may leave the global box: the library replays the reference's swap-from-end
            # renumbering (core.jl:72-81) across ranks after every exchange
            check(lib.sphmw_comm_open_box(self.sys.ctx, 1))
        self._lib_comm = True
        return self

    def comm_info(self) -> dict:
        out = (C.c_int64 * 6)()
        check(_capi.lib().sphmw_comm_info(self.sys.ctx, out))
        return {"world": out[0], "exchanges": out[1], "renegotiations": out[2], "message_rows": out[3],
                "lost": out[4], "capacity": out[5]}

    def create_cell_list(self):
        """≙ create_cell_list!(sys): (halo exchange +) sort.  Ghosts exist from here on."""
        if self.backend is None:
            self.sys.create_cell_list()
        elif self._lib_comm:
            self.sys.create_cell_list(want_count=False)   # the library exchanges the halo itself
        else:
            self._halo()
            self.backend.build()

    def step(self, nsteps: int, overlap: bool = True):
        """nsteps of verlet_step!.  On slabs all but the last step run the overlapped schedule:
        the halo records of step k+1 travel (on a second CUDA stream) while the interior columns
        of step k are in the force pass.  Same bits either way."""
        b = self.backend
        if b is None:
            self.sys.step(nsteps)
            return
        if nsteps <= 0:
            return
        if self._lib_comm:
            if overlap:
                self.sys.step(nsteps)
            else:
                for _ in range(nsteps):
                    self.sys.step(1)      # single steps take the plain schedule
            return
        if not (overlap and nsteps > 1 and getattr(b, "can_overlap", False)):
            for _ in range(nsteps):
                b.pre()
                self._halo()
                b.post()
            return
        import torch
        if getattr(self, "_comm_stream", None) is None:
            self._comm_stream = torch.cuda.Stream(b.dev)
        comm = self._comm_stream
        b.pre()
        self._halo()
        for _ in range(nsteps - 1):
            b.overlap_enqueue()
            sl, sr, ml, mr = b.pack_finish()       # the host waits for the edge columns only
            with torch.cuda.stream(comm):          # transport beside the interior force pass
                b.pack_wait(comm.cuda_stream)
                (rl, nml), (rr, nmr) = exchange(self.plan, sl, sr, ml, mr, b.empty)
            comm.synchronize()                     # records have arrived (and the sends have left)
            b.unpack(rl, nml)
            b.unpack(rr, nmr)
            self._in_flight = (rl, rr)
        b.post()

    # ------------------------------------------------------------------ read-back (tests)
    def owned_fields(self, names=("x", "v", "rho", "h")):
        """(global indices, {field: array}) of the particles this rank owns"""
        from .system import FIELD_NCOMP, canonical
        lib = _capi.lib()
        n = self.sys.n_device
        if self.backend is None:
            return np.arange(n, dtype=np.int64), {f: self.sys.field(f) for f in names}
        gidx = np.empty(n, dtype=np.int64)
        tag = np.empty(n, dtype=np.int32)
        check(lib.sphmw_download_index(self.sys.ctx, _capi.ptr(gidx), _capi.ptr(tag), n))
        own = tag == 0
        out = {}
        for f in names:
            nc = FIELD_NCOMP[canonical(f)]
            buf = np.empty((nc, n) if nc == 3 else n, dtype=np.float64)
            check(lib.sphmw_download_raw(self.sys.ctx, canonical(f).encode(), _capi.ptr(buf), n, nc))
            a = np.ascontiguousarray(buf.T) if nc == 3 else buf
            out[f] = a[own]
        return gidx[own], out

    # ------------------------------------------------------------------ end to end
    def e2e_cycle(self, cycles: int, barrier: Callable[[], None]):
        """Through the public API with HOST buffers: upload the carried state from pinned
        host memory, run one output interval of steps (the reference saves a frame every
        Int(round(dt_frame/dt)) steps, wcsph_perturbed_witch.jl:375), download the exported
        fields (x + export_vars, :18) back to pinned host memory."""
        import time

        import torch
        from .system import FIELD_NCOMP, canonical
        sys = self.sys
        lib = _capi.lib()
        carried = list(wpw.CORE_FIELDS)
        out_fields = sorted(set(self.export) | {"x"})
        every = int(self.case_info.get("frame_every", 8))
        slab = self.backend is not None
        if self._pinned is None:
            self._pinned = {}
            if slab:
                host, gidx = self._owned_host
                n0 = len(gidx)
                for f in carried:
                    a = host[canonical(f)]
                    t = torch.empty(a.T.shape if a.ndim == 2 else a.shape, dtype=torch.float64, pin_memory=True)
                    t.copy_(torch.from_numpy(np.ascontiguousarray(a.T if a.ndim == 2 else a)))
                    self._pinned[f] = t
                # global indices travel with every batch: pinned, staged by sphmw_upload_index_async
                self._gidx = torch.empty((n0,), dtype=torch.int64, pin_memory=True)
                self._gidx.copy_(torch.from_numpy(np.ascontiguousarray(gidx, dtype=np.int64)))
            else:
                n0 = sys.n_device
                for f in carried:
                    nc = FIELD_NCOMP[canonical(f)]
                    self._pinned[f] = torch.empty((nc, n0) if nc == 3 else (n0,), dtype=torch.float64,
                                                  pin_memory=True)
                    sys.download_ptr(f, self._pinned[f].data_ptr(), n0)
            self._n0 = n0
            cap = int(n0 * 1.5) + 65536
            for f in out_fields:
                nc = FIELD_NCOMP[canonical(f)]
                self._pinned["out:" + f] = torch.empty((nc * cap,), dtype=torch.float64, pin_memory=True)
        n0 = self._n0
        h2d = sum(self._pinned[f].numel() * 8 for f in carried) + (n0 * 8 if slab else 0)
        d2h = 0
        names = (C.c_char_p * len(out_fields))(*[canonical(f).encode() for f in out_fields])
        comps = sum(FIELD_NCOMP[canonical(f)] for f in out_fields)

        def prefetch():
            # the next cycle's inputs travel on the library's copy stream while this cycle steps
            for f in carried:
                check(lib.sphmw_upload_async(sys.ctx, canonical(f).encode(), C.c_void_p(self._pinned[f].data_ptr()),
                                             n0, FIELD_NCOMP[canonical(f)]))
            if slab:
                check(lib.sphmw_upload_index_async(sys.ctx, C.c_void_p(self._gidx.data_ptr()), n0))

        def wait(slot):
            ptrs = (C.c_void_p * len(out_fields))()
            n = C.c_int64()
            check(lib.sphmw_frame_wait(sys.ctx, slot, ptrs, len(out_fields), C.byref(n)))
            return n.value

        def run_cycles(count):
            moved = 0
            prefetch()
            pending = None
            for k in range(count):
                check(lib.sphmw_upload_commit(sys.ctx))       # staged fields (+ indices) -> particle state, no host wait
                if k + 1 < count:
                    prefetch()
                self.create_cell_list()
                self.step(every)
                slot = C.c_int32()
                check(lib.sphmw_frame_capture(sys.ctx, names, len(out_fields), C.byref(slot)))   # D2H beside the next cycle
                if pending is not None:
                    moved += comps * wait(pending) * 8
                pending = slot.value
            moved += comps * wait(pending) * 8
            return moved

        if not getattr(self, "_e2e_warm", False):
            run_cycles(2)          # untimed: the library allocates its pinned snapshot and staging buffers
            self._e2e_warm = True
        barrier()
        t0 = time.perf_counter()
        d2h = run_cycles(cycles)
        barrier()
        dt = time.perf_counter() - t0
        return {"seconds": dt, "steps": cycles * every, "h2d_bytes": h2d * cycles, "d2h_bytes": d2h,
                "what": f"{cycles} x (upload {len(carried)} carried fields from pinned host [sphmw_upload_async/commit: "
                        f"the next cycle's copy runs beside this cycle's steps], create_cell_list, {every} steps = one "
                        f"frame interval, x + {len(self.export)} export fields to pinned host [sphmw_frame_capture/wait: "
                        f"device snapshot, copy beside the next cycle])"}


class LocalCluster:
    """All ranks of a slab decomposition driven in lockstep by ONE process (loop-back
    transport: the records are handed over as device tensors).  The kernels of different
    contexts never wait on one another, so running them back to back on one GPU — or on
    several GPUs of the box from a single host thread — is safe."""

    def __init__(self, runs: List[SlabRun]):
        self.runs = runs

    def _halo(self):
        self._handover([r.backend.pack() for r in self.runs])

    def create_cell_list(self):
        self._halo()
        for r in self.runs:
            r.backend.build()

    def _handover(self, packs):
        import torch
        keep = []
        for r, run in enumerate(self.runs):
            dev = run.backend.dev
            inbox = []
            if r > 0:
                sl, sr, ml, mr = packs[r - 1]
                inbox.append((sr.to(dev), mr))          # my left neighbour's right-going records
            if r < len(self.runs) - 1:
                sl, sr, ml, mr = packs[r + 1]
                inbox.append((sl.to(dev), ml))          # my right neighbour's left-going records
            # the copies run on torch's current stream, the unpack on the context's own
            torch.cuda.current_stream(dev).synchronize()
            for rec, migr in inbox:
                run.backend.unpack(rec, migr)
            keep.append(inbox)
        self._in_flight = keep   # alive until the next handover: unpack is asynchronous

    def step(self, nsteps: int, overlap: bool = True):
        if nsteps <= 0:
            return
        if not (overlap and nsteps > 1 and all(r.backend.can_overlap for r in self.runs)):
            for _ in range(nsteps):
                for r in self.runs:
                    r.backend.pre()
                self._halo()
                for r in self.runs:
                    r.backend.post()
            return
        for r in self.runs:
            r.backend.pre()
        self._halo()
        for _ in range(nsteps - 1):
            for r in self.runs:
                r.backend.overlap_enqueue()
            self._handover([r.backend.pack_finish() for r in self.runs])
            for r in self.runs:
                r.sys.sync()   # a sender's next pack must not overtake the receiver's unpack
        for r in self.runs:
            r.backend.post()

    def gather(self, names=("x", "v", "rho", "h")):
        """fields of all owned particles in reference index order"""
        parts = [r.owned_fields(names) for r in self.runs]
        gidx = np.concatenate([p[0] for p in parts])
        order = np.argsort(gidx, kind="stable")
        return gidx[order], {f: np.concatenate([p[1][f] for p in parts])[order] for f in names}

"""Host-side mirror of the reference's particle-operator API over libsphmw.so.

Mirrors (names and argument meaning kept; `!` dropped, Python has none):
  ParticleSystem(T, domain, h)          src/structs.jl:43-92
  generate_particles(sys, grid, shape, ctor)   src/grids.jl:305-310
  create_cell_list(sys)                 src/core.jl:51-90
  apply(sys, f; self=False), apply_unary, apply_binary   src/core.jl:125-161
  ParticleField(sys, name)              src/structs.jl:118-125
  new_pvd_file / save_frame / save_pvd_file    src/IO.jl:20-75

State lives in HBM inside the library context; the host only stages particles
between `generate_particles` and the first device call, and gathers fields on
demand.  A closure that is not in the device operator menu raises
UnsupportedOperator — there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Callable, Dict, Iterable, Optional

import numpy as np

from . import _capi
from ._capi import Config, SphmwError, UnsupportedOperator, check
from .geometry import Shape

# canonical ASCII field names and their component counts (a1 in SURVEY.md §8)
FIELD_NCOMP: Dict[str, int] = {
    "h": 1, "x": 3, "m": 1, "v": 3, "Dv": 3, "rho_bg": 1, "rho_p": 1, "rho": 1, "P_bg": 1,
    "P_p": 1, "P": 1, "theta_bg": 1, "theta_p": 1, "theta": 1, "T_bg": 1, "T_p": 1, "T": 1,
    "type": 1, "A": 1, "A_bg": 1, "Drho": 1, "rho0": 1, "S": 1, "s": 1,
}
ALIASES = {"ρ_bg": "rho_bg", "ρ′": "rho_p", "ρ": "rho", "P′": "P_p", "θ_bg": "theta_bg",
           "θ′": "theta_p", "θ": "theta", "T′": "T_p", "a": "Dv", "u": "v"}


def canonical(name: str) -> str:
    name = ALIASES.get(name, name)
    if name not in FIELD_NCOMP:
        # structs.jl:128-133
        raise KeyError("Variable " + name + " does not exist!")
    return name


@dataclass(frozen=True)
class Operator:
    """A driver closure that exists in the device menu, e.g.
    Operator("wcsph.compute_density") ≙ compute_density! of
    src/current/wcsph_perturbed_witch.jl:226-228."""
    name: str

    def __call__(self, *a, **k):
        raise TypeError("device operators are applied with apply(sys, op), not called on the host")


@dataclass
class ParticleType:
    """≙ a driver's `mutable struct Particle <: AbstractParticle`: the field list and
    the scheme it belongs to.  `x` is mandatory (structs.jl:61)."""
    name: str
    fields: Iterable[str]
    scheme: str = "wcsph"

    def __post_init__(self):
        self.fields = tuple(canonical(f) for f in self.fields)


class ParticleSystem:
    """≙ ParticleSystem{T}(T, domain, h) — src/structs.jl:43-92."""

    def __init__(self, T: ParticleType, domain: Shape, h: float, *, params: Optional[dict] = None,
                 capacity: Optional[int] = None, device: int = 0, slab=None, stream=None, flags: int = 0):
        # structs.jl:59-61
        assert h > 0.0, "invalid ParticleSystem declaration! (h must be a positive float)"
        assert isinstance(T, ParticleType), \
            "invalid ParticleSystem declaration! (" + str(T) + " is not an AbstractParticle subtype)"
        assert "x" in T.fields, \
            "invalid ParticleSystem declaration! (particles must have a field `x::RealVector`)"
        self.T = T
        self.h = float(h)
        self.domain = domain.boundarybox()  # structs.jl:63,87 keeps the bounding box only
        self.params = dict(params or {})
        self.device = device
        self._capacity = capacity
        self._slab = slab
        self._stream = stream
        self._flags = int(flags)
        self._ctx = None
        self._staged: Dict[str, list] = {}
        self._staged_n = 0
        self._pvd = None

    # ------------------------------------------------------------------ context
    def _make_ctx(self, n_needed: int):
        cfg = Config()
        b = self.domain
        cfg.box_min[:] = (b.x1_min, b.x2_min, b.x3_min)
        cfg.box_max[:] = (b.x1_max, b.x2_max, b.x3_max)
        cfg.h = self.h
        cap = self._capacity if self._capacity is not None else max(1024, int(n_needed * 1.05) + 64)
        cfg.capacity = max(cap, n_needed)
        cfg.device = self.device
        cfg.flags = self._flags
        cfg.slab_lo, cfg.slab_hi = (-1, -1) if self._slab is None else self._slab
        h = C.c_void_p()
        check(_capi.lib().sphmw_create(C.byref(cfg), C.byref(h)))
        self._ctx = h
        if self._stream is not None:
            check(_capi.lib().sphmw_set_stream(self._ctx, C.c_void_p(self._stream)))
        for k, v in self.params.items():
            check(_capi.lib().sphmw_set_param(self._ctx, k.encode(), float(v)))

    @property
    def ctx(self):
        if self._ctx is None:
            self._make_ctx(self._staged_n)
        return self._ctx

    def set_param(self, name: str, value: float):
        self.params[name] = float(value)
        if self._ctx is not None:
            check(_capi.lib().sphmw_set_param(self._ctx, name.encode(), float(value)))

    def close(self):
        if self._ctx is not None:
            _capi.lib().sphmw_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ particles
    def append(self, fields: Dict[str, np.ndarray]):
        """≙ push!(sys.particles, p) for a batch: `fields[name]` is (N,) or (N,3)."""
        n = len(np.asarray(fields["x"]))
        for name in self.T.fields:
            ncomp = FIELD_NCOMP[name]
            if name in fields or ALIASES_INV.get(name) in fields:
                a = np.asarray(fields.get(name, fields.get(ALIASES_INV.get(name))), dtype=np.float64)
            else:
                a = np.zeros((n, 3) if ncomp == 3 else n)
            if ncomp == 3:
                assert a.shape == (n, 3), f"field {name}: expected ({n},3), got {a.shape}"
            else:
                assert a.shape == (n,), f"field {name}: expected ({n},), got {a.shape}"
            self._staged.setdefault(name, []).append(a)
        self._staged_n += n

    def _flush(self):
        if self._staged_n == 0:
            return
        lib = _capi.lib()
        ctx = self.ctx
        n0 = self.n_device
        n1 = n0 + self._staged_n
        new = {k: np.concatenate(v) for k, v in self._staged.items()}
        old = {}
        if n0 > 0:
            old = {k: self._download(k) for k in self.T.fields}
        check(lib.sphmw_resize(ctx, n1))
        for name in self.T.fields:
            a = new[name]
            if n0 > 0:
                a = np.concatenate([old[name], a])
            self._upload(name, a)
        self._staged.clear()
        self._staged_n = 0

    @property
    def n_device(self) -> int:
        if self._ctx is None:
            return 0
        n = C.c_int64()
        check(_capi.lib().sphmw_count(self._ctx, C.byref(n)))
        return n.value

    def __len__(self):
        return self.n_device + self._staged_n

    @property
    def n(self) -> int:
        return len(self)

    def _upload(self, name: str, a: np.ndarray):
        ncomp = FIELD_NCOMP[name]
        n = a.shape[0]
        soa = np.ascontiguousarray(a.T if ncomp == 3 else a, dtype=np.float64)
        check(_capi.lib().sphmw_upload(self.ctx, name.encode(), _capi.ptr(soa), n, ncomp))

    def _download(self, name: str) -> np.ndarray:
        ncomp = FIELD_NCOMP[name]
        n = self.n_device
        buf = np.empty((ncomp, n) if ncomp == 3 else n, dtype=np.float64)
        if n:
            check(_capi.lib().sphmw_download(self.ctx, name.encode(), _capi.ptr(buf), n, ncomp))
        return np.ascontiguousarray(buf.T) if ncomp == 3 else buf

    def field(self, name: str) -> np.ndarray:
        """≙ collect(ParticleField(sys, name)): values in particle index order."""
        self._flush()
        return self._download(canonical(name))

    def set_field(self, name: str, values):
        self._flush()
        name = canonical(name)
        a = np.asarray(values, dtype=np.float64)
        self._upload(name, a)

    # raw SoA transfer for callers that already hold component-major (pinned) buffers
    def upload_soa(self, name: str, soa: np.ndarray):
        name = canonical(name)
        ncomp = FIELD_NCOMP[name]
        n = soa.shape[-1]
        check(_capi.lib().sphmw_upload(self.ctx, name.encode(), _capi.ptr(soa), n, ncomp))

    def download_soa(self, name: str, soa: np.ndarray):
        name = canonical(name)
        ncomp = FIELD_NCOMP[name]
        n = soa.shape[-1]
        check(_capi.lib().sphmw_download(self.ctx, name.encode(), _capi.ptr(soa), n, ncomp))

    def upload_ptr(self, name: str, data_ptr: int, n: int):
        name = canonical(name)
        check(_capi.lib().sphmw_upload(self.ctx, name.encode(), C.c_void_p(data_ptr), n, FIELD_NCOMP[name]))

    def download_ptr(self, name: str, data_ptr: int, n: int):
        name = canonical(name)
        check(_capi.lib().sphmw_download(self.ctx, name.encode(), C.c_void_p(data_ptr), n, FIELD_NCOMP[name]))

    def resize(self, n: int):
        check(_capi.lib().sphmw_resize(self.ctx, n))

    # ------------------------------------------------------------------ operators
    def create_cell_list(self, want_count: bool = True) -> Optional[int]:
        self._flush()
        if want_count:
            n = C.c_int64()
            check(_capi.lib().sphmw_create_cell_list(self.ctx, C.byref(n)))
            return n.value
        check(_capi.lib().sphmw_create_cell_list(self.ctx, None))
        return None

    def apply(self, op, self_: bool = False):
        self._flush()
        if isinstance(op, Operator):
            name = op.name
        elif isinstance(op, str):
            name = op
        else:
            raise UnsupportedOperator(
                _capi.E_UNSUPPORTED_OP,
                f"{getattr(op, '__name__', op)!r} is a host closure; only operators of the device "
                "menu can be applied (no CPU fallback)")
        check(_capi.lib().sphmw_apply(self.ctx, name.encode(), 1 if self_ else 0))

    def step(self, nsteps: int = 1, scheme: Optional[str] = None):
        """Fused fast path ≙ `for k in 1:nsteps verlet_step!(sys) end`."""
        self._flush()
        check(_capi.lib().sphmw_step(self.ctx, (scheme or self.T.scheme).encode(), nsteps))

    def generate_mountain_wave(self, setup) -> tuple:
        """device-side make_system() (sphmw_generate_mountain_wave); returns the three group sizes"""
        self._flush()
        n = C.c_int64()
        gc = (C.c_int64 * 3)()
        check(_capi.lib().sphmw_generate_mountain_wave(self.ctx, C.byref(setup), C.byref(n), gc))
        return tuple(gc)

    def flow_add_new_particles(self) -> int:
        """≙ add_new_particles!(sys) — src/legacy/isothermal_flow_witch.jl:175-186"""
        self._flush()
        n = C.c_int64()
        check(_capi.lib().sphmw_flow_add_new_particles(self.ctx, C.byref(n)))
        return n.value

    def aflow_add_new_particles(self) -> int:
        """≙ add_new_particles!(sys) — src/legacy/adiabatic_flow_witch.jl:197-208"""
        self._flush()
        n = C.c_int64()
        check(_capi.lib().sphmw_aflow_add_new_particles(self.ctx, C.byref(n)))
        return n.value

    def set_flags(self, flags: int):
        self._flags = int(flags)
        check(_capi.lib().sphmw_set_flags(self.ctx, int(flags)))

    def pair_list_info(self) -> dict:
        """stride, lists built, particles that overflowed the stride, device bytes"""
        out = (C.c_int64 * 4)()
        check(_capi.lib().sphmw_pair_list_info(self.ctx, out))
        info = {"stride": out[0], "builds": out[1], "overflow": out[2], "bytes": out[3]}
        t = (C.c_int64 * 6)()
        check(_capi.lib().sphmw_tile_info(self.ctx, t))
        if t[0]:
            info["tiles"] = {"blocks": t[0], "staged": t[1], "max_slots": t[2],
                             "mean_slots": (t[3] / t[1]) if t[1] else None, "capacity": t[4],
                             "too_many_rows": t[5]}
        return info

    def sync(self):
        if self._ctx is not None:
            check(_capi.lib().sphmw_sync(self._ctx))

    # ------------------------------------------------------------------ diagnostics / hooks
    def reduce(self, what: str) -> float:
        self._flush()
        out = C.c_double()
        check(_capi.lib().sphmw_reduce(self.ctx, what.encode(), C.byref(out)))
        return out.value

    def point_sum(self, points, ops):
        """≙ sum(sys, f, x) of src/core.jl:240-291 at many points (sphmw_point_sum): row o of the result
        is op o ("count", "mW", "VW", "mW*<field>", "VW*<field>", e.g. "VW*v[1]") summed over the particles
        within h of each point, in the reference's traversal order.  `points` is an (n, 3) float64 numpy
        array, or a CUDA torch tensor, which stays on the device (the result is then a CUDA tensor).
        Points outside the box give NaN.  Needs a current cell list."""
        self._flush()
        ops = [ops] if isinstance(ops, str) else list(ops)
        arr = (C.c_char_p * len(ops))(*[o.encode() for o in ops])
        if type(points).__module__.split(".")[0] == "torch":
            import torch
            if not points.is_cuda or points.dtype != torch.float64 or points.dim() != 2 or points.shape[1] != 3:
                raise ValueError("points: expected a CUDA float64 tensor of shape (n, 3)")
            soa = points.t().contiguous()
            out = torch.empty((len(ops), points.shape[0]), dtype=torch.float64, device=points.device)
            torch.cuda.current_stream(points.device).synchronize()  # the library runs on its own stream
            check(_capi.lib().sphmw_point_sum(self.ctx, arr, len(ops), C.c_void_p(soa.data_ptr()),
                                              points.shape[0], C.c_void_p(out.data_ptr())))
            self.sync()
            return out
        pts = np.asarray(points, dtype=np.float64)
        if pts.ndim != 2 or pts.shape[1] != 3:
            raise ValueError(f"points: expected shape (n, 3), got {pts.shape}")
        soa = np.ascontiguousarray(pts.T)
        out = np.empty((len(ops), pts.shape[0]), dtype=np.float64)
        check(_capi.lib().sphmw_point_sum(self.ctx, arr, len(ops), _capi.ptr(soa), pts.shape[0], _capi.ptr(out)))
        return out

    def interpolate(self, points, fields) -> dict:
        """Shepard interpolant Σ VW*f / Σ VW of each field at the points, from one point_sum call
        (len(fields) + 1 <= 8 ops); NaN where no particle is within h or the point is outside the box."""
        fields = [fields] if isinstance(fields, str) else list(fields)
        s = self.point_sum(points, ["VW"] + [f"VW*{f}" for f in fields])
        den = s[0]
        if isinstance(s, np.ndarray):
            with np.errstate(invalid="ignore", divide="ignore"):
                return {f: np.where(den == 0.0, np.nan, s[k + 1] / den) for k, f in enumerate(fields)}
        nan = den.new_full((), float("nan"))
        return {f: (s[k + 1] / den).where(den != 0.0, nan) for k, f in enumerate(fields)}

    def key_tables(self):
        ph = (C.c_int64 * 3)()
        lim = (C.c_int64 * 3)()
        km = C.c_int64()
        dim = C.c_int32()
        check(_capi.lib().sphmw_key_tables(self.ctx, ph, lim, C.byref(km), C.byref(dim)))
        return tuple(ph), tuple(lim), km.value, dim.value

    def cell_keys(self) -> np.ndarray:
        n = self.n_device
        keys = np.empty(n, dtype=np.int64)
        check(_capi.lib().sphmw_cell_keys(self.ctx, _capi.ptr(keys), n))
        return keys

    def cell_entries(self, key: int) -> np.ndarray:
        cnt = C.c_int64()
        check(_capi.lib().sphmw_cell_entries(self.ctx, key, None, 0, C.byref(cnt)))
        out = np.empty(cnt.value, dtype=np.int64)
        if cnt.value:
            check(_capi.lib().sphmw_cell_entries(self.ctx, key, _capi.ptr(out), cnt.value, C.byref(cnt)))
        return out

    def pairs(self):
        cnt = C.c_int64()
        check(_capi.lib().sphmw_pairs_dump(self.ctx, None, None, 0, C.byref(cnt)))
        pi = np.empty(cnt.value, dtype=np.int64)
        pj = np.empty(cnt.value, dtype=np.int64)
        if cnt.value:
            check(_capi.lib().sphmw_pairs_dump(self.ctx, _capi.ptr(pi), _capi.ptr(pj), cnt.value, C.byref(cnt)))
        return pi, pj

    def count_pairs(self, enable: bool = True):
        check(_capi.lib().sphmw_count_pairs(self.ctx, 1 if enable else 0))

    def pair_count(self) -> int:
        n = C.c_int64()
        check(_capi.lib().sphmw_pair_count(self.ctx, C.byref(n)))
        return n.value

    def timing(self, enable: bool = True, prefix: str = ""):
        """per-kernel CUDA-event timers; `prefix` limits them to the kernels named so"""
        check(_capi.lib().sphmw_timing_filter(self.ctx, prefix.encode()))
        check(_capi.lib().sphmw_timing_enable(self.ctx, 1 if enable else 0))

    def timing_reset(self):
        check(_capi.lib().sphmw_timing_reset(self.ctx))

    def timing_report(self) -> Dict[str, tuple]:
        cap = 1 << 14
        names = C.create_string_buffer(cap)
        ms = (C.c_double * 256)()
        calls = (C.c_int64 * 256)()
        n = _capi.lib().sphmw_timing_report(self.ctx, names, cap, ms, calls, 256)
        check(int(n))
        ns = names.value.decode().split("\n")
        return {ns[i]: (ms[i], calls[i]) for i in range(min(n, 256))}

    def launch_count(self) -> int:
        n = C.c_int64()
        check(_capi.lib().sphmw_launch_count(self.ctx, C.byref(n)))
        return n.value


ALIASES_INV = {v: k for k, v in ALIASES.items()}


# ---------------------------------------------------------------------- free functions
def generate_particles(sys: ParticleSystem, grid, geometry: Shape, constructor: Callable):
    """≙ generate_particles!(sys, grid, geometry, constructor) — src/grids.jl:305-310.
    `constructor(xs)` is vectorised: (N,3) positions -> dict of field arrays."""
    from .grids import covering
    xs = covering(grid, geometry)
    if len(xs):
        sys.append(constructor(xs))
    return len(xs)


def create_cell_list(sys: ParticleSystem):
    """≙ create_cell_list!(sys) — src/core.jl:51-90."""
    sys.create_cell_list()


def apply_unary(sys: ParticleSystem, action):
    """≙ apply_unary!(sys, action!) — src/core.jl:138-142."""
    sys.apply(action, False)


def apply_binary(sys: ParticleSystem, action):
    """≙ apply_binary!(sys, action!) — src/core.jl:125-129."""
    sys.apply(action, False)


def apply(sys: ParticleSystem, action, self: bool = False):
    """≙ apply!(sys, action!; self) — src/core.jl:151-161."""
    sys.apply(action, self)


def ParticleField(sys: ParticleSystem, name: str) -> np.ndarray:
    """≙ ParticleField(sys, varS) — src/structs.jl:118-125 (a gathered copy)."""
    return sys.field(name)


def op_menu() -> Dict[str, str]:
    n = _capi.lib().sphmw_op_list(None, 0)
    buf = C.create_string_buffer(int(n))
    _capi.lib().sphmw_op_list(buf, n)
    out = {}
    for line in buf.value.decode().splitlines():
        name, kind = line.split()
        out[name] = kind
    return out


# ---------------------------------------------------------------------- IO.jl
class DataStorage:
    """≙ DataStorage — src/IO.jl:9-13"""

    def __init__(self, path: str):
        self.path = path
        self.frame = 0
        self.sys = None


def new_pvd_file(path: str) -> DataStorage:
    """≙ new_pvd_file(path) — src/IO.jl:20-26"""
    return DataStorage(path)


def save_frame(data: DataStorage, sys: ParticleSystem, *vars: str):
    """≙ save_frame!(data, sys, vars...) — src/IO.jl:53-75"""
    sys._flush()
    lib = _capi.lib()
    if data.sys is not sys:
        check(lib.sphmw_pvd_open(sys.ctx, data.path.encode()))
        data.sys = sys
    names = [canonical(v) for v in vars]
    # the reference writes the Julia field names into the file (IO.jl:60,68)
    arr = (C.c_char_p * len(vars))(*[v.encode() for v in vars])
    del names
    check(lib.sphmw_pvd_save_frame(sys.ctx, arr, len(vars)))
    data.frame += 1


def save_pvd_file(data: DataStorage):
    """≙ save_pvd_file(data) — src/IO.jl:33-35"""
    if data.sys is not None:
        check(_capi.lib().sphmw_pvd_close(data.sys.ctx))


def read_vtp(path: str) -> Dict[str, np.ndarray]:
    """All arrays of a PolyData .vtp file: "Points" (N,3) plus every PointData array,
    (N,) or (N,ncomp).  Host-only (libsphmw's reader, no GPU)."""
    lib = _capi.lib()
    h = C.c_void_p()
    check(lib.sphmw_vtp_open(path.encode(), C.byref(h)))
    try:
        n, na = C.c_int64(), C.c_int32()
        check(lib.sphmw_vtp_info(h, C.byref(n), C.byref(na)))
        out = {}
        for i in range(na.value):
            name = C.create_string_buffer(256)
            nc = C.c_int32()
            check(lib.sphmw_vtp_array(h, i, name, 256, C.byref(nc)))
            a = np.empty(n.value * nc.value, dtype=np.float64)
            check(lib.sphmw_vtp_read(h, name.value, _capi.ptr(a), a.size))
            out[name.value.decode()] = a.reshape(n.value, nc.value) if nc.value > 1 else a
        return out
    finally:
        lib.sphmw_vtp_close(h)


def write_vtp(path: str, points: np.ndarray, fields: Dict[str, np.ndarray]):
    """One frame in WriteVTK's layout (what save_frame! writes), from host arrays."""
    pts = np.ascontiguousarray(points, dtype=np.float64)
    names = list(fields)
    arrs = [np.ascontiguousarray(fields[k], dtype=np.float64) for k in names]
    nc = (C.c_int32 * len(names))(*[1 if a.ndim == 1 else a.shape[1] for a in arrs])
    cn = (C.c_char_p * len(names))(*[k.encode() for k in names])
    dp = (C.c_void_p * len(names))(*[a.ctypes.data for a in arrs])
    check(_capi.lib().sphmw_vtp_write(path.encode(), len(pts), _capi.ptr(pts), len(names), cn, nc, dp))


def import_particles(sys: ParticleSystem, path: str, particle_constructor: Callable):
    """≙ import_particles!(sys, path, ctor) — src/IO.jl:83-122: particles are created by
    `ctor(x)` at the file's points, then every field whose name matches a PointData array is
    overwritten with the file's values; the new particles are appended to `sys`."""
    data = read_vtp(path)
    x = data["Points"]
    fields = dict(particle_constructor(x))
    fields["x"] = x
    for name in sys.T.fields:
        for key in (name, ALIASES_INV.get(name)):
            if key is not None and key in data and name != "x":
                fields[name] = data[key]
    sys.append(fields)
    return len(x)

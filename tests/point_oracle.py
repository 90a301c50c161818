"""ctypes wrapper of tests/c/point_sum_oracle.c, the CPU restatement of the point sum `sum(sys, f, x)`
(src/core.jl:240-291) that the point-sum tests check the device against.  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
SRC = HERE / "c" / "point_sum_oracle.c"
LIB = HERE / "c" / "build" / "libpoint_sum_oracle.so"
KIND = {"count": 0, "mW": 1, "VW": 3}
JULIA = {"ρ′": "rho_p", "ρ": "rho", "θ′": "theta_p", "θ": "theta", "P′": "P_p", "T′": "T_p", "u": "v", "a": "Dv"}

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not LIB.exists() or LIB.stat().st_mtime < SRC.stat().st_mtime:
            LIB.parent.mkdir(exist_ok=True)
            subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-o", str(LIB),
                            str(SRC), "-lm"], check=True)
        _lib = C.CDLL(str(LIB))
        _lib.pso_point_sum.argtypes = [C.c_void_p, C.c_double, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    return _lib


def _column(fields, op):
    """the per-particle array an op multiplies in: 'v[1]' -> fields['v'][:, 1], 'ρ′' -> fields['rho_p']"""
    name, _, comp = op.partition("[")
    a = np.asarray(fields[JULIA.get(name, name)], dtype=np.float64)
    return a[:, int(comp[0])] if comp else a


def point_sum(box_min, box_max, h, fields, points, ops) -> np.ndarray:
    """(len(ops), n) point sums of `ops` at the rows of `points` (n, 3) over the particles `fields`
    (reference index order: x (N, 3), m, rho and the fields the ops name), each particle inside the box"""
    x = np.ascontiguousarray(np.asarray(fields["x"], dtype=np.float64).T)
    n = x.shape[1]
    keep = []
    kinds = np.empty(len(ops), dtype=np.int32)
    fptr = (C.c_void_p * max(1, len(ops)))()
    for o, op in enumerate(ops):
        base, _, name = op.partition("*")
        kinds[o] = KIND[base] + (1 if name else 0)
        if name:
            col = np.ascontiguousarray(_column(fields, name))
            keep.append(col)
            fptr[o] = col.ctypes.data
    m = np.ascontiguousarray(fields["m"], dtype=np.float64)
    rho = np.ascontiguousarray(fields.get("rho", np.zeros(n)), dtype=np.float64)
    box = np.array(list(box_min) + list(box_max), dtype=np.float64)
    pts = np.ascontiguousarray(np.asarray(points, dtype=np.float64).T)
    out = np.empty((len(ops), pts.shape[1]), dtype=np.float64)
    rc = lib().pso_point_sum(box.ctypes.data, float(h), n, x.ctypes.data, m.ctypes.data, rho.ctypes.data, len(ops),
                             kinds.ctypes.data, fptr, pts.ctypes.data, pts.shape[1], out.ctypes.data)
    assert rc == 0, f"point_sum_oracle failed ({rc}): every particle must be inside the box"
    return out


def for_case(case, points, ops) -> np.ndarray:
    return point_sum(case.box_min, case.box_max, case.h, case.fields, points, ops)

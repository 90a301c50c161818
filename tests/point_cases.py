"""Lattices and sample points shared by the point-sum tests (emulated, oracle and GPU)."""
from __future__ import annotations

import numpy as np

from sph_mountain_waves_b200 import cases

OPS_2D = ["count", "mW", "VW", "mW*rho_p", "VW*v[0]", "VW*v[1]", "VW*ρ′", "mW*v[0]"]
OPS_3D = ["count", "mW", "VW", "mW*rho_p", "VW*v[0]", "VW*v[1]", "VW*rho_p", "VW*v[2]"]


def ops_for(case):
    return OPS_2D if case.dim == 2 else OPS_3D


def witch_2d():
    """small 2D Witch of Agnesi case (hexagonal lattice, wall fence, mountain)"""
    return cases.mountain_wave_2d(n_y=24.0, dom_length=80e3, h_m=3000.0, a=10e3, U=20.0)


def hex_2d():
    """the shipped driver's hexagonal lattice without a mountain"""
    return cases.mountain_wave_2d(n_y=24.0, dom_length=70e3)


def hill_3d():
    """small 3D bell hill case (cubic lattice)"""
    return cases.bell_hill_3d(24, 12, 10, h_m=3000.0, a=8e3, U=20.0)


def narrow(dim: int, seed: int = 3):
    """a box two cells wide in x (h = 1): the reference's linear key wrap adds cells of the next row.
    Particles sit on a lattice of spacing 1/4 (dyadic), so a point h away from one is exactly h away."""
    rng = np.random.default_rng(seed)
    hi = (1.75, 5.0, 0.0 if dim == 2 else 3.0)
    axes = [np.arange(0.0, hi[a] + 1e-9, 0.25) for a in range(dim)]
    grid = np.stack(np.meshgrid(*axes, indexing="ij"), -1).reshape(-1, dim)
    x = np.zeros((len(grid), 3))
    x[:, :dim] = grid
    n = len(x)
    fields = {"x": x, "m": rng.uniform(0.5, 1.5, n), "rho": rng.uniform(0.8, 1.2, n),
              "rho_p": rng.normal(size=n), "v": rng.normal(size=(n, 3)) * (np.arange(3) < dim),
              "h": np.ones(n), "type": np.zeros(n)}
    return cases.Case(f"narrow{dim}d", "wcsph", dim, (0.0, 0.0, 0.0), hi, 1.0, {"fluid": 0.0}, fields)


def sample_points(case, n_random: int = 400, seed: int = 7) -> np.ndarray:
    """random points in the box, points on particles (r = 0), points h away from a particle along x,
    points on cell faces (a coordinate a multiple of h), on the closed box faces, outside the box and NaN"""
    rng = np.random.default_rng(seed)
    lo = np.array(case.box_min, dtype=np.float64)
    hi = np.array(case.box_max, dtype=np.float64)
    dim, h = case.dim, case.h
    x = case.fields["x"]
    k = min(len(x), 64)
    pick = rng.choice(len(x), size=k, replace=False)
    rand = lo + rng.random((n_random, 3)) * (hi - lo)
    on = x[pick].copy()
    away = x[pick].copy()
    away[:, 0] += h
    away = away[(away[:, 0] <= hi[0])]
    faces = lo + rng.random((k, 3)) * (hi - lo)
    for a in range(dim):
        faces[: k // 2, a] = np.floor(faces[: k // 2, a] / h) * h
    faces = np.clip(faces, lo, hi)
    box = lo + rng.random((2 * dim, 3)) * (hi - lo)
    for a in range(dim):
        box[2 * a, a] = lo[a]
        box[2 * a + 1, a] = hi[a]
    out = np.array([hi + h * 0.5, lo - h * 0.25, [lo[0] - 1e-9, lo[1], lo[2]], [np.nan, lo[1], lo[2]],
                    [lo[0], np.nan, lo[2]]])
    if dim == 2:
        out = np.vstack([out, [0.5 * (lo[0] + hi[0]), 0.5 * (lo[1] + hi[1]), 1e-3]])
    else:
        out = np.vstack([out, [lo[0], lo[1], np.nan]])
    for p in (rand, faces, box):
        if dim == 2:
            p[:, 2] = 0.0
    pts = np.vstack([rand, on, away, faces, box, out])
    return pts[rng.permutation(len(pts))]

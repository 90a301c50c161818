"""One verlet_step! of the WCSPH driver (wcsph_perturbed_witch.jl:309-332) restated in extended
precision (np.longdouble: a 64-bit significand on x86-64, unit roundoff 2^-64 ~ 5.4e-20), in
three stages that each start from given FP64 inputs, so that one stage's FP64 rounding on the
device does not enter the next stage's reference:

  kick_drift      accelerate! (Dv = 0, :302) and move! from the carried state     (:311-312)
  density         compute_density! (old h, no self term), finalize_density!,
                  update_smoothing! with rho_floor, compute_pressure!             (:316-323)
  force_kick      balance_of_momentum! (h_ij kernel, viscosity on dot < 0) and the
                  closing accelerate!                                             (:330-331)

Every branch the device decides on FP64 values that are inputs here is decided here on the same
FP64 values: the neighbour set (`dist`: dx*dx + dy*dy + dz*dz left to right, sqrt, r <= h), the
sponge test y >= z_t - z_b and the fluid test.  The branches on computed values (x > 1 inside the
kernels, dot < 0) are taken on the extended values; where the device may decide differently the
term is near zero and inside the error scale (see `_mag_*`).

Every output comes with an error scale: the quantity a backward-stable FP64 evaluation of the
same formula can be wrong by, in units of u = 2^-53, per operation.  For a pair sum it is the sum
over accepted pairs of a magnitude bound of each term, which includes the term's condition with
respect to r (|x dW/dx| next to |W|) and the magnitudes of every operand that can cancel; for a
per-particle formula it is the magnitude of its inputs, propagated.  `n_p` is each particle's
accepted-pair count.  A device result y is then expected within K * u * scale of the extended
value, with K = n_p + c (tests/test_xp_wcsph_emulated.py derives c).

Non-finite values follow the reference: an isolated fluid particle gets rho = 0 and its buoyancy
divides by zero, to +-inf or NaN; the same expressions in the same order produce the same class.
"""
from __future__ import annotations

import numpy as np

LD = np.longdouble
U = 2.0 ** -53                                    # FP64 unit roundoff
PI = LD("3.14159265358979323846264338327950288")  # not np.pi: that is pi rounded to FP64

# kernels.jl:108-195, in extended precision: W = CW (1-x)^4 (1+4x) / h^d, rDW = CD (1-x)^3 / h^(d+2)
CW = {2: LD(7) / PI, 3: LD(21) / (LD(2) * PI)}
CD = {2: -LD(140) / PI, 3: -LD(210) / PI}


def _ld(a):
    return np.asarray(a, dtype=np.float64).astype(LD)


def sponge_y(p):
    """damping_structure :245-251 in extended precision"""
    z_t, z_b = LD(p["z_t"]), LD(p["z_b"])
    if z_b == 0:
        return LD(0)
    sn = np.sin(PI / 2 * (1 - (z_t - z_b) / z_b))
    return -LD(p["gamma_r"]) * sn * sn


def neighbour_pairs(x, h, targets=None):
    """ordered pairs (i, j), i != j, i in `targets` (all particles if None), with the FP64 `dist`
    of core.jl:104-105 <= h.  A k-d tree with a margin proposes candidates; the test itself is
    the reference's, in FP64 and left to right."""
    from scipy.spatial import cKDTree
    x = np.asarray(x, dtype=np.float64)
    tree = cKDTree(x)
    if targets is None:
        und = tree.query_pairs(h * (1 + 1e-9), output_type="ndarray")
        i = np.concatenate([und[:, 0], und[:, 1]])
        j = np.concatenate([und[:, 1], und[:, 0]])
    else:
        lists = tree.query_ball_point(x[targets], h * (1 + 1e-9))
        i = np.repeat(np.asarray(targets), [len(l) for l in lists])
        j = np.concatenate([np.asarray(l, dtype=np.int64) for l in lists]) if len(lists) else np.zeros(0, np.int64)
        keep = i != j
        i, j = i[keep], j[keep]
    d = x[i] - x[j]
    r = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])
    keep = r <= h
    order = np.argsort(i[keep], kind="stable")
    return i[keep][order], j[keep][order]


def _segment_sum(i, w, n):
    """per-particle sums of pair terms `w` (pairs sorted by i), in extended precision; 0 where a
    particle has no pair"""
    out = np.zeros((n,) + w.shape[1:], dtype=LD)
    if len(i) == 0:
        return out
    starts = np.flatnonzero(np.r_[True, i[1:] != i[:-1]])
    out[i[starts]] = np.add.reduceat(w, starts, axis=0)
    return out


def kick_drift(f, p):
    """accelerate! with Dv = 0 and move! (:311-312, :298-303, :292-296).  Returns v_half and the
    new x (extended) with their scales."""
    fluid = np.asarray(f["type"]) == p["fluid"]
    x, v = _ld(f["x"]), _ld(f["v"])
    rho, rho_p = _ld(f["rho"]), _ld(f["rho_p"])
    g, hdt, dt = LD(p["g"]), LD(0.5) * LD(p["dt"]), LD(p["dt"])
    sponge = np.asarray(f["x"])[:, 1] >= p["z_t"] - p["z_b"]      # FP64 test, as the device
    sy = sponge_y(p)
    with np.errstate(all="ignore"):
        buoy = np.stack([(-g * LD(e)) * rho_p / rho for e in (0.0, 1.0, 0.0)], axis=1)
    damp = np.zeros_like(v)
    damp[sponge, 1] = sy
    kick = hdt * (buoy + damp)
    vh = np.where(fluid[:, None], v + kick, v)
    xn = np.where(fluid[:, None], x + dt * vh, x)
    with np.errstate(all="ignore"):
        s_v = np.where(fluid[:, None], np.abs(v) + hdt * (np.abs(buoy) + np.abs(damp)), LD(0))
        s_x = np.where(fluid[:, None], np.abs(x) + dt * (np.abs(vh) + s_v), LD(0))
    return dict(v=vh, x=xn, s_v=s_v, s_x=s_x)


def density(f, p, h_cut, dim, targets=None, pairs=None):
    """compute_density! (old h, no self term), finalize_density!, update_smoothing! (rho_floor)
    and compute_pressure! (:316-323, :177-179, :195-199, :226-238) from FP64 x, h, m.  Returns
    rho, rho_p, h, P, P_p (extended), their scales, and n_p."""
    x64 = np.asarray(f["x"], dtype=np.float64)
    n = len(x64)
    i, j = neighbour_pairs(x64, h_cut, targets) if pairs is None else pairs
    x, h, m = _ld(x64), _ld(f["h"]), _ld(f["m"])
    d = x[i] - x[j]
    r = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])
    q = r / h[i]
    inside = q <= 1
    t = np.where(inside, 1 - q, LD(0))
    cw = CW[dim] / h[i] ** dim
    w = m[j] * cw * t ** 4 * (1 + 4 * q)
    # |W| + |x dW/dx|: the term's own size and its condition with respect to r / h
    mag = m[j] * cw * t ** 3 * (t * (1 + 4 * q) + 20 * q * q)
    rho = _segment_sum(i, w, n)
    s_rho = _segment_sum(i, mag, n)
    n_p = np.bincount(i, minlength=n)
    # finalize_density! / update_smoothing! / compute_pressure!
    y = x[:, 1]
    arg = -y * LD(p["g"]) / (LD(p["R_mass"]) * LD(p["T_bg"]))
    rbg = LD(p["rho0"]) * np.exp(arg)
    s_rbg = np.abs(rbg) * (1 + np.abs(arg))                 # exp amplifies the argument's rounding
    rho_p = rho - rbg
    s_rho_p = s_rho + s_rbg
    floor = LD(p["rho_floor"])
    rfl = np.where(np.isnan(rho), rho, np.maximum(rho, floor))
    ratio = m / rfl
    hn = LD(p["eta"]) * (np.cbrt(ratio) if dim == 3 else np.sqrt(ratio))
    s_h = np.abs(hn) * (1 + np.where(rho > floor, s_rho / np.abs(rfl), LD(0)))
    c2 = LD(p["c"]) * LD(p["c"])
    RT = LD(p["R_mass"]) * LD(p["T_bg"])
    P_p = c2 * rho_p
    P = RT * rbg + P_p
    s_P_p = c2 * s_rho_p
    s_P = RT * s_rbg + s_P_p + np.abs(P)
    return dict(rho=rho, rho_p=rho_p, h=hn, P=P, P_p=P_p, s_rho=s_rho, s_rho_p=s_rho_p, s_h=s_h, s_P=s_P,
                s_P_p=s_P_p, n_p=n_p)


def force_kick(f, p, h_cut, dim, targets=None, pairs=None):
    """balance_of_momentum! (:261-286) and the closing accelerate! (:330-331) from FP64 x, v (the
    half-step velocity), h, m, rho, rho_p, P, P_p.  Returns the new v (extended), its scale per
    component, and n_p.  Non-fluid particles keep v."""
    x64 = np.asarray(f["x"], dtype=np.float64)
    n = len(x64)
    i, j = neighbour_pairs(x64, h_cut, targets) if pairs is None else pairs
    x, v, h, m = _ld(x64), _ld(f["v"]), _ld(f["h"]), _ld(f["m"])
    rho, rho_p, P, P_p = _ld(f["rho"]), _ld(f["rho_p"]), _ld(f["P"]), _ld(f["P_p"])
    floor = LD(p["rho_floor"])
    rfl = np.where(np.isnan(rho), rho, np.maximum(rho, floor))
    pr2 = P_p / (rfl * rfl)
    with np.errstate(invalid="ignore"):
        cs = np.sqrt(LD(p["gamma"]) * P / rfl)
    d = x[i] - x[j]
    r2 = d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2]
    r = np.sqrt(r2)
    vd = v[i] - v[j]
    dot = (d[:, 0] * vd[:, 0] + d[:, 1] * vd[:, 1]) + d[:, 2] * vd[:, 2]
    s_dot = (np.abs(d) * (np.abs(v[i]) + np.abs(v[j]))).sum(-1)
    h_ij = LD(0.5) * (h[i] + h[j])
    q = r / h_ij
    t = np.where(q <= 1, 1 - q, LD(0))
    cd = CD[dim] / h_ij ** (dim + 2)
    ker = cd * t ** 3
    s_ker = np.abs(cd) * t * t * (1 + 2 * q)                  # |ker| + |x dker/dx|
    fc = -m[j] * (pr2[i] + pr2[j]) * ker
    s_fc = m[j] * (np.abs(pr2[i]) + np.abs(pr2[j])) * s_ker
    visc = dot < 0
    eps, alpha, beta = LD(p["eps"]), LD(p["alpha"]), LD(p["beta"])
    den = r2 + eps * h_ij * h_ij
    with np.errstate(all="ignore"):
        mu = h_ij * dot / den
        c_ij = LD(0.5) * (cs[i] + cs[j])
        rho_ij = LD(0.5) * (rfl[i] + rfl[j])
        pi_ij = (-alpha * c_ij * mu + beta * mu * mu) / rho_ij
        fv = np.where(visc, -m[j] * pi_ij * ker, LD(0))
        s_mu = h_ij * s_dot / den
        s_fv = m[j] * (alpha * np.abs(c_ij) * s_mu + 2 * beta * s_mu * s_mu) / rho_ij * s_ker
    # where the device's FP64 dot may have the other sign, its viscous term is within s_fv
    s_fv = np.where(visc | (np.abs(dot) <= 64 * U * s_dot), s_fv, LD(0))
    term = (fc + fv)[:, None] * d
    s_term = (s_fc + s_fv)[:, None] * np.abs(d)
    Dv = _segment_sum(i, term, n)
    s_Dv = _segment_sum(i, s_term, n)
    n_p = np.bincount(i, minlength=n)
    # accelerate! (:298-303)
    fluid = np.asarray(f["type"]) == p["fluid"]
    g, hdt = LD(p["g"]), LD(0.5) * LD(p["dt"])
    sponge = x64[:, 1] >= p["z_t"] - p["z_b"]
    with np.errstate(all="ignore"):
        buoy = np.stack([(-g * LD(e)) * rho_p / rho for e in (0.0, 1.0, 0.0)], axis=1)
    damp = np.zeros_like(v)
    damp[sponge, 1] = sponge_y(p)
    if dim == 2:
        Dv[:, 2] = 0
        s_Dv[:, 2] = 0
    with np.errstate(all="ignore"):
        vn = np.where(fluid[:, None], v + hdt * (Dv + buoy + damp), v)
        s_v = np.where(fluid[:, None], np.abs(v) + hdt * (s_Dv + np.abs(buoy) + np.abs(damp)), LD(0))
    if dim == 2:
        vn[:, 2] = v[:, 2]
    return dict(v=vn, s_v=s_v, Dv=Dv, s_Dv=s_Dv, n_p=n_p)


def ratios(dev, ref, scale):
    """|dev - ref| / (u * scale) element-wise (extended), with non-finite reference values taken
    out: there the device must give the same class (NaN, or the same infinity).  Returns (ratio
    array over the finite entries, number of class mismatches).  A zero scale demands equality."""
    dev = np.asarray(dev, dtype=np.float64)
    ref = np.asarray(ref, dtype=LD)
    scale = np.asarray(scale, dtype=LD)
    fin = np.isfinite(ref)
    ref64 = ref.astype(np.float64)
    bad_class = int(np.sum(~fin & ~((np.isnan(ref) & np.isnan(dev)) | (np.isinf(ref) & (dev == ref64)))))
    with np.errstate(all="ignore"):
        err = np.abs(dev.astype(LD) - ref)
        rat = np.where(scale > 0, err / (LD(U) * scale), np.where(err == 0, LD(0), LD(np.inf)))
    rat = np.where(np.isnan(rat), LD(np.inf), rat)
    return rat[fin], bad_class

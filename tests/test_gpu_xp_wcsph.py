"""The device's fused WCSPH step per particle against the extended-precision restatement of
tests/xp_wcsph.py, in strict and FAST_MATH arithmetic and through every pair-pass variant.

A case is warmed up by a few steps; its carried state is downloaded, the mean fluid velocity is
removed from v and uploaded again (so that the kick's 0.5 dt Dv is resolved in v instead of lost
below an ulp of the mean flow; not in the hand-built edge case, whose velocities are part of its
construction), and one sphmw_step runs.  The step is then checked in stages,
each from FP64 inputs the device had:
  x                      against xp's kick and drift of the carried state;
  rho, rho', h, P        against xp's density pass run on the device's new x and the old h;
  v                      against xp's force pass and kick run on the device's x, h, rho, rho', P,
                         P' and xp's half-step v;
with the two gates of test_xp_wcsph_emulated.py (the rigorous per-particle bound and the
median / 99th-percentile ceilings), and the pair count against xp's accepted pairs."""
import numpy as np
import pytest

import xp_wcsph as X
from sph_mountain_waves_b200 import cases
from test_gpu_edge_cases import tiny_case
from test_xp_wcsph_emulated import C_OPS, GATES
from util import load_gpu

pytestmark = pytest.mark.gpu

FAST_MATH, CELL_PAIRS, NO_PAIR_LIST, NO_PRETEST, TILES, NO_PACKED_RECORDS = 1, 2, 4, 16, 64, 128
VARIANTS = {"list": 0, "no_list": NO_PAIR_LIST, "no_pretest": NO_PRETEST, "no_records": NO_PACKED_RECORDS,
            "tiles": TILES}
MATRIX = [(a, v) for a in ("strict", "fast") for v in VARIANTS] + [("strict", "cell_pairs")]


def flags_of(arith, variant):
    return (FAST_MATH if arith == "fast" else 0) | (CELL_PAIRS if variant == "cell_pairs" else VARIANTS[variant])


def disordered_3d():
    """fluid jittered by +-0.3 dr, velocity noise (about half the pairs approach: the viscosity
    branch), h varied x[0.8, 1.3] so that pairs with h_p < r <= h exist in the density pass (it
    runs on this h: the case is checked without a warm-up step, which would rewrite h from rho)"""
    case = cases.bell_hill_3d(16, 10, 8, h_m=2000.0, a=8e3, U=20.0)
    rng = np.random.default_rng(21)
    dr = case.info["dr"]
    fl = case.fields["type"] == 0.0
    nf = int(fl.sum())
    case.fields["x"][fl] += rng.uniform(-0.3 * dr, 0.3 * dr, (nf, 3))
    case.fields["v"][fl] += rng.normal(scale=3.0, size=(nf, 3))
    case.fields["h"] = case.fields["h"] * rng.uniform(0.8, 1.3, case.n)
    return case


def edge_2d():
    """built by hand (h = 1), so that after the kick and drift of the checked step (rho' = 0 in the
    carried state: the kick leaves v as it is, and the drift is x + dt v): pairs at r == h and one
    ulp inside and outside (exact FP64 dist), coincident particles, a pair with dot == 0 and a
    relative velocity across it, particles whose rho stays below rho_floor, an isolated fluid
    particle, a crowded cell far beyond the list stride, walls and mountain.  `edge_2d_holds`
    checks these on the device's positions."""
    rng = np.random.default_rng(5)
    crowd = np.c_[rng.uniform(0.05, 0.95, (300, 2)), np.zeros(300)]
    dt = tiny_case(np.zeros((1, 3))).params["dt"]
    pts = [[-2.0, 0.0, 0], [-1.0, 0.0, 0], [-2.0, np.nextafter(1.0, 2.0), 0], [-2.0, -np.nextafter(1.0, 0.0), 0],
           [-2.6, 0.8, 0],
           [2.0, -2.0, 0], [2.0, -2.0, 0],                   # coincident, same velocity
           [2.0, 2.0, 0], [2.5, 2.0 + dt * 1.0, 0],          # 7 drifts onto 8's y: d = (-0.5, 0), vd = (0, 1)
           [-2.5, 2.5, 0], [-2.5, 2.0, 0],                   # tiny masses: rho < rho_floor
           [2.8, 0.0, 0],                                    # isolated
           [0.5, -0.5, 0], [0.5, -0.8, 0], [1.5, -0.5, 0]]   # walls, mountain
    x = np.r_[np.array(pts, dtype=np.float64), crowd]
    n = len(x)
    v = rng.normal(scale=0.3, size=(n, 3))
    v[:, 2] = 0.0
    v[:5] = 0.0                                              # the cut-off group stays put
    v[6] = v[5]
    v[7] = [0.0, 1.0, 0.0]
    v[8] = [0.0, 0.0, 0.0]
    m = rng.uniform(0.5, 1.5, n)
    m[9:11] = 1e-12
    t = np.zeros(n)
    t[12:14], t[14] = 1.0, 2.0
    return tiny_case(x, v=v, m=m, type=t)


def _dist(x, i, j):
    d = x[i] - x[j]
    return np.sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2])   # core.jl:104-105


def edge_2d_holds(case, r):
    """the edges edge_2d is built for, on the positions the device's passes ran on"""
    x, vh, h = r["got"]["x"], r["kd"]["v"].astype(np.float64), case.h
    assert _dist(x, 0, 1) == h
    assert _dist(x, 0, 2) == np.nextafter(h, 2 * h)
    assert _dist(x, 0, 3) == np.nextafter(h, 0.0)
    assert _dist(x, 5, 6) == 0.0
    d, vd = x[7] - x[8], vh[7] - vh[8]
    assert d[0] * vd[0] + d[1] * vd[1] == 0.0 and vd[1] != 0.0
    floor = case.params["rho_floor"]
    assert all(0.0 < r["got"]["rho"][k] < floor for k in (9, 10))
    assert r["got"]["rho"][11] == 0.0 and not np.isfinite(r["got"]["v"][11]).all()
    assert r["den"]["n_p"].max() > 92                           # above the largest list stride


def disordered_3d_holds(case, r):
    """pairs beyond the support of the particle's own h in the density pass (old h) and of h_ij in
    the force pass (new h) take part, as zero terms"""
    x, p = r["got"]["x"], case.params
    i, j = X.neighbour_pairs(x, case.h)
    dd = x[i] - x[j]
    rr = np.sqrt(dd[:, 0] * dd[:, 0] + dd[:, 1] * dd[:, 1] + dd[:, 2] * dd[:, 2])
    assert (rr > r["st"]["h"][i]).sum() > 0
    assert (rr > 0.5 * (r["got"]["h"][i] + r["got"]["h"][j])).sum() > 0
    vh = r["kd"]["v"].astype(np.float64)
    ff = (r["st"]["type"][i] == p["fluid"]) & (r["st"]["type"][j] == p["fluid"])
    dot = ((vh[i] - vh[j]) * dd).sum(1)[ff]
    assert 0.3 < (dot < 0).mean() < 0.7                      # the viscosity branch: about half the fluid pairs


# name: (case, warm-up steps, remove the mean flow, what the case is built to contain)
CASES = {
    "witch2d": (lambda: cases.mountain_wave_2d(n_y=24.0, dom_length=80e3, h_m=3000.0, a=10e3, U=20.0), 3, True, None),
    "hill3d": (lambda: cases.bell_hill_3d(24, 12, 10, h_m=3000.0, a=8e3, U=20.0), 3, True, None),
    "disordered3d": (disordered_3d, 0, True, disordered_3d_holds),
    # rigorous gate only: its 300-particle cell sums ~300 terms per particle, where rounding
    # alone takes the median past the ceilings set for the lattices' ~25 to ~40 neighbours
    "edge2d": (edge_2d, 0, False, edge_2d_holds),
}
STATISTICAL = {"witch2d", "hill3d", "disordered3d"}
STATE = ("x", "v", "m", "h", "rho", "rho_p", "type")


def measure(label, field, dev, ref, scale, K, statistical=True):
    """(p50, p99, max) of err / (u scale) and the list of broken gates"""
    rat, bad = X.ratios(dev, ref, scale)
    fails = [f"{label} {field}: {bad} non-finite values of the wrong class"] if bad else []
    K = np.asarray(K, dtype=np.float64).reshape(len(K), *([1] * (np.ndim(dev) - 1)))
    K = np.broadcast_to(K, np.shape(dev))[np.isfinite(np.asarray(ref, dtype=X.LD))]
    r = rat.astype(np.float64)
    if not r.size:
        return (0.0, 0.0, 0.0), fails
    if (r > K + C_OPS).any():
        fails.append(f"{label} {field}: rigorous bound broken at {int((r > K + C_OPS).sum())} values (worst {r.max():.3g})")
    st = (float(np.percentile(r, 50)), float(np.percentile(r, 99)), float(r.max()))
    lim = GATES["v"] if field == "x" else GATES[field]
    if statistical and (st[0] > lim[0] or st[1] > lim[1]):
        fails.append(f"{label} {field}: median {st[0]:.3g} (<= {lim[0]}), p99 {st[1]:.3g} (<= {lim[1]})")
    return st, fails


def prepare(case, flags, warm, remove_mean=True):
    s = load_gpu(case, flags=flags)
    s.create_cell_list()
    if warm:
        s.step(warm)
    if not remove_mean:
        return s
    v = s.field("v")
    fl = s.field("type") == case.params["fluid"]
    v[fl] -= v[fl].mean(axis=0)
    s.set_field("v", v)
    return s


def staged_step(label, case, s, targets=None, statistical=True):
    """one sphmw_step of s checked in stages; returns ({field: (p50, p99, max)}, failures, and the
    carried state, the device's results and xp's stages)"""
    p, dim = case.params, case.dim
    st = {k: s.field(k) for k in STATE}
    s.count_pairs(True)
    s.step(1)
    assert len(s) == len(st["m"])
    got = {k: s.field(k) for k in ("x", "v", "rho", "rho_p", "h", "P", "P_p")}
    sel = slice(None) if targets is None else targets
    stats, fails = {}, []
    kd = X.kick_drift(st, p)
    fluid = st["type"] == p["fluid"]
    # walls and mountain: x and v come back bit-unchanged
    for k in ("x", "v"):
        if not np.array_equal(got[k][~fluid].view(np.int64), st[k][~fluid].view(np.int64)):
            fails.append(f"{label}: a non-fluid particle's {k} changed")
    stats["x"], f = measure(label, "x", got["x"][sel], kd["x"][sel], kd["s_x"][sel], np.zeros(len(kd["x"][sel])),
                          statistical)
    fails += f
    den = X.density(dict(st, x=got["x"]), p, case.h, dim, targets=targets)
    for k, sk in (("rho", "s_rho"), ("rho_p", "s_rho_p"), ("h", "s_h"), ("P", "s_P")):
        stats[k], f = measure(label, k, got[k][sel], den[k][sel], den[sk][sel], den["n_p"][sel], statistical)
        fails += f
    fin = dict(st, x=got["x"], v=kd["v"].astype(np.float64), h=got["h"], rho=got["rho"], rho_p=got["rho_p"],
               P=got["P"], P_p=got["P_p"])
    fk = X.force_kick(fin, p, case.h, dim, targets=targets)
    fsel = np.nonzero(fluid)[0] if targets is None else np.asarray(targets)[fluid[targets]]
    stats["v"], f = measure(label, "v", got["v"][fsel, :dim], fk["v"][fsel, :dim], fk["s_v"][fsel, :dim],
                            2 * fk["n_p"][fsel], statistical)
    fails += f
    if targets is None and s.pair_count() != int(den["n_p"].sum()):
        fails.append(f"{label}: pair count {s.pair_count()} != {int(den['n_p'].sum())}")
    return stats, fails, dict(st=st, got=got, kd=kd, den=den, fk=fk)


@pytest.mark.parametrize("arith,variant", MATRIX, ids=[f"{a}-{v}" for a, v in MATRIX])
@pytest.mark.parametrize("name", list(CASES))
def test_step_against_extended_precision(gpu, name, arith, variant):
    make, warm, remove_mean, holds = CASES[name]
    case = make()
    s = prepare(case, flags_of(arith, variant), warm, remove_mean)
    _, fails, run = staged_step(f"{name} {arith} {variant}", case, s, statistical=name in STATISTICAL)
    s.close()
    if holds:
        holds(case, run)
    assert not fails, "\n".join(fails)


BIG_SAMPLE = 10_000


@pytest.mark.parametrize("arith", ["strict", "fast"])
def test_1m_particles_on_a_sample(gpu, arith):
    """bell_hill_3d_1M, where the packed records run at their realistic density, checked on a
    fixed random sample of particles"""
    case = cases.bell_hill_3d(480, 38, 48, lean=True)
    s = prepare(case, flags_of(arith, "list"), 2)
    sample = np.sort(np.random.default_rng(0).choice(case.n, BIG_SAMPLE, replace=False))
    _, fails, _ = staged_step(f"1M {arith}", case, s, targets=sample)
    s.close()
    assert not fails, "\n".join(fails)


@pytest.mark.parametrize("arith", ["strict", "fast"])
def test_four_step_call_against_four_staged_steps(gpu, arith):
    """step(4) (the force pass folds the next step's kick and drift, B_force_advance) equals four
    one-step calls bit for bit, and each of those passes the staged check"""
    case = CASES["hill3d"][0]()
    a = prepare(case, flags_of(arith, "list"), 2)
    b = prepare(case, flags_of(arith, "list"), 2)
    a.step(4)
    fails = []
    for k in range(4):
        fails += staged_step(f"4-step {arith} #{k}", case, b)[1]
    for f in ("x", "v", "rho", "h", "P"):
        assert np.array_equal(a.field(f), b.field(f)), f
    a.close()
    b.close()
    assert not fails, "\n".join(fails)
